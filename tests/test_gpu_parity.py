"""GPU parity tests: the CUDA path, called through the C ABI (libmgbx.so), against
  (a) the reference's golden vectors (tol 1e-6 on |z - gold|_2, test/runtests.jl:13-52, test/test_algebraic.jl:38-69),
  (b) the CPU oracle on the same inputs, stage by stage (f0, f1, f2 values + pattern, Newton solve, whole solve),
  (c) size-independent properties at the bench size (gradient consistency, residuals, determinism).
Tolerances (north-star): CSR pattern bit-exact; objective 1e-8 relative; z 1e-6 relative L2; Newton counts +-1
per barrier step."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spl

import mgb_oracle as O
from helpers import (GEOMS, PARABOLIC_CASES, SOLVE_CASES, default_problem, gold, lower_bound_problem)
from mgbx import geometry as G, hierarchy as H, native, problem as P, solver

pytestmark = pytest.mark.gpu
TOL = 1e-6


def rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300)


# ------------------------------------------------------------------------------------------ goldens
@pytest.mark.parametrize("name,geom,p", SOLVE_CASES)
def test_mgb_solve_golden(name, geom, p):
    sol = solver.mgb_solve(default_problem(geom, p))
    assert np.linalg.norm(sol["z"] - gold(name)) < TOL
    assert sol["stats"]["gpu_launches"] > 0


@pytest.mark.parametrize("name,geom", PARABOLIC_CASES)
def test_parabolic_golden(name, geom):
    sol = solver.parabolic_solve(H.amg(GEOMS[geom]()), h=0.5, p=1.0)
    assert np.linalg.norm(np.stack(sol["u"], axis=2) - gold(name)) < TOL


@pytest.mark.parametrize("name,geom,p", [c for c in SOLVE_CASES if c[1] in ("fem2d_P1_L2", "fem3d_k1_L2", "fem2d_P2_L2")])
def test_golden_with_pcg_forced(name, geom, p):
    """Same goldens with every Newton system solved by V-cycle PCG (no direct dense solve at the top)."""
    sol = solver.mgb_solve(default_problem(geom, p), config=dict(dense_direct_max=0, coarse_max=0))
    assert np.linalg.norm(sol["z"] - gold(name)) < TOL
    assert sol["stats"]["pcg_iters"] > 0


# ------------------------------------------------------------------------------------------ failure semantics
def test_feasibility_escalation():
    sol = solver.mgb_solve(lower_bound_problem(50.0))
    assert sol["SOL_feasibility"] is not None
    assert np.max(np.abs(sol["z"] - 50.0)) < 1e-3
    assert "bounding box R=100.0" in sol["log"]


def test_infeasible_certified():
    with pytest.raises(solver.MGBConvergenceFailure) as e:
        solver.mgb_solve(lower_bound_problem(0.0, infeasible_pair=True))
    assert e.value.code == "infeasible"


def test_feasibility_rmax():
    with pytest.raises(solver.MGBConvergenceFailure) as e:
        solver.mgb_solve(lower_bound_problem(1.0e6), feasibility_Rmax=1000.0)
    assert e.value.code == "feasibility_Rmax"


def test_feasible_start_skips_phase1():
    sol = solver.mgb_solve(lower_bound_problem(-50.0))
    assert sol["SOL_feasibility"] is None
    assert np.max(np.abs(sol["z"] + 50.0)) < 1e-3


def test_tiny_tolerance_is_a_convergence_failure():
    """test/test_algebraic_coverage.jl:119-127: tol=1e-50 cannot be reached."""
    with pytest.raises((solver.MGBConvergenceFailure, FloatingPointError)):
        solver.mgb_solve(default_problem("fem1d_3nodes", 1.0), tol=1e-50, maxit=40)


# ------------------------------------------------------------------------------------------ edge cases and argument errors
def test_smallest_problems_and_single_level():
    """One element / two nodes (fem1d with 2 nodes: no interior unknown of u, only the slack) and a hierarchy of one level."""
    mg = H.amg(G.fem1d(nodes=np.linspace(-1, 1, 2)))
    prob = P.assemble(mg, p=1.0)
    sd = solver.mgb_solve(prob)
    so = O.mgb_solve(prob)
    assert rel(sd["z"], so["z"]) < 1e-6
    # a u-only problem (no slack at all): linear barrier, one state variable, one D row
    sol = solver.mgb_solve(lower_bound_problem(-3.0, nodes=2))
    assert np.all(np.isfinite(sol["z"]))


def test_bad_arguments_are_errors_not_crashes():
    prob = default_problem("fem1d_5nodes", 1.0)
    h = native.Handle(prob)
    try:
        o = h.step_opts()
        r = native.StepResult()
        L = native.lib()
        import ctypes as C
        assert L.mgbx_step(h._h, 5, 0.1, C.byref(o), C.byref(r)) == native.ERR_ARG          # no such AMG
        assert L.mgbx_step(h._h, 1, 0.1, C.byref(o), C.byref(r)) == native.ERR_ARG          # feasibility AMG not attached
        o.line_search = 7
        assert L.mgbx_step(h._h, 0, 0.1, C.byref(o), C.byref(r)) == native.ERR_ARG
        assert b"line_search" in L.mgbx_last_error(h._h)
        assert L.mgbx_level_size(h._h, 0, 99) == -1
        s = np.zeros(3)
        out = np.zeros(3)
        assert L.mgbx_barrier_eval(h._h, 0, 99, 1.0, native._ptr(s), 0, native._ptr(out)) == native.ERR_ARG
        assert L.mgbx_barrier_eval(h._h, 0, 0, 1.0, native._ptr(s), 2, native._ptr(out)) == native.ERR_ARG
        # the handle is still usable after the errors
        o = h.step_opts(initial_step=1)
        rc, r = h.step(0, 0.1, o)
        assert rc in (native.OK, native.NOT_CONVERGED)
    finally:
        h.close()
    # inconsistent problem descriptions are rejected at create time
    bad = default_problem("fem1d_5nodes", 1.0)
    bad.Q.pieces[0].idx = (0, 7)          # D row 7 does not exist
    with pytest.raises(native.MgbxError) as e:
        native.Handle(bad)
    assert e.value.code == native.ERR_ARG and "D row" in str(e.value)


def test_start_outside_the_domain_is_reported_by_value():
    """A starting point outside the barrier's domain: mgbx_step returns MGBX_NON_FINITE (the reference raises from newton)."""
    prob = default_problem("fem2d_P1_L2", 1.0)
    h = native.Handle(prob)
    try:
        n = prob.geometry.n
        z = prob.g.T.reshape(-1).copy()
        z[n:] = -1.0                         # slack below zero everywhere
        h.set_z(z, 0)
        rc, r = h.step(0, 0.1, h.step_opts(initial_step=1))
        assert rc == native.NON_FINITE and r.converged == 0
        need, b, zabs = h.phase1_init()      # ... and phase I is what the driver does about it
        assert need and b >= 2.0
    finally:
        h.close()


# ------------------------------------------------------------------------------------------ stage-by-stage vs oracle
def _obstacle_problem():
    """two-sided obstacle + p-Laplace cone as an intersection (linear + EP pieces, select grid)."""
    mg = H.amg(G.subdivide(G.fem2d_P1(), 3))
    n = mg.geometry.n
    x = mg.geometry.xflat()
    lin = P.convex_linear(mg, idx=(0,), A_grid=np.tile([1.0, -1.0], (n, 1)),
                          b_grid=np.stack([3.0 + 0 * x[:, 0], 3.0 + x[:, 0] ** 2], axis=1))
    ep = P.convex_Euclidian_power(mg, idx=(1, 2, 3), p_grid=np.where(x[:, 0] > 0, 1.5, 3.0))
    sel = np.stack([(x[:, 1] > -0.5).astype(float), np.ones(n)], axis=1)   # obstacle only on part of the domain
    Q = P.convex_piecewise(mg, [lin, ep], select_grid=sel)
    return P.assemble(mg, Q=Q, p=1.5)


STAGE_PROBLEMS = {
    "p1L3_p1.5": lambda: default_problem_l("p1", 3, 1.5),
    "p2L2_p1": lambda: default_problem("fem2d_P2_L2", 1.0),
    "q1L2_p1.5": lambda: default_problem("fem3d_k1_L2", 1.5),
    "spectral2d": lambda: default_problem("spectral2d_n5", 1.0),
    "piecewise": _obstacle_problem,
}


def default_problem_l(kind, L, p):
    return P.assemble(H.amg(G.subdivide(G.fem2d_P1(), L)), p=p)


@pytest.mark.parametrize("name", list(STAGE_PROBLEMS))
@pytest.mark.parametrize("which", [0, 1])
def test_stages_match_oracle(name, which):
    prob = STAGE_PROBLEMS[name]()
    M = prob.M[which]
    n = M.geometry.n
    t = 0.7
    rng = np.random.default_rng(5)
    bw = O.barrier_weights(M.w) if which == 0 else None
    h = native.Handle(prob, barrier_weights=bw)
    try:
        Qo, c = prob.Q, t * prob.f
        z0 = prob.g.T.reshape(-1).copy()
        if which == 1:
            # move the main state off-domain so that phase I is armed, then compare on the feasibility AMG
            need, b, zabs = h.phase1_init()
            if not need:
                z_bad = z0.copy()
                z_bad[-n:] = -1.0          # negative slack: outside every cone
                h.set_z(z_bad, 0)
                need, b, zabs = h.phase1_init()
            assert need
            h.set_feasibility_box(b, 50.0)
            Qo = O.FeasibilityConvex(prob.Q, b, 50.0, prob.M[0].nD + 1)
            c = np.zeros((n, M.nD))
            c[:, prob.M[0].nD] = t
            z0 = h.get_z(1)
        B = O.Barrier(Qo, bw)
        ops = O.operators(M)
        for J in range(len(M.R_fine)):
            R = M.R_fine[J]
            s = 1e-3 * rng.normal(size=R.shape[1])
            y_o = B.f0(s, M.w, c, R, ops, z0)
            assert np.isfinite(y_o)
            g_o = B.f1(s, M.w, c, R, ops, z0)
            H_o = sp.csr_matrix(B.f2(s, M.w, c, R, ops, z0))
            assert abs(h.barrier_eval(which, J, t, s, 0) - y_o) <= 1e-12 * max(1.0, abs(y_o))
            assert rel(h.barrier_eval(which, J, t, s, 1), g_o) < 1e-11
            H_d = h.hessian(which, J, t, s)
            optr, oind = O.hessian_pattern(M, J)
            assert np.array_equal(H_d.indptr, optr) and np.array_equal(H_d.indices, oind)   # bit-exact pattern
            assert abs(H_d - H_o).sum() <= 1e-11 * abs(H_o).sum()
            x_o = O.solve_sym(H_o, g_o)
            x_d, _ = h.solve_newton_system(which, J, t, s, g_o)
            assert rel(x_d, x_o) < 1e-8
    finally:
        h.close()


def test_domain_escape_is_signalled_by_value():
    """Log(x<=0) = -Inf, _safe_pow(s<=0) = 0 => f0 = +Inf outside the cone (src/utils.jl:14, convex_linear.jl:388-390)."""
    prob = default_problem("fem2d_P1_L2", 1.0)
    M = prob.M[0]
    h = native.Handle(prob)
    try:
        J = len(M.R_fine) - 1
        s = np.zeros(M.R_fine[J].shape[1])
        s[-M.geometry.n:] = -1000.0      # slack far below |grad u|
        assert not np.isfinite(h.barrier_eval(0, J, 1.0, s, 0))      # +Inf (or NaN from 0*Inf, as in the reference)
    finally:
        h.close()


# ------------------------------------------------------------------------------------------ whole solve vs oracle
def _check_newton_counts(idv, iov):
    """Newton counts +-1 per barrier step (north-star gate).  The LAST column also holds the finalize pass
    (mgb.jl:76-80), a second Newton run whose only stop rule is floating-point stagnation
    (`stopping_exact`, newton.jl:187: ynext >= ymin && |gnext| >= 0.9 gmin at roundoff level): its length is a
    roundoff random walk: at t ~ 1e8 the objective is ~1e9 and the Armijo test compares differences of ~1e-8, i.e.
    it is decided by the summation order of f0; when the full step is rejected by noise the search accepts s = 1/2
    and |g| merely halves per iteration until it reaches its floor (observed: 1 iteration in the oracle, 3 with one
    GPU kernel variant, 7 with another, all ending at the same z to 1e-12).  That column is therefore only held to
    +-1 for the t-step plus the halving tail (<= log2 of the gradient's dynamic range, ~10); the no-finalize runs
    pin +-1 on every barrier step, and z / objective parity is asserted separately."""
    d = np.abs(idv.sum(axis=0) - iov.sum(axis=0))
    assert np.max(d[:-1], initial=0) <= 1
    assert d[-1] <= 11


@pytest.mark.parametrize("L,p,cfg", [(5, 1.5, {}), (6, 1.0, {}), (6, 1.5, dict(dense_direct_max=64, coarse_max=32))])
def test_solve_matches_oracle_midsize(L, p, cfg):
    prob = P.assemble(H.amg(G.subdivide(G.fem2d_P1(), L)), p=p)
    sd = solver.mgb_solve(prob, config=cfg)
    so = O.mgb_solve(prob)
    assert rel(sd["z"], so["z"]) < 1e-6
    od, oo = sd["SOL_main"]["c_dot_Dz"][-1], so["SOL_main"]["c_dot_Dz"][-1]
    assert abs(od - oo) <= 1e-8 * abs(oo)
    idv, iov = sd["SOL_main"]["its"], so["SOL_main"]["its"]
    assert idv.shape == iov.shape
    _check_newton_counts(idv, iov)
    assert np.allclose(sd["SOL_main"]["ts"], so["SOL_main"]["ts"])
    # the same ramp without the finalize pass: every barrier step within +-1
    sd2 = solver.mgb_solve(prob, config=cfg, finalize=False)
    so2 = O.mgb_solve(prob, finalize=False)
    assert np.max(np.abs(sd2["SOL_main"]["its"].sum(axis=0) - so2["SOL_main"]["its"].sum(axis=0))) <= 1
    assert rel(sd2["z"], so2["z"]) < 1e-6


def test_fem3d_midsize_matches_oracle():
    prob = P.assemble(H.amg(G.subdivide(G.fem3d(k=1), 3)), p=1.0)
    sd = solver.mgb_solve(prob, config=dict(dense_direct_max=64, coarse_max=32))
    so = O.mgb_solve(prob)
    assert rel(sd["z"], so["z"]) < 1e-6
    _check_newton_counts(sd["SOL_main"]["its"], so["SOL_main"]["its"])
    sd2 = solver.mgb_solve(prob, config=dict(dense_direct_max=64, coarse_max=32), finalize=False)
    so2 = O.mgb_solve(prob, finalize=False)
    assert np.max(np.abs(sd2["SOL_main"]["its"].sum(axis=0) - so2["SOL_main"]["its"].sum(axis=0))) <= 1
    assert rel(sd2["z"], so2["z"]) < 1e-6


def test_illinois_line_search_matches_oracle():
    """linesearch_illinois (newton.jl:84-103): exact line search by Illinois root finding, device evaluations."""
    prob = P.assemble(H.amg(G.subdivide(G.fem2d_P1(), 4)), p=1.5)
    sd = solver.mgb_solve(prob, line_search=1)
    so = O.mgb_solve(prob, line_search=O.linesearch_illinois())
    assert rel(sd["z"], so["z"]) < 1e-6
    assert sd["SOL_main"]["its"].shape == so["SOL_main"]["its"].shape
    d = np.abs(sd["SOL_main"]["its"].sum(axis=0) - so["SOL_main"]["its"].sum(axis=0))
    assert np.max(d[:-1], initial=0) <= 1


def test_parabolic_midsize_matches_oracle():
    """parabolic_solve (Parabolic.jl:126-173) on fem2d_P2 at level 4 (n = 896): 3 state variables, a piecewise intersection of
    two Euclidean-power cones, phase I at every time step (feasibility AMG attached lazily), one handle reused across steps."""
    mg = H.amg(G.subdivide(G.fem2d_P2(), 4))
    sd = solver.parabolic_solve(mg, h=0.5, p=1.0)
    so = O.parabolic_solve(mg, P.assemble, P.intersect, P.convex_Euclidian_power, H.prepare_amg, P.default_slack_space, h=0.5, p=1.0)
    ud, uo = np.stack(sd["u"], axis=2), np.stack(so["u"], axis=2)
    assert rel(ud, uo) < 1e-6


@pytest.mark.parametrize("L,cfg", [(3, {}), (4, {})])
def test_pure_p2_masked_barrier_matches_oracle(L, cfg):
    """Pure P2 (no bubble): the corner nodes carry zero quadrature weight, so the barrier is averaged over the masked node
    set (`_masked_barrier`, convex.jl:213-257, weights convex.jl:279-304) and the slack lives in :broken_P1 (not node-local:
    no condensation, the Newton system couples u and s and carries the 1/slack^2 entries: it is solved directly -- forcing
    the V-cycle PCG onto it degrades the t-ramp, DESIGN.md "known limits").  test/test_pure_p2.jl:53-63 pins this family."""
    prob = P.assemble(H.amg(G.subdivide(G.fem2d_P2(bubble=False), L)), p=1.5)
    assert (prob.M[0].w == 0).any()
    sd = solver.mgb_solve(prob, config=cfg)
    so = O.mgb_solve(prob)
    assert rel(sd["z"], so["z"]) < 1e-6
    od, oo = sd["SOL_main"]["c_dot_Dz"][-1], so["SOL_main"]["c_dot_Dz"][-1]
    assert abs(od - oo) <= 1e-8 * abs(oo)
    assert sd["SOL_main"]["its"].shape == so["SOL_main"]["its"].shape
    d = np.abs(sd["SOL_main"]["its"].sum(axis=0) - so["SOL_main"]["its"].sum(axis=0))
    assert np.max(d[:-1], initial=0) <= 1


# ------------------------------------------------------------------------------------------ persistent solve kernel
def _newton_system(prob, seed):
    M = prob.M[0]
    J = len(M.R_fine) - 1
    m = M.R_fine[J].shape[1]
    rng = np.random.default_rng(seed)
    s = 1e-3 * rng.normal(size=m)
    g = rng.normal(size=m)
    return J, s, g


def _pcg_solve(prob, J, s, g, **cfg):
    """One Newton system solved twice by k_pcg2 on a fresh handle: the residual and determinism checks, then (x, its, H)."""
    h = native.Handle(prob, dense_direct_max=0, coarse_max=40, pcg_rtol=1e-11, **cfg)
    try:
        x, its = h.solve_newton_system(0, J, 2.0, s, g)
        Hm = h.hessian(0, J, 2.0, s)
        assert np.linalg.norm(Hm @ x - g) <= 1e-9 * np.linalg.norm(g)
        x2, its2 = h.solve_newton_system(0, J, 2.0, s, g)
        assert np.array_equal(x, x2) and its == its2          # deterministic
    finally:
        h.close()
    return x, its, Hm


# bound on rel(x, spsolve(H, g)) of the solves below: 10x the largest distance measured on a B200 (1e-14 on these systems)
# rounded up to a power of ten, but not below 1e-8, the agreement two PCG solves are held to
EXACT_SOLVE_RTOL = 1e-8


@pytest.mark.parametrize("tail_max", [0, 300, 10 ** 9])
def test_persistent_pcg_tail_splits_agree(tail_max):
    """k_pcg2 runs the V-cycle levels with more than tail_max unknowns grid-wide and the others in CTA 0 alone.  Every split
    runs the same arithmetic: the iteration count (+-1) and the solution (to the PCG tolerance) of the split without a tail
    (tail_max = 0), and the solution of the exact sparse solve."""
    prob = P.assemble(H.amg(G.subdivide(G.fem2d_P1(), 6)), p=1.5)
    J, s, g = _newton_system(prob, 3)
    x0, its0, _ = _pcg_solve(prob, J, s, g, tail_max=0, smoother=0)
    x, its, Hm = _pcg_solve(prob, J, s, g, tail_max=tail_max, smoother=0)
    assert abs(its0 - its) <= 1
    assert rel(x, x0) < 1e-8
    assert rel(x, spl.spsolve(Hm.tocsc(), g)) <= EXACT_SOLVE_RTOL


# PCG iterations of k_pcg2 on the systems of the test below, measured on a B200 (the first-generation CSR kernel that k_pcg2
# replaced took the same counts)
PINNED_PCG_ITS = {  # (problem, tail_max, smoother, precond_fp32): iterations
    ("p1L7", 1200, 1, 0): 9, ("box12", 0, 1, 0): 9, ("box12", 300, 1, 0): 9,
    ("p1L7", 1200, 1, 1): 9, ("box12", 0, 1, 1): 9, ("box12", 300, 1, 1): 9,
    ("p1L7", 1200, 0, 0): 9, ("box12", 0, 0, 0): 9, ("box12", 300, 0, 0): 9,
}


@pytest.mark.parametrize("smoother,fp32", [(1, 0), (1, 1), (0, 0)])
def test_persistent_pcg_iterations_and_exact_solution(smoother, fp32):
    """csrc/pcg2.cu (sliced-ELL levels, row ownership, tail out of shared memory with FP32 matrix values): pinned iteration
    counts (+-1) and the solution of the exact sparse solve, with the Chebyshev and the l1-Jacobi smoother, with FP64 and FP32
    preconditioner matrices, on a 2-D and a 3-D hierarchy, with and without a tail."""
    for name, prob, tail_max in (("p1L7", P.assemble(H.amg(G.subdivide(G.fem2d_P1(), 7)), p=1.5), 1200),
                                 ("box12", P.assemble(H.amg(G.structured_box(3, 12, k=1)), p=1.0), 0),
                                 ("box12", P.assemble(H.amg(G.structured_box(3, 12, k=1)), p=1.0), 300)):
        J, s, g = _newton_system(prob, 11)
        # lambda_power = 0: the Gershgorin bound of lambda_max, as when the counts were pinned
        x, its, Hm = _pcg_solve(prob, J, s, g, smoother=smoother, precond_fp32=fp32, lambda_power=0, tail_max=tail_max)
        pinned = PINNED_PCG_ITS[(name, tail_max, smoother, fp32)]
        assert abs(its - pinned) <= 1, (name, tail_max, its, pinned)
        assert rel(x, spl.spsolve(Hm.tocsc(), g)) <= EXACT_SOLVE_RTOL


def test_persistent_pcg_uncondensed_and_coarse_levels():
    """Newton systems on coarse levels (the recovery path of mgb_step) and without node-local condensation."""
    prob = P.assemble(H.amg(G.subdivide(G.fem2d_P1(), 5)), p=1.0)
    M = prob.M[0]
    L = len(M.R_fine)
    rng = np.random.default_rng(4)
    h = native.Handle(prob, dense_direct_max=0, coarse_max=20, condense=0, pcg_rtol=1e-11)
    try:
        for J in (L - 1, L - 2, L - 3):
            m = M.R_fine[J].shape[1]
            s = np.zeros(m)
            g = rng.normal(size=m)
            x, its = h.solve_newton_system(0, J, 1.0, s, g)
            Hm = h.hessian(0, J, 1.0, s)
            assert np.linalg.norm(Hm @ x - g) <= 1e-8 * np.linalg.norm(g)
    finally:
        h.close()


# ------------------------------------------------------------------------------------------ element kernel variants
@pytest.mark.parametrize("name", ["p1L4_p1.5", "q1L2_p1", "fem1d_p1", "p2L2_p1.5"])
def test_element_kernel_variants_agree(name):
    """fused=1 (specialised kernel of the default (u, s) Euclidean-power family), fused=2 (generic fused kernel) and
    fused=0 (separate node / block kernels) evaluate the same f0, f1 and Newton direction."""
    prob = {"p1L4_p1.5": lambda: P.assemble(H.amg(G.subdivide(G.fem2d_P1(), 4)), p=1.5),
            "q1L2_p1": lambda: default_problem("fem3d_k1_L2", 1.0),
            "fem1d_p1": lambda: default_problem("fem1d_5nodes", 1.0),
            "p2L2_p1.5": lambda: default_problem("fem2d_P2_L2", 1.5)}[name]()
    M = prob.M[0]
    J = len(M.R_fine) - 1
    m = M.R_fine[J].shape[1]
    rng = np.random.default_rng(9)
    s = 1e-3 * rng.normal(size=m)
    rhs = rng.normal(size=m)
    bw = O.barrier_weights(M.w)
    res = []
    for fused in (1, 2, 0):
        h = native.Handle(prob, barrier_weights=bw, fused=fused)
        try:
            f0 = h.barrier_eval(0, J, 0.9, s, 0)
            g = h.barrier_eval(0, J, 0.9, s, 1)
            x, _ = h.solve_newton_system(0, J, 0.9, s, rhs)
            res.append((f0, g, x))
        finally:
            h.close()
    for f0, g, x in res[1:]:
        assert abs(f0 - res[0][0]) <= 1e-13 * max(1.0, abs(res[0][0]))
        assert rel(g, res[0][1]) < 1e-12
        assert rel(x, res[0][2]) < 1e-8


# ------------------------------------------------------------------------------------------ spectral (dense) path
@pytest.mark.parametrize("name,geom,cfg", [("spectral2d_n9", lambda: G.spectral2d(n=9), {}), ("spectral2d_n16", lambda: G.spectral2d(n=16), {}),
                                           ("spectral2d_n16_unstructured", lambda: G.spectral2d(n=16), {"spectral_kron": 0}),
                                           ("spectral1d_n96", lambda: G.spectral1d(n=96), {})])
def test_spectral_dense_path_matches_oracle(name, geom, cfg):
    """Spectral discretisations with more than 64 nodes take the dense path: per-node Hessian samples, then R'HR as FP64 DMMA
    GEMMs into a full matrix, dense Cholesky solve.  spectral2d (operators and prolongations are Kronecker products,
    src/spectral2d.jl:22-35) assembles sum-factorised by default; cfg.spectral_kron = 0 and spectral1d take the unstructured
    products H = sum D_j' diag(h) D_k, R'(H R)."""
    prob = P.assemble(H.amg(geom()), p=1.0)
    M = prob.M[0]
    t = 0.7
    rng = np.random.default_rng(2)
    h = native.Handle(prob, barrier_weights=O.barrier_weights(M.w), **cfg)
    try:
        B = O.Barrier(prob.Q, O.barrier_weights(M.w))
        ops = O.operators(M)
        z0 = prob.g.T.reshape(-1).copy()
        for J in (len(M.R_fine) - 1, len(M.R_fine) - 2):
            R = M.R_fine[J]
            s = 1e-3 * rng.normal(size=R.shape[1])
            H_o = np.asarray(sp.csr_matrix(B.f2(s, M.w, t * prob.f, R, ops, z0)).todense())
            g_o = B.f1(s, M.w, t * prob.f, R, ops, z0)
            assert rel(h.barrier_eval(0, J, t, s, 1), g_o) < 1e-10
            H_d = np.asarray(h.hessian(0, J, t, s).todense())
            assert np.abs(H_d - H_o).max() <= 1e-10 * np.abs(H_o).max()
            x_d, _ = h.solve_newton_system(0, J, t, s, g_o)
            assert np.linalg.norm(H_o @ x_d - g_o) <= 1e-7 * np.linalg.norm(g_o)
    finally:
        h.close()
    sd = solver.mgb_solve(prob, config=cfg)
    so = O.mgb_solve(prob)
    assert rel(sd["z"], so["z"]) < 1e-6
    assert sd["SOL_main"]["its"].shape == so["SOL_main"]["its"].shape
    d = np.abs(sd["SOL_main"]["its"].sum(axis=0) - so["SOL_main"]["its"].sum(axis=0))
    assert np.max(d[:-1], initial=0) <= 1


# ------------------------------------------------------------------------------------------ bench-size properties
@pytest.fixture(scope="module")
def big_problem():
    return P.assemble(H.amg(G.subdivide(G.fem2d_P1(), 9)), p=1.5)     # n = 393 216 (same family as the bench config)


def test_bench_size_properties(big_problem):
    prob = big_problem
    M = prob.M[0]
    J = len(M.R_fine) - 1
    m = M.R_fine[J].shape[1]
    rng = np.random.default_rng(11)
    h = native.Handle(prob, pcg_rtol=1e-10)      # the residual gate below is 1e-8 (the shipped default tolerance is 1e-7)
    try:
        s = 1e-3 * rng.normal(size=m)
        d = rng.normal(size=m)
        d /= np.linalg.norm(d)
        t = 3.0
        # f1 is the gradient of f0: central difference along a random direction
        eps = 1e-6
        fd = (h.barrier_eval(0, J, t, s + eps * d, 0) - h.barrier_eval(0, J, t, s - eps * d, 0)) / (2 * eps)
        g = h.barrier_eval(0, J, t, s, 1)
        assert abs(fd - g @ d) <= 1e-6 * max(1.0, abs(g @ d))
        # f2 is the Jacobian of f1 and is symmetric
        Hm = h.hessian(0, J, t, s)
        assert abs(Hm - Hm.T).max() <= 1e-12 * abs(Hm).max()
        gd = (h.barrier_eval(0, J, t, s + eps * d, 1) - h.barrier_eval(0, J, t, s - eps * d, 1)) / (2 * eps)
        assert rel(Hm @ d, gd) < 1e-5
        # the condensed V-cycle PCG solve satisfies the full (uncondensed) Newton system
        x, its = h.solve_newton_system(0, J, t, s, g)
        assert its > 0
        assert np.linalg.norm(Hm @ x - g) <= 1e-8 * np.linalg.norm(g)
        # run-to-run determinism (fixed-order reductions and assembly)
        g2 = h.barrier_eval(0, J, t, s, 1)
        x2, _ = h.solve_newton_system(0, J, t, s, g)
        assert np.array_equal(g, g2) and np.array_equal(x, x2)
    finally:
        h.close()


def test_bench_size_solve_is_a_minimiser(big_problem):
    prob = big_problem
    sol = solver.mgb_solve(prob)
    SM = sol["SOL_main"]
    assert SM["ts"][-1] >= 1.0 / np.sqrt(np.finfo(float).eps)
    # the duality-gap scalar decreases monotonically to the optimum along the t-ramp (up to roundoff)
    cd = SM["c_dot_Dz"]
    assert np.all(np.diff(cd) <= 1e-7 * abs(cd[-1]))
    # boundary data kept, slack dominates |grad u| (cone constraint s >= |grad u|^p) at every node
    z = sol["z"]
    assert np.all(np.isfinite(z))
    Mm = prob.M[0]
    Dz = O.operators(Mm).apply(z.T.reshape(-1))
    assert np.all(Dz[:, 3] >= np.hypot(Dz[:, 1], Dz[:, 2]) ** 1.5 - 1e-9)
