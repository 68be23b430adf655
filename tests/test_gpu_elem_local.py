"""Element-local elimination of a slack variable (csrc/elem_schur.cuh): a slack in :broken_P1 is eliminated exactly, element
by element, before the Newton solve.  Newton systems against the exact sparse solve of the oracle's full (u, s) Hessian, whole
solves against the oracle and its fixtures, and the refusals that remain above the dense solver's size."""
import time

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spl

import mgb_oracle as O
from mgbx import geometry as G, hierarchy as H, native, problem as P, solver
from test_gpu_fixtures import check_solution, fixture

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps


def rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300))


def pure_p2(L, p=1.0):
    return P.assemble(H.amg(G.subdivide(G.fem2d_P2(bubble=False), L)), p=p)


def bubble_p2(L, p=1.0):
    """fem2d_P2 with its bubble (7 nodes, every weight non-zero) and the slack in :broken_P1: P_e is 7 x 3, so the elimination
    couples the element's nodes (pure P2 masks the corners and its P_e is the identity on the three midpoints)."""
    return P.assemble(H.amg(G.subdivide(G.fem2d_P2(), L)), p=p, state_variables=[("u", "dirichlet"), ("s", "broken_P1")])


def kappa1(Hm):
    """1-norm condition number estimate of a sparse SPD matrix (LU of H for the inverse)."""
    lu = spl.splu(Hm.tocsc())
    m = Hm.shape[0]
    inv = spl.LinearOperator((m, m), matvec=lu.solve, rmatvec=lambda v: lu.solve(v, trans="T"), dtype=float)
    return spl.onenormest(Hm) * spl.onenormest(inv)


# Forward error of x against spsolve on the full system, in units of eps * kappa_1(H_full).  Both solves are backward stable, so
# their distance is bounded by a small multiple of eps kappa; the condensed solve factors the Schur complement, whose condition
# number is at most the full one's.  Measured on a B200 (1000 W) over the cases below: 6e-5 to 5.5e-3 (kappa_1 from 1.7e12 to
# 1e15, relative errors 1.8e-6 to 1.4e-5); the bound is 0.1, about 20x the largest.
KAPPA_FACTOR = 0.1


@pytest.mark.parametrize("kind,L", [("pure", 4), ("pure", 5), ("bubble", 3), ("bubble", 4)])
def test_element_condensed_newton_system_matches_exact_solve(kind, L):
    prob = (pure_p2 if kind == "pure" else bubble_p2)(L)
    M = prob.M[0]
    J = len(M.R_fine) - 1
    R = M.R_fine[J]
    so = O.mgb_solve(prob)
    z = np.asarray(so["z"]).T.reshape(-1).copy()      # interior point: the oracle's minimiser, (u, s) blocks
    bw = O.barrier_weights(M.w)
    B = O.Barrier(prob.Q, bw)
    ops = O.operators(M)
    s = np.zeros(R.shape[1])
    h = native.Handle(prob, barrier_weights=bw)
    try:
        h.set_z(z, 0)
        for t in (1.0, 1e4, 1e7):
            g = B.f1(s, M.w, t * prob.f, R, ops, z)
            Hm = sp.csr_matrix(B.f2(s, M.w, t * prob.f, R, ops, z))
            x_ref = spl.spsolve(Hm.tocsc(), g)
            x, _ = h.solve_newton_system(0, J, t, s, g)
            k = kappa1(Hm)
            err = rel(x, x_ref)
            print("%s L%d t=%g: m=%d kappa_1=%.2e rel err %.2e  err / (eps kappa) %.2e" % (kind, L, t, Hm.shape[0], k, err, err / (EPS * k)))
            assert err <= max(KAPPA_FACTOR * EPS * k, 1e-12), (t, err, k)
    finally:
        h.close()


def _check_against_oracle(sd, so):
    assert rel(sd["z"], so["z"]) < 1e-6
    od, oo = sd["SOL_main"]["c_dot_Dz"][-1], so["SOL_main"]["c_dot_Dz"][-1]
    assert abs(od - oo) <= 1e-8 * abs(oo)
    assert sd["SOL_main"]["its"].shape == so["SOL_main"]["its"].shape
    d = np.abs(sd["SOL_main"]["its"].sum(axis=0) - so["SOL_main"]["its"].sum(axis=0))
    assert np.max(d[:-1], initial=0) <= 1


@pytest.mark.parametrize("L", [3, 4, 5])
def test_bubble_p2_broken_p1_slack_matches_oracle(L):
    prob = bubble_p2(L)
    sd = solver.mgb_solve(prob)
    so = O.mgb_solve(prob)
    _check_against_oracle(sd, so)
    print("bubble P2 L%d: %s" % (L, {k: sd["stats"][k] for k in ("linear_solves", "pcg_iters", "direct_fallbacks", "ms_solve")}))


def test_pure_p2_L6_is_solved_after_condensation():
    """Refused before (10 113 unknowns with the slack); 3 969 after the element-local elimination: PCG, then the dense fallback."""
    fx, meta = fixture("pure_p2_L6_p1")
    prob = pure_p2(6)
    t0 = time.time()
    sol = solver.mgb_solve(prob)
    wall = time.time() - t0
    st = sol["stats"]
    print("pure P2 L6:", check_solution(sol, fx, meta), "wall %.1f s" % wall,
          {k: st[k] for k in ("linear_solves", "pcg_iters", "direct_fallbacks", "ms_f2", "ms_solve")})


def test_pure_p2_condensed_matches_uncondensed_dense_path():
    """condense = 0 keeps (u, s) in the system and solves it densely (609 unknowns at L4, 225 after the elimination): the exact
    elimination must land on the same minimiser with the same Newton counts.  As in the fixture gate, the finalize pass (a Newton
    run stopped only by floating-point stagnation, src/mgb.jl:76-80) is counted apart and held to the halving tail."""
    prob = pure_p2(4)
    a = solver.mgb_solve(prob, config=dict(condense=0))
    b = solver.mgb_solve(prob, config=dict(condense=1))
    assert rel(b["z"], a["z"]) < 1e-10

    def counts(sol):
        its = np.array(sol["SOL_main"]["its"])
        c = its.sum(axis=0)
        c[-1] -= int(sol["SOL_main"]["its_finalize"])
        return c, int(sol["SOL_main"]["its_finalize"])
    (ca, fa), (cb, fb) = counts(a), counts(b)
    assert np.array_equal(ca, cb), (ca.tolist(), cb.tolist())
    assert abs(fa - fb) <= 11, (fa, fb)


def _refused(prob):
    t0 = time.time()
    with pytest.raises(native.MgbxError) as e:
        solver.mgb_solve(prob)
    return e.value, time.time() - t0


def test_pure_p2_L7_still_refused_with_condensed_size():
    err, wall = _refused(pure_p2(7))
    assert err.code == native.ERR_UNSUPPORTED
    assert "element-local" in str(err) and "16129" in str(err), str(err)
    assert wall < 5.0, wall


def test_slack_that_is_not_element_local_is_still_refused():
    """A slack in :dirichlet (only :id rows, but continuous across elements) is neither node- nor element-local."""
    prob = P.assemble(H.amg(G.subdivide(G.fem2d_P2(bubble=False), 7)), p=1.0, state_variables=[("u", "dirichlet"), ("s", "dirichlet")])
    err, wall = _refused(prob)
    assert err.code == native.ERR_UNSUPPORTED
    assert "neither node-locally nor element-locally" in str(err), str(err)
