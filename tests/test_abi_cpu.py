"""CPU-side checks of the C-ABI library: it loads, exports every symbol include/mgbx.h declares, fails
loudly without a GPU, and its host-only assembly-plan pattern is bit-exact with the oracle's restatement
of src/BlockMatrices.jl:344-446."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp

import mgb_oracle as O
from helpers import GEOMS, default_problem
from mgbx import native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_matches_header_symbols_and_abi_version():
    """Every symbol include/mgbx.h declares is exported, and the library reports the header's ABI version (2: mgbx_config
    without use_graphs and pcg_lanes)."""
    hdr = open(os.path.join(ROOT, "include", "mgbx.h")).read()
    declared = set(re.findall(r"\b(mgbx_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no prototypes found"
    L = native.lib()
    for name in sorted(declared):
        assert hasattr(L, name), name
    assert set(native.EXPORTS) == declared
    assert re.search(r"#define MGBX_ABI_VERSION (\d+)", hdr).group(1) == "2"
    assert L.mgbx_abi_version() == 2


def test_struct_sizes_match_header():
    cfg = native.default_config()
    assert cfg.dense_direct_max == 2048 and cfg.condense == 1
    o = native.StepOpts()
    native.lib().mgbx_default_step_opts(C.byref(o), 100)
    assert o.max_newton == 8 and o.maxit == 10000 and abs(o.stop_lambda_tol - 0.025) < 1e-15
    assert o.ls_beta == 0.5 and o.ls_c1 == 0.1 and o.finalize_theta == 0.9


@pytest.mark.parametrize("geom", ["fem1d_5nodes", "fem2d_P2_quickstart", "fem2d_P1_L2", "fem2d_P2_L2", "fem3d_k1_L2"])
def test_plan_pattern_bit_exact(geom):
    prob = default_problem(geom, 1.0)
    for M in prob.M:
        g = M.geometry
        D_var = [v for (v, _) in M.D]
        for J in range(len(M.R_fine)):
            ptr, ind = native.plan_pattern(sp.csr_matrix(M.R_fine[J]), g.N, g.V, M.nu, D_var)
            optr, oind = O.hessian_pattern(M, J)
            assert np.array_equal(ptr, optr) and np.array_equal(ind, oind)


@pytest.mark.parametrize("geom", ["fem1d_5nodes", "fem2d_P2_quickstart", "fem2d_P1_L2", "fem2d_P2_L2", "fem3d_k1_L2", "spectral1d_n5", "spectral2d_n5"])
def test_level_transfers_recovered_from_R_fine(geom):
    """The reference keeps only the composed R_fine[l] (src/multigrid.jl:166-170); the library recovers the level transfers
    with R_fine[l] = R_fine[l+1] T[l] (mgbx_amg.T == NULL).  Checked against the ladder the host mirror retains, for both
    AMGs (main, feasibility) of every discretisation family: selector rows (FEM) and matching columns (spectral)."""
    prob = default_problem(geom, 1.0)
    for M in prob.M:
        for l in range(len(M.R_fine) - 1):
            Rn, Rc = sp.csr_matrix(M.R_fine[l + 1]), sp.csr_matrix(M.R_fine[l])
            T = native.recover_transfer(Rn, Rc)
            assert T.shape == (Rn.shape[1], Rc.shape[1])
            assert abs(Rn @ T - Rc).max() <= 1e-13 * max(1.0, abs(Rc).max())
            d = abs(T - sp.csr_matrix(M.T[l]))
            assert (d.max() if d.nnz else 0.0) <= 1e-13


def test_level_transfer_recovery_fallbacks_and_errors():
    rng = np.random.default_rng(0)
    # no selector rows, no matching columns (a smoothed-aggregation-like prolongation): dense normal equations
    Rn = sp.random(60, 12, density=0.5, random_state=1, format="csr") + sp.csr_matrix(np.ones((60, 12)) * 0.01)
    T0 = sp.random(12, 5, density=0.4, random_state=2, format="csr")
    T = native.recover_transfer(sp.csr_matrix(Rn), sp.csr_matrix(Rn @ T0))
    assert abs(T - T0).max() < 1e-10
    # a coarse space that is not nested in the fine one is refused
    with pytest.raises(native.MgbxError) as e:
        native.recover_transfer(sp.csr_matrix(Rn), sp.csr_matrix(rng.normal(size=(60, 3))))
    assert e.value.code == native.ERR_ARG and "nested" in str(e.value)


def test_no_gpu_is_a_loud_error():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    prob = default_problem("fem1d_3nodes", 1.0)
    with pytest.raises(native.MgbxError) as e:
        native.Handle(prob)
    assert e.value.code == native.ERR_CUDA
    assert "no CPU fallback" in str(e.value)


def test_solve_kernel_other_than_2_is_refused():
    """k_pcg2 is the only solve kernel: any other mgbx_config.persistent is an argument error, checked before the device."""
    prob = default_problem("fem1d_3nodes", 1.0)
    for persistent in (0, 1, 3):
        with pytest.raises(native.MgbxError) as e:
            native.Handle(prob, persistent=persistent)
        assert e.value.code == native.ERR_ARG
        assert "persistent" in str(e.value)


def test_bad_arguments_are_reported():
    # column index out of range in R
    R = sp.csr_matrix(np.eye(4))
    keep = native._Keep()
    Rc = keep.csr(R)
    Rc.cols = 2
    nnz = C.c_int64()
    dv = np.zeros(1, np.int32)
    rc = native.lib().mgbx_plan_pattern(C.byref(Rc), 2, 2, 1, 1, native._ptr(dv, native.c_i32p), C.byref(nnz), None, None)
    assert rc == native.ERR_ARG
    assert b"out of range" in native.lib().mgbx_last_error(None)


def test_ctypes_layouts_match_the_c_header(tmp_path):
    """sizeof / offsetof of every struct that crosses the ABI, computed by the C compiler from include/mgbx.h, against the
    ctypes mirrors in native.py (guards against silent ABI drift between the header, the library and the binding)."""
    import subprocess
    structs = {"mgbx_csr": native.Csr, "mgbx_piece": native.Piece, "mgbx_convex": native.Convex, "mgbx_amg": native.Amg,
               "mgbx_problem": native.Problem, "mgbx_config": native.Config, "mgbx_step_opts": native.StepOpts,
               "mgbx_step_result": native.StepResult, "mgbx_scalars_out": native.ScalarsOut, "mgbx_solver_info_t": native.SolverInfo}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "mgbx.h"', 'int main(void) {']
    for cname, ct in structs.items():
        lines.append('  printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in ct._fields_:
            lines.append('  printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines += ['  return 0;', '}']
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, ct in structs.items():
        assert int(out[cname]) == C.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert int(out["%s.%s" % (cname, fname)]) == getattr(ct, fname).offset, (cname, fname)


def test_kronecker_structure_of_the_spectral2d_operators_and_prolongations():
    """mgbx_kron_factor (host-only): the test mgbx_create applies before assembling R'HR sum-factorised.  spectral2d's operators are
    kron(DX, I), kron(I, DX), kron(I, I) and its prolongations kron(R1, R1) (src/spectral2d.jl:22-35): every one must be recognised
    and reproduced to 1e-12; spectral1d's dense matrices and a perturbed product must be rejected; and the sum-factorised formula for
    one block of R'HR must equal the unstructured product (NumPy emulation of dense_kernels.cuh k_kron_w + GEMM + k_kron_scatter)."""
    from mgbx import geometry as G, hierarchy as H
    n1 = 7
    g = G.spectral2d(n=n1)
    mg = H.amg(g)
    facs = {}
    for name in ("id", "dx", "dy"):
        D = np.asarray(g.operators[name][0])
        out = native.kron_factor(D, n1, n1, n1, n1)
        assert out is not None, name
        assert np.abs(np.kron(out[0], out[1]) - D).max() <= 1e-12 * np.abs(D).max()
        facs[name] = out
    Rf = {}
    for X in ("dirichlet", "full"):
        for R in mg.R[X]:
            R = np.asarray(R)
            c = int(round(np.sqrt(R.shape[1])))
            if c == 0 or c * c != R.shape[1]:
                continue
            out = native.kron_factor(R, n1, n1, c, c)
            assert out is not None, (X, R.shape)
            assert np.abs(np.kron(out[0], out[1]) - R).max() <= 1e-12 * np.abs(R).max()
            Rf[X] = (R, out)
    rng = np.random.default_rng(0)
    bad = np.kron(rng.normal(size=(3, 2)), rng.normal(size=(4, 5)))
    assert native.kron_factor(bad, 3, 4, 2, 5) is not None
    bad[5, 7] += 1e-6
    assert native.kron_factor(bad, 3, 4, 2, 5) is None
    g1 = G.spectral1d(n=16)
    assert native.kron_factor(np.asarray(g1.operators["dx"][0]), 4, 4, 4, 4) is None
    assert native.kron_factor(np.zeros((4, 4)), 2, 2, 2, 2) is None
    # one block of R'HR: sum over (j, k) in {id, dx, dy}^2 of (D_j R)' diag(h_jk) (D_k R), unstructured vs sum-factorised
    R, (Ra, Rb) = Rf["dirichlet"]
    c = Ra.shape[1]
    ops = ["id", "dx", "dy"]
    h = {(j, k): rng.normal(size=n1 * n1) for j in range(3) for k in range(j, 3)}
    ref = np.zeros((c * c, c * c))
    for j in range(3):
        for k in range(3):
            hv = h[(min(j, k), max(j, k))]
            Dj, Dk = np.asarray(g.operators[ops[j]][0]), np.asarray(g.operators[ops[k]][0])
            ref += (Dj @ R).T @ (hv[:, None] * (Dk @ R))
    P = [facs[o][0] @ Ra for o in ops]          # n1 x c  (slow index)
    Q = [facs[o][1] @ Rb for o in ops]          # n1 x c  (fast index)
    # scale ambiguity of the factor pairs cancels in P (x) Q only if both come from the same factorisation: check that first
    for o, (A, B) in facs.items():
        assert np.abs(np.kron(A @ Ra, B @ Rb) - np.asarray(g.operators[o][0]) @ R).max() <= 1e-11
    K = 9 * n1
    AA = np.zeros((c * c, K))
    W = np.zeros((c * c, K))
    col = 0
    for j in range(3):
        for k in range(3):
            hv = h[(min(j, k), max(j, k))].reshape(n1, n1)          # node q = e * n1 + f
            for e in range(n1):
                AA[:, col * n1 + e] = np.outer(P[j][e], P[k][e]).reshape(-1)                      # [(i, l)]
                W[:, col * n1 + e] = (Q[j].T @ (hv[e][:, None] * Q[k])).reshape(-1)              # [(i', l')]
            col += 1
    Cm = AA @ W.T                                                    # [(i, l), (i', l')]
    out = Cm.reshape(c, c, c, c).transpose(0, 2, 1, 3).reshape(c * c, c * c)   # -> [(i, i'), (l, l')]
    assert np.abs(out - ref).max() <= 1e-10 * np.abs(ref).max()


def test_cpp_ruge_stuben_is_bitwise_the_host_mirror():
    """mgbx_rs_* (csrc/host_amg.hpp): the classical Ruge-Stueben hierarchy in C++ against hierarchy.ruge_stuben (numba) -- the same
    number of levels and bitwise the same prolongations (pattern and values) on 2-D P1 / P2, 3-D Q1 / Q2 stiffness matrices and on a
    random SPD matrix with positive off-diagonals; then whole amg() hierarchies built on either implementation are identical."""
    import scipy.sparse as sp
    from mgbx import geometry as G, hierarchy as H

    def same(Pa, Pb):
        assert len(Pa) == len(Pb), (len(Pa), len(Pb))
        for a, b in zip(Pa, Pb):
            a, b = sp.csr_matrix(a), sp.csr_matrix(b)
            a.sort_indices()
            b.sort_indices()
            assert a.shape == b.shape
            assert np.array_equal(a.indptr, b.indptr) and np.array_equal(a.indices, b.indices)
            assert np.array_equal(a.data, b.data)

    captured = []
    for g in (G.subdivide(G.fem2d_P1(), 5), G.subdivide(G.fem2d_P2(), 3), G.structured_box(3, 7, k=1), G.subdivide(G.fem3d(k=2), 3),
              G.structured_triangles(11)):
        H.amg(g, prolongator=lambda K: (captured.append(sp.csr_matrix(K)), H.ruge_stuben(K, max_coarse=2))[1])
    assert len(captured) >= 8
    for K in captured:
        same(native.ruge_stuben(K, max_coarse=2), H.ruge_stuben(K, max_coarse=2))
    rng = np.random.default_rng(4)
    R = sp.random(300, 300, density=0.02, random_state=5, format="csr")
    K = (R + R.T + sp.identity(300) * 3.0).tocsr()
    K.data[::7] *= -1.0
    K = (K + K.T).tocsr()
    same(native.ruge_stuben(K, max_coarse=10, theta=0.5), H.ruge_stuben(K, max_coarse=10, theta=0.5))
    # whole hierarchies
    g = G.structured_box(3, 6, k=1)
    ma, mb = H.amg(g), H.amg(g, prolongator=H.amg_ruge_stuben_native())
    for X in ma.R:
        same(ma.R[X], mb.R[X])
        same(ma.T[X], mb.T[X])
