"""The dense direct Newton solves and the FP64 DMMA GEMM against extended-precision references.

The kernels of csrc/solver_kernels.cuh and csrc/dense_kernels.cuh are driven one by one through the harness
tests/devcheck/dense_check.cu (the engine's grids and shared-memory limits, host arrays in and out), and the engine's own
launch sequence through the C ABI.  Every reference is computed on the CPU in np.longdouble (80-bit on x86-64).

Test matrices have a known spectrum: A = P C' diag(lam) C P' with C the orthonormal DCT-II matrix and P a random
permutation, rounded to float64, so kappa(A) = max|lam| / min|lam| and A^{-1} = P C' diag(1/lam) C P' are known without
a factorisation (O(m^2 log m) to build, which keeps the 8192-unknown cases cheap).  SPD inputs are then scaled by a
diagonal S with entries from 1e-8 to 1e8, B = S A S, which only the kernels' 1/sqrt(b_ii) scaling makes solvable to full
accuracy.  Errors are therefore measured on the equilibrated system  Bt = D B D,  D = diag(b_ii)^(-1/2),  in the
infinity norm:
    backward error  |D (b - B x)| / (|Bt| |D^-1 x| + |D b|)      <= 32 m eps
    forward error   |D^-1 (x - x_ref)| / |D^-1 x_ref|            <= 10 kappa eps
with kappa = kappa(A) max(a_ii) / min(a_ii), an upper bound of kappa_2(Bt) (Bt is the Jacobi-scaled A)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import scipy.fft as fft
import scipy.sparse as sp
import scipy.sparse.linalg as spl

import mgb_oracle as O
from mgbx import geometry as G, hierarchy as H, native, problem as P

pytestmark = pytest.mark.gpu

EPS = np.finfo(float).eps
LD = np.longdouble
HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "multigridbarrier.jl_b200", "csrc")
SRC = os.path.join(HERE, "devcheck", "dense_check.cu")
SO = os.path.join(HERE, "devcheck", "_dense_check.so")
c_f64p, c_i64p, c_i32p = C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int32)


# ------------------------------------------------------------------------------------------------ harness
@pytest.fixture(scope="module")
def dc():
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("solver_kernels.cuh", "dense_kernels.cuh", "device_common.cuh", "node_barrier.cuh")]
    if (not os.path.exists(SO)) or os.path.getmtime(SO) < max(os.path.getmtime(f) for f in deps):
        from mgbx import build as B
        subprocess.check_call([B.nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-shared",
                               "-Xcompiler", "-fPIC,-Wall", "-I", CSRC, SRC, "-o", SO])
    lib = C.CDLL(SO)
    lib.dc_error_string.restype = C.c_char_p
    lib.dc_error_string.argtypes = [C.c_int]
    lib.dc_dgemm_nt.argtypes = [C.c_int, C.c_int, C.c_int, c_f64p, C.c_int64, c_f64p, C.c_int64, c_f64p, c_f64p, C.c_int64,
                                C.c_int, C.c_double, C.c_int]
    csr = [C.c_int64, c_i64p, c_i32p, c_f64p]
    lib.dc_dense_solve_small.argtypes = csr + [c_f64p, c_f64p, c_i32p]
    lib.dc_chol_factor_solve.argtypes = csr + [c_f64p, c_f64p, C.c_int]
    lib.dc_coarse_inverse.argtypes = csr + [c_f64p]
    return lib


def _p(a, t=c_f64p):
    return None if a is None else a.ctypes.data_as(t)


def _ok(lib, rc):
    assert rc == 0, lib.dc_error_string(rc).decode()


def _csr(A, drop=()):
    """Dense symmetric A as CSR arrays (int64 row pointers, int32 columns); entries (i, i) for i in drop are left out."""
    if not drop and A.shape[0] > 512:     # dense pattern without building a scipy copy of the big matrices
        m = A.shape[0]
        return (np.arange(0, m * m + 1, m, dtype=np.int64), np.tile(np.arange(m, dtype=np.int32), m),
                np.ascontiguousarray(A).reshape(-1))
    M = sp.csr_matrix(A)
    M.sort_indices()
    for i in drop:
        M[i, i] = 0.0
    M.eliminate_zeros()
    return M.indptr.astype(np.int64), M.indices.astype(np.int32), M.data.astype(np.float64)


def gemm(lib, A, B, s, C0, accumulate, alpha, M, N, K, inplace=False):
    C = np.array(C0, dtype=np.float64, copy=True)
    _ok(lib, lib.dc_dgemm_nt(M, N, K, _p(A), A.shape[1], _p(B), B.shape[1], _p(s), _p(C), C.shape[1], accumulate, alpha,
                             1 if inplace else 0))
    return C


def solve_small(lib, A, b, drop=()):
    ptr, idx, val = _csr(A, drop)
    x = np.empty(A.shape[0])
    info = np.full(1, -7, np.int32)
    _ok(lib, lib.dc_dense_solve_small(A.shape[0], _p(ptr, c_i64p), _p(idx, c_i32p), _p(val), _p(b), _p(x), _p(info, c_i32p)))
    return x, int(info[0])


def chol_solve(lib, A, b, refine):
    ptr, idx, val = _csr(A)
    x = np.empty(A.shape[0])
    _ok(lib, lib.dc_chol_factor_solve(A.shape[0], _p(ptr, c_i64p), _p(idx, c_i32p), _p(val), _p(b), _p(x), 1 if refine else 0))
    return x


def coarse_inverse(lib, A):
    ptr, idx, val = _csr(A)
    m = A.shape[0]
    Minv = np.empty((m, m))
    _ok(lib, lib.dc_coarse_inverse(m, _p(ptr, c_i64p), _p(idx, c_i32p), _p(val), _p(Minv)))
    return Minv


# ------------------------------------------------------------------------------------------------ test matrices
class Spectral:
    """A = P C' diag(lam) C P' (float64, exactly symmetric) with its exact inverse as an operator; optionally B = S A S."""

    def __init__(self, m, kappa, rng, neg=0, scale=False):
        lam = np.geomspace(1.0, 1.0 / kappa, m) if m > 1 else np.ones(1)
        if neg:
            lam[rng.choice(m, neg, replace=False)] *= -1.0
        rng.shuffle(lam)
        self.lam, self.perm = lam, rng.permutation(m)
        self.kappa = float(np.abs(lam).max() / np.abs(lam).min())
        X = fft.idct(np.diag(lam), type=2, norm="ortho", axis=0, workers=-1)          # C' diag(lam)
        A = fft.idct(np.ascontiguousarray(X.T), type=2, norm="ortho", axis=0, workers=-1)   # C' diag(lam) C
        A = A[np.ix_(self.perm, self.perm)]
        A += A.T
        A *= 0.5
        self.s = 10.0 ** rng.uniform(-8, 8, m) if scale else np.ones(m)
        if scale:
            A *= self.s[:, None]
            A *= self.s[None, :]
        self.B = A
        dg = np.abs(np.diag(A))
        self.d = 1.0 / np.sqrt(np.where(dg > 0, dg, 1.0))                 # the kernels' scaling (1 for a non-positive diagonal)
        a = dg / self.s ** 2
        self.kappa_eq = self.kappa * a.max() / a.min() if neg == 0 else self.kappa

    def inv_apply(self, r):
        """B^{-1} r in float64 through the known spectrum (used only for the O(eps) correction of the reference)."""
        u = np.empty_like(r)
        u[self.perm] = r / self.s
        v = fft.idct(fft.dct(u, type=2, norm="ortho") / self.lam, type=2, norm="ortho")
        return v[self.perm] / self.s


def ld_matvec(A, x, rows=256):
    """A x in long double, in row blocks (the long double copy of an 8192^2 matrix would need 1 GB)."""
    xl = x.astype(LD)
    out = np.empty(A.shape[0], LD)
    for i in range(0, A.shape[0], rows):
        out[i:i + rows] = A[i:i + rows].astype(LD) @ xl
    return out


def ld_lu_solve(A, b):
    """x = A^{-1} b by Gaussian elimination with partial pivoting in long double (small m)."""
    S = A.astype(LD)
    r = b.astype(LD).copy()
    m = S.shape[0]
    for k in range(m):
        p = k + int(np.argmax(np.abs(S[k:, k])))
        if p != k:
            S[[k, p]] = S[[p, k]]
            r[[k, p]] = r[[p, k]]
        l = S[k + 1:, k] / S[k, k]
        S[k + 1:, k:] -= np.outer(l, S[k, k:])
        r[k + 1:] -= l * r[k]
    x = np.zeros(m, LD)
    for k in range(m - 1, -1, -1):
        x[k] = (r[k] - S[k, k + 1:] @ x[k + 1:]) / S[k, k]
    return x


def rhs_for(T, rng):
    """b = B x* with x* = D y*, y* ~ N(0, 1): the right-hand side rounded to float64, and the exact solution of the rounded
    system in long double, x* + B^{-1} (b - B x*) (the correction is O(kappa eps) and needs no more than a few digits)."""
    xs = T.d * rng.normal(size=T.B.shape[0])
    bl = ld_matvec(T.B, xs)
    b = bl.astype(np.float64)
    return b, xs.astype(LD) + T.inv_apply((b.astype(LD) - bl).astype(np.float64)).astype(LD)


def errors(Bm, d, b, x, xref):
    """(backward, forward) errors of x on the equilibrated system D B D (infinity norms), residual in long double."""
    r = b.astype(LD) - ld_matvec(Bm, x)
    Bt_inf = float(np.max(np.abs(Bm * d[:, None] * d[None, :]).sum(axis=1)))
    y = x / d
    bwd = float(np.max(np.abs(r * d))) / (Bt_inf * np.max(np.abs(y)) + np.max(np.abs(b * d)))
    yref = xref / d.astype(LD)
    fwd = float(np.max(np.abs(y.astype(LD) - yref)) / np.max(np.abs(yref)))
    return bwd, fwd


# ------------------------------------------------------------------------------------------------ GEMM
GEMM_DIMS = (1, 7, 8, 15, 16, 17, 63, 64, 65, 129)


def gemm_check(C, C0, A, B, s, M, N, K, accumulate, alpha):
    """Entrywise |C - C_ref| <= 4 K eps (|alpha| |A| |s| |B|) + 2 eps |C_ref| against the long-double product; padding columns
    (j >= N) untouched."""
    sv = np.ones(K) if s is None else s[:K]
    Al, Bl = A[:M, :K].astype(LD) * sv.astype(LD), B[:N, :K].astype(LD)
    ref = LD(alpha) * (Al @ Bl.T) + (C0[:M, :N].astype(LD) if accumulate else 0)
    bound = 4 * K * EPS * abs(alpha) * (np.abs(A[:M, :K]) * np.abs(sv)) @ np.abs(B[:N, :K]).T + 2 * EPS * np.abs(ref.astype(np.float64))
    err = np.abs(C[:M, :N].astype(LD) - ref).astype(np.float64)
    assert np.all(err <= bound), (M, N, K, accumulate, alpha, float(np.max(err / np.maximum(bound, 1e-300))))
    assert np.array_equal(C[:, N:], C0[:, N:]), "k_dgemm_nt wrote outside the N columns of C"
    return float(np.max(err / np.maximum(bound / (4 * max(K, 1)), 1e-300)))    # error in units of eps |A||s||B|


def test_dgemm_nt_all_shapes(dc):
    """Every (M, N, K) of GEMM_DIMS^3 with row strides beyond the logical width, with and without the k-scaling s (with zeros
    in s), overwrite and accumulate, alpha = 1 and -1."""
    rng = np.random.default_rng(1)
    worst = 0.0
    q = 0
    for M in GEMM_DIMS:
        for N in GEMM_DIMS:
            for K in GEMM_DIMS:
                q += 1
                A = rng.normal(size=(M, K + 3))
                B = rng.normal(size=(N, K + 5))
                s = None
                if q % 3:
                    s = rng.uniform(0.5, 2.0, K + 2) * 10.0 ** rng.integers(-3, 4, K + 2)
                    s[rng.random(K + 2) < 0.2] = 0.0
                acc, alpha = q % 2, (-1.0 if q % 4 >= 2 else 1.0)
                C0 = rng.normal(size=(M, N + 7))
                C = gemm(dc, A, B, s, C0, acc, alpha, M, N, K)
                worst = max(worst, gemm_check(C, C0, A, B, s, M, N, K, acc, alpha))
    print("dgemm_nt: largest entrywise error %.2f eps |A||s||B|" % worst)


@pytest.mark.parametrize("m,k0,nb", [(200, 0, 64), (129, 0, 64), (257, 128, 64), (150, 64, 22)])
def test_dgemm_nt_in_place_panel(dc, m, k0, nb):
    """The panel step of the blocked Cholesky, L21 = A21 inv(L11)', in place (C = A = A21 with the row stride m of the dense
    matrix), with a ragged last row tile (rem = m - k0 - 64 not a multiple of 64) and with a ragged panel width: A21 is right,
    and nothing outside it changes."""
    rng = np.random.default_rng(m + nb)
    rem = m - k0 - nb
    rows = rng.normal(size=(rem, m))                  # the rows of A21 in the dense matrix
    Li = np.zeros((64, 64))                           # inv(L11) as k_chol_diag_inv leaves it: zero outside nb x nb
    Li[:nb, :nb] = np.tril(rng.normal(size=(nb, nb)))
    # A21 starts at column k0 of the first row: the harness copies rem * m doubles from there
    Cpad = np.concatenate([rows.reshape(-1)[k0:], np.zeros(k0)]).reshape(rem, m)
    res = gemm(dc, Cpad, Li, None, Cpad, 0, 1.0, rem, nb, nb, inplace=True)
    A21 = rows[:, k0:k0 + nb]
    ref = A21.astype(LD) @ Li[:nb, :nb].astype(LD).T
    bound = 4 * nb * EPS * np.abs(A21) @ np.abs(Li[:nb, :nb]).T
    assert np.all(np.abs(res[:, :nb].astype(LD) - ref).astype(np.float64) <= bound)
    assert np.array_equal(res[:, nb:], Cpad[:, nb:])


# ------------------------------------------------------------------------------------------------ small solve (m <= 128)
SMALL_M = (1, 2, 31, 32, 33, 63, 64, 65, 127, 128)
KAPPAS = (1e2, 1e8, 1e12)


def _gates(bwd, fwd, m, kappa, what):
    assert bwd <= 32 * m * EPS, (what, "backward error %.3g > 32 m eps" % bwd)
    assert fwd <= 10 * kappa * EPS, (what, "forward error %.3g > 10 kappa eps (kappa %.3g)" % (fwd, kappa))


@pytest.mark.parametrize("m", SMALL_M)
def test_dense_solve_small_spd(dc, m):
    """k_dense_solve_small on badly scaled SPD inputs: the scaled Cholesky runs (info 0) and solves to the gates."""
    rng = np.random.default_rng(10 + m)
    worst = [0.0, 0.0]
    for kappa in KAPPAS:
        T = Spectral(m, kappa, rng, scale=True)
        b, _ = rhs_for(T, rng)
        xref = ld_lu_solve(T.B, b)
        x, info = solve_small(dc, T.B, b)
        assert info == 0, (m, kappa)
        bwd, fwd = errors(T.B, T.d, b, x, xref)
        _gates(bwd, fwd, m, T.kappa_eq, ("spd", m, kappa))
        worst = [max(worst[0], bwd / EPS), max(worst[1], fwd / (T.kappa_eq * EPS))]
    print("small SPD m=%d: backward %.2f eps, forward %.3f kappa eps" % (m, worst[0], worst[1]))


def _indefinite_case(dc, A, m, drop=(), what=""):
    b = np.random.default_rng(m).normal(size=m)
    Af = A.copy()
    for i in drop:
        Af[i, i] = 0.0
    xref = ld_lu_solve(Af, b)
    x, info = solve_small(dc, A, b, drop)
    assert info == 1, (what, m, info)
    kappa = float(np.linalg.cond(Af))
    one = np.ones(m)
    bwd, fwd = errors(Af, one, b, x, xref)
    _gates(bwd, fwd, m, kappa, (what, m))
    return bwd, fwd / (kappa * EPS)


@pytest.mark.parametrize("m", SMALL_M)
def test_dense_solve_small_indefinite(dc, m):
    """Symmetric indefinite inputs: the Cholesky finds a non-positive pivot and the pivoted elimination runs (info 1),
    against a long-double LU.  Includes a zero first diagonal entry (the first step must swap rows) and a row with no
    diagonal entry in the CSR pattern."""
    rng = np.random.default_rng(20 + m)
    res = []
    for kappa in KAPPAS:
        T = Spectral(m, kappa, rng, neg=max(1, m // 3))
        res.append(_indefinite_case(dc, T.B, m, what="indefinite kappa %g" % kappa))
    if m >= 2:
        T = Spectral(m, 1e4, rng, neg=m // 2)
        A = T.B.copy()
        A[0, 0] = 0.0                              # stored as an explicit zero
        res.append(_indefinite_case(dc, A, m, what="zero first diagonal"))
        res.append(_indefinite_case(dc, T.B, m, drop=(m // 2,), what="no diagonal entry"))
    print("small indefinite m=%d: backward %.2f eps, forward %.3f kappa eps"
          % (m, max(r[0] for r in res) / EPS, max(r[1] for r in res)))


# ------------------------------------------------------------------------------------------------ blocked Cholesky
BLOCKED_M = (129, 191, 192, 193, 255, 256, 257, 1000, 2047, 2048, 2049, 4097, 8191, 8192)


@pytest.mark.parametrize("m", BLOCKED_M)
def test_blocked_cholesky(dc, m):
    """The blocked DMMA Cholesky (k_chol_diag_inv, two k_dgemm_nt per panel, k_chol_solve_blocked) at the panel edges
    m = 64 k +- 1 and up to the direct-solve limit: the factor alone (refinement off) and the engine's solve with one step
    of refinement both meet the gates, and refinement makes the forward error no worse."""
    rng = np.random.default_rng(30 + m)
    # the three conditionings everywhere below 4096 unknowns; above, where one case costs seconds of CPU time, one
    kappas = KAPPAS if m < 4096 else (1e8,)
    for kappa in kappas:
        T = Spectral(m, kappa, rng, scale=True)
        b, xref = rhs_for(T, rng)
        out = []
        for refine in (False, True):
            x = chol_solve(dc, T.B, b, refine)
            assert np.all(np.isfinite(x)), (m, kappa, refine)
            bwd, fwd = errors(T.B, T.d, b, x, xref)
            _gates(bwd, fwd, m, T.kappa_eq, ("blocked", m, kappa, "refined" if refine else "factor only"))
            out.append((bwd, fwd))
        # one refinement step with a working-precision residual (|b - B x| is rounded to eps |B| |x|) leaves a forward
        # error of order kappa eps: no worse than the factor's own, up to that level (measured: up to 0.8 kappa eps)
        assert out[1][1] <= max(out[0][1], T.kappa_eq * EPS), (m, kappa, out)
        print("blocked m=%d kappa=%.0e (eq %.2g): factor bwd %.2f eps fwd %.3f kappa eps | refined bwd %.2f eps fwd %.3f kappa eps"
              % (m, kappa, T.kappa_eq, out[0][0] / EPS, out[0][1] / (T.kappa_eq * EPS), out[1][0] / EPS,
                 out[1][1] / (T.kappa_eq * EPS)))


@pytest.mark.parametrize("m", (129, 193, 1000))
def test_blocked_cholesky_indefinite_is_not_finite(dc, m):
    """k_chol_diag_inv has no pivot guard: an indefinite input gives sqrt of a negative pivot, and the NaN reaches every
    entry of x -- the loud failure Newton's non-finite test relies on, never a finite wrong answer."""
    rng = np.random.default_rng(40 + m)
    for neg in (1, m // 2):
        T = Spectral(m, 1e3, rng, neg=neg)
        b = rng.normal(size=m)
        for refine in (False, True):
            x = chol_solve(dc, T.B, b, refine)
            assert not np.any(np.isfinite(x)), (m, neg, refine, int(np.isfinite(x).sum()))


# ------------------------------------------------------------------------------------------------ coarse inverse
@pytest.mark.parametrize("m", (1, 32, 33, 127, 128))
def test_coarse_inverse(dc, m):
    """k_coarse_inverse (the V-cycle's dense bottom level) on badly scaled SPD inputs: |Mt Bt - I| <= 10 kappa eps on the
    equilibrated system (Mt = D^-1 Minv D^-1), residual in long double; Minv is symmetric to its last bit."""
    rng = np.random.default_rng(50 + m)
    worst = 0.0
    for kappa in KAPPAS:
        T = Spectral(m, kappa, rng, scale=True)
        Minv = coarse_inverse(dc, T.B)
        assert np.all(np.abs(Minv - Minv.T) <= 2 * EPS * np.abs(Minv))    # (s d_i) d_j against (s d_j) d_i
        dl = T.d.astype(LD)
        Mt = Minv.astype(LD) / dl[:, None] / dl[None, :]
        Bt = T.B.astype(LD) * dl[:, None] * dl[None, :]
        R = Mt @ Bt - np.eye(m, dtype=LD)
        err = float(np.max(np.abs(R).sum(axis=1)))
        assert err <= 10 * T.kappa_eq * EPS, (m, kappa, err, T.kappa_eq)
        worst = max(worst, err / (T.kappa_eq * EPS))
    print("coarse inverse m=%d: |Mt Bt - I| %.3f kappa eps" % (m, worst))


def _assert_spd(Minv, what):
    """SPD up to the rounding of the Gram matrix Li' Li that k_coarse_inverse forms: after a decoupled pivot, later positive
    pivots may be tiny, and eigenvalues below m eps |Minv| carry no sign."""
    ev = np.linalg.eigvalsh(0.5 * (Minv + Minv.T))
    assert ev.min() >= -Minv.shape[0] * EPS * np.abs(ev).max() and np.all(np.diag(Minv) > 0), (what, ev.min(), np.abs(ev).max())


@pytest.mark.parametrize("m", (32, 33, 127, 128))
def test_coarse_inverse_non_positive_pivot_stays_finite_spd(dc, m):
    """A non-positive pivot (an indefinite or singular input) must still give a finite SPD matrix: the V-cycle uses Minv as
    a preconditioner, for which any SPD approximation is valid and a non-finite one is fatal."""
    rng = np.random.default_rng(60 + m)
    for neg in (1, m // 4, m // 2):
        T = Spectral(m, 1e3, rng, neg=neg)
        Minv = coarse_inverse(dc, T.B)
        assert np.all(np.isfinite(Minv)), (m, neg)
        _assert_spd(Minv, (m, neg))
    # positive semi-definite with an exactly singular direction: the zero pivot of roundoff size
    T = Spectral(m, 1e3, rng)
    v = rng.normal(size=m)
    v /= np.linalg.norm(v)
    Av = T.B @ v
    A = T.B - np.outer(Av, Av) / (v @ Av)             # A v = 0
    A = 0.5 * (A + A.T)
    Minv = coarse_inverse(dc, A)
    assert np.all(np.isfinite(Minv)), m
    _assert_spd(Minv, m)


# ------------------------------------------------------------------------------------------------ through the C ABI
def _fem1d(m):
    """fem1d with m + 2 nodes: the condensed top system (the slack eliminated node-locally) has m unknowns of u."""
    return P.assemble(H.amg(G.fem1d(nodes=np.linspace(-1, 1, m + 2))), p=1.0)


def _fem2d(L):
    return P.assemble(H.amg(G.subdivide(G.fem2d_P1(), L)), p=1.5)


# (name, problem builder, condensed top size): the fem1d sizes sit on the panel edges, the fem2d P1 levels have 2-D fill
ABI_CASES = {"fem1d_129": (lambda: _fem1d(129), 129), "fem1d_192": (lambda: _fem1d(192), 192), "fem1d_257": (lambda: _fem1d(257), 257),
             "fem1d_2047": (lambda: _fem1d(2047), 2047), "fem1d_2048": (lambda: _fem1d(2048), 2048),
             "fem1d_2049": (lambda: _fem1d(2049), 2049), "fem1d_4097": (lambda: _fem1d(4097), 4097),
             "fem1d_8192": (lambda: _fem1d(8192), 8192),
             "fem2d_P1_L5": (lambda: _fem2d(5), 225), "fem2d_P1_L6": (lambda: _fem2d(6), 961)}


def _condensed_size(prob):
    """Unknowns of the condensed fine-level system: the kept variables, i.e. all but the node-local slack (the last state
    variable, an identity block of the fine prolongation)."""
    M = prob.M[0]
    off = M.var_offsets[len(M.R_fine) - 1]
    return int(off[-2] - off[0])


def _late_ramp_state(prob):
    """Initial state with the slack moved to within 1e-4 (relative) of the cone s >= |q|^p at every node."""
    M = prob.M[0]
    n = M.geometry.n
    z = prob.g.T.reshape(-1).copy()
    Y = O.operators(M).apply(z)
    pc = prob.Q.pieces[0]
    q = Y[:, list(pc.idx[:-1])]
    cone = np.linalg.norm(q, axis=1) ** pc.p
    z[-n:] = cone + 1e-4 * (1.0 + cone)
    return z


def _ld_spmv(Hm, x):
    xl = x.astype(LD)
    prod = Hm.data.astype(LD) * xl[Hm.indices]
    out = np.zeros(Hm.shape[0], LD)
    nz = np.diff(Hm.indptr) > 0
    out[nz] = np.add.reduceat(prod, Hm.indptr[:-1][nz])
    return out


def _kappa_spd(Hm):
    """An upper bound of kappa_2 of the sparse SPD Hessian: the Gershgorin bound of the largest eigenvalue over the
    smallest by shift-invert Lanczos (np.linalg.cond would need a dense SVD of up to 25 000 unknowns)."""
    lmax = float(abs(Hm).sum(axis=1).max())
    lmin = spl.eigsh(Hm.tocsc(), k=1, sigma=0, which="LM", return_eigenvectors=False)[0]
    assert lmin > 0
    return float(lmax / lmin)


@pytest.mark.parametrize("name,route", [(k, "direct") for k in ABI_CASES]
                         + [(k, "fallback") for k, (_, m) in ABI_CASES.items() if 2049 <= m <= 8192])
def test_engine_direct_solve_through_the_c_abi(name, route):
    """Engine::dense_factor / dense_apply / direct_solve in the engine's own launch sequence: mgbx_solve_newton_system with
    condensation on, the condensed top system of the sizes above reached by dense_direct_max >= m (direct) or by a
    one-iteration PCG that falls back to the direct solve (dense_direct_max = 0, pcg_maxit = 1).  Against the full uncondensed
    Hessian solved in float64 plus one long-double refinement, at a moderate t and at a late-ramp point (t = 1e6, slack
    within 1e-4 of the cone) where kappa is large."""
    build, m = ABI_CASES[name]
    prob = build()
    assert _condensed_size(prob) == m
    M = prob.M[0]
    J = len(M.R_fine) - 1
    mf = M.R_fine[J].shape[1]
    cfg = dict(dense_direct_max=8192) if route == "direct" else dict(dense_direct_max=0, pcg_maxit=1, direct_fallback=1)
    rng = np.random.default_rng(m)
    h = native.Handle(prob, condense=1, **cfg)
    try:
        for t, z in ((1.0, None), (1e6, _late_ramp_state(prob))):
            if z is not None:
                h.set_z(z)
            s = np.zeros(mf)
            assert np.isfinite(h.barrier_eval(0, J, t, s, 0))
            g = rng.normal(size=mf)
            x, its = h.solve_newton_system(0, J, t, s, g)
            if route == "direct":
                assert its == 0
            Hm = h.hessian(0, J, t, s).tocsr()
            xr = spl.spsolve(Hm.tocsc(), g)
            r = g.astype(LD) - _ld_spmv(Hm, xr)
            xref = xr.astype(LD) + spl.spsolve(Hm.tocsc(), r.astype(np.float64)).astype(LD)
            kappa = _kappa_spd(Hm)
            fwd = float(np.max(np.abs(x.astype(LD) - xref)) / np.max(np.abs(xref)))
            assert fwd <= 10 * kappa * EPS, (name, route, t, fwd, kappa)
            print("%s %s t=%g m=%d: forward %.3g (%.3g kappa eps, kappa %.2g)" % (name, route, t, m, fwd, fwd / (kappa * EPS), kappa))
    finally:
        h.close()
