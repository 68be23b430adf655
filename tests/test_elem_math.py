"""CPU check of the element-local elimination of a slack (csrc/elem_schur.cuh, __host__ __device__) against 50-digit arithmetic
-- no GPU needed.  One element of the default problem family with its slack in :broken_P1: p = 6 (pure P2, the corners masked,
P_e the identity on the midpoints) and p = 7 (P2 with bubble, every node weighted, P_e 7 x 3), one Euclidean-power cone per
node approaching its boundary (rho = s^2 - |D u|^2 from 1 down to 1e-9), barrier weights spread over 16 orders of magnitude.
The shim under tests/hostcheck is test infrastructure only."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SLOT = np.array([[1, -1, 1], [1, 0, 0], [1, 1, -1], [0, 1, 0], [-1, 1, 1], [0, 0, 1]], float)   # fem2d_P2.jl:355-380
DIM = 2
f64p = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    src = os.path.join(HERE, "hostcheck", "elem_check.cpp")
    so = str(tmp_path_factory.mktemp("elem_check") / "_elem_check.so")
    subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", src, "-o", so])
    lib = C.CDLL(so)
    lib.hostcheck_elem_schur.argtypes = [C.c_int, C.c_int, C.c_int, f64p, f64p, f64p, f64p, C.c_double, C.c_double, C.c_int, f64p, f64p]
    lib.hostcheck_elem_backsubst.argtypes = [C.c_int, C.c_int, C.c_int, f64p, f64p, f64p, f64p, C.c_double, C.c_double, f64p, f64p, f64p,
                                             f64p]
    return lib


def ptr(a):
    return a.ctypes.data_as(f64p)


def element(p, rho, seed):
    """Inputs of one element: P (p x 3), operators D (DIM blocks, column-major p x p), node inputs Z = (D_1 u, D_2 u, s), weights.
    D u is drawn on a 2^-20 grid with |D u| >= 1 so that |D u|^2 is exact in double precision and rho = s^2 - |D u|^2 is the
    exact difference of the inputs the reference below sees (Sterbenz); s^2 is formed as exp(2 log s), as the kernels do."""
    rng = np.random.default_rng(seed)
    P = SLOT.copy() if p == 6 else np.vstack([SLOT, [1 / 3, 1 / 3, 1 / 3]])
    D = rng.normal(size=(DIM, p, p))
    Z = np.zeros((p, DIM + 1))
    for i in range(p):
        w = np.round(rng.uniform(0.8, 1.4, size=DIM) * 2 ** 20) / 2 ** 20
        Z[i, :DIM] = w
        Z[i, DIM] = math.sqrt(float(w @ w) + rho * rng.uniform(0.5, 2.0))
    sc = 10.0 ** (-16.0 * rng.random(p))
    sc[np.argmax(sc)] = 1.0
    sc[np.argmin(sc)] = 1e-16
    if p == 6:
        sc[[0, 2, 4]] = 0.0          # masked corners (zero quadrature weight)
    return P, np.ascontiguousarray(D), Z, sc


def exact(P, D, Z, sc, gc=None, du=None):
    """H_uu - H_us H_ss^-1 H_su (and the back-substitution) at 50 digits from the same double inputs (alpha = 2, mu = 0)."""
    import mpmath as mp
    mp.mp.dps = 50
    p, nc = P.shape
    Huu = mp.zeros(p, p)
    Hus = mp.zeros(p, nc)
    Hss = mp.zeros(nc, nc)
    q = []
    for i in range(p):
        w = [mp.mpf(float(Z[i, a])) for a in range(DIM)]
        s = mp.mpf(float(Z[i, DIM]))
        sa = mp.mpf(math.exp(2.0 * math.log(float(Z[i, DIM]))))     # s^alpha as the kernels form it
        r = sa - sum(x * x for x in w)
        c = mp.mpf(float(sc[i]))
        hss = c * (4 * (sa / s) ** 2 / r ** 2 - 2 * (sa / s) / s / r)
        hws = [c * (-4 * (sa / s) * w[a] / r ** 2) for a in range(DIM)]
        hww = [[c * (4 * w[a] * w[b] / r ** 2 + (2 / r if a == b else 0)) for b in range(DIM)] for a in range(DIM)]
        Di = [[mp.mpf(float(D[a, c2, i])) for c2 in range(p)] for a in range(DIM)]   # row i of D_a (column-major blocks)
        q.append((hws, Di))
        for r1 in range(p):
            for c1 in range(p):
                Huu[r1, c1] += sum(Di[a][r1] * hww[a][b] * Di[b][c1] for a in range(DIM) for b in range(DIM))
            for k in range(nc):
                Hus[r1, k] += sum(Di[a][r1] * hws[a] for a in range(DIM)) * mp.mpf(float(P[i, k]))
        for k in range(nc):
            for l in range(nc):
                Hss[k, l] += mp.mpf(float(P[i, k])) * hss * mp.mpf(float(P[i, l]))
    Hinv = Hss ** -1
    S = Huu - Hus * Hinv * Hus.T
    dc = None
    if gc is not None:
        g, u = mp.matrix([mp.mpf(float(x)) for x in gc]), mp.matrix([mp.mpf(float(x)) for x in du])
        dc = Hinv * (g - Hus.T * u)
        # componentwise size of what the solve combines, |H_ss^-1| (|g_c| + |H_su| |du|): forming g_c - H_su du rounds at that scale
        ab = lambda M: mp.matrix([[abs(M[i, j]) for j in range(M.cols)] for i in range(M.rows)])
        dc = (dc, ab(Hinv) * (ab(g) + ab(Hus.T) * ab(u)))
    return S, dc


def shim_schur(shim, P, D, Z, sc, stable):
    p, nc = P.shape
    H = np.zeros((p, p))
    Rf = np.zeros(nc * (nc + 1) // 2 + nc)
    Pc, Dc, Zc, scc = (np.ascontiguousarray(a, dtype=float) for a in (P, D, Z, sc))
    assert shim.hostcheck_elem_schur(p, nc, DIM, ptr(Pc), ptr(Dc), ptr(Zc), ptr(scc), 1.0, 0.0, stable, ptr(H), ptr(Rf)) == 0
    return H, Rf


def mp_rel(H, S):
    import mpmath as mp
    p = H.shape[0]
    num = mp.sqrt(sum((mp.mpf(float(H[r, c])) - S[r, c]) ** 2 for r in range(p) for c in range(p)))
    den = mp.sqrt(sum(S[r, c] ** 2 for r in range(p) for c in range(p)))
    return float(num / den)


@pytest.mark.parametrize("p", [6, 7])
def test_element_schur_complement_keeps_its_digits(shim, p):
    """The closed-form node-local part plus Y'Y holds the condensed element block to 1e-10 relative at every rho; the plain
    subtraction H_uu - H_us H_ss^-1 H_su in double precision does not once the cone is approached (so the check discriminates)."""
    worst_plain = worst_stable = 0.0
    for k, rho in enumerate([1.0, 1e-3, 1e-5, 1e-7, 1e-9]):
        P, D, Z, sc = element(p, rho, 100 * p + k)
        S, _ = exact(P, D, Z, sc)
        e_st = mp_rel(shim_schur(shim, P, D, Z, sc, 1)[0], S)
        e_pl = mp_rel(shim_schur(shim, P, D, Z, sc, 0)[0], S)
        print("p=%d rho=%.0e: rel err stable %.1e, plain subtraction %.1e" % (p, rho, e_st, e_pl))
        assert e_st <= 1e-10, (p, rho, e_st)
        worst_plain, worst_stable = max(worst_plain, e_pl), max(worst_stable, e_st)
    assert worst_plain > 1e-9 and worst_plain > 1e5 * worst_stable, (worst_plain, worst_stable)


@pytest.mark.parametrize("p", [6, 7])
def test_element_back_substitution(shim, p):
    """dc = H_ss^-1 (g_c - H_su du) through the stored factor R of W = A^{1/2} P, against 50 digits.  The difference
    g_c - H_su du is formed in double precision, as in k_backsubst for a node-local slack: each component is held to a small
    multiple of eps times the size of what it combines (|H_ss^-1| (|g_c| + |H_su| |du|)), relative to itself."""
    rng = np.random.default_rng(p)
    for k, rho in enumerate([1.0, 1e-3, 1e-5, 1e-7, 1e-9]):
        P, D, Z, sc = element(p, rho, 200 * p + k)
        _, Rf = shim_schur(shim, P, D, Z, sc, 1)
        gc, du = rng.normal(size=3), rng.normal(size=p)
        _, (dce, size) = exact(P, D, Z, sc, gc, du)
        dc = np.zeros(3)
        Pc, Zc, scc = (np.ascontiguousarray(a, dtype=float) for a in (P, Z, sc))
        assert shim.hostcheck_elem_backsubst(p, 3, DIM, ptr(Pc), ptr(D), ptr(Zc), ptr(scc), 1.0, 0.0, ptr(Rf), ptr(gc), ptr(du), ptr(dc)) == 0
        err = max(abs(float(dce[i]) - dc[i]) / float(size[i]) for i in range(3))
        rel = max(abs(float(dce[i]) - dc[i]) / abs(float(dce[i])) for i in range(3))
        print("p=%d rho=%.0e: back-substitution error / (|H_ss^-1| (|g_c| + |H_su| |du|)) %.1e, componentwise rel %.1e" % (p, rho, err, rel))
        assert err <= 64 * np.finfo(float).eps, (p, rho, err)
