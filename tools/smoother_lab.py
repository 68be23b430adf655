"""CPU laboratory for the V-cycle preconditioner of the GPU solve (csrc/pcg2.cu), NumPy/SciPy only.

Runs the CPU oracle on a small 3-D (or 2-D) problem, records the finest-level Newton systems (H, g) along the t-ramp,
condenses the node-local slack exactly as the library does, and counts PCG iterations to a relative residual of 1e-9
for variants of the preconditioner: Chebyshev degree / interval, l1-Jacobi, V- vs W-cycle, symmetric Gauss-Seidel.
Cost column: fine-level mat-vec equivalents per PCG iteration (what the persistent kernel pays per iteration).

    python tools/smoother_lab.py q1c12            # fem3d k=1 on 12^3 hexahedra, p = 1, t0 = 0.01
    python tools/smoother_lab.py p1l5             # fem2d_P1 level 5, p = 1.5

Test/tuning infrastructure: imports oracle/, never used by the product path.
"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

import mgbx  # noqa: F401
import mgb_oracle as O
from mgbx import geometry as G, hierarchy as H, problem as P


def record_systems(prob, kw, every=7, cap=12):
    """Finest-level (H, g) pairs seen by the oracle's Newton iterations."""
    M = prob.M[0]
    Lfine = M.R_fine[-1].shape[1]
    seen = []
    count = [0]
    f1_orig, f2_orig = O.Barrier.f1, O.Barrier.f2

    def f2(self, s, w, c, R, ops, z0):
        Hm = f2_orig(self, s, w, c, R, ops, z0)
        if R.shape[1] == Lfine and R.shape[0] == M.R_fine[-1].shape[0]:
            count[0] += 1
            if count[0] % every == 1 and len(seen) < cap:
                seen.append((sp.csr_matrix(Hm), f1_orig(self, s, w, c, R, ops, z0), float(np.max(np.abs(c)))))
        return Hm

    O.Barrier.f2 = f2
    try:
        O.mgb_solve(prob, **kw)
    finally:
        O.Barrier.f2 = f2_orig
    return seen


def condense(Hm, g, M):
    """Eliminate the node-local slack block (last variable, identity R block): S = Huu - Hus Hss^-1 Hsu."""
    offs = M.var_offsets[-1]
    nu_ = offs[1] - offs[0]
    Huu = Hm[:nu_, :nu_].tocsr()
    Hus = Hm[:nu_, nu_:].tocsr()
    Hss = Hm[nu_:, nu_:].tocsr()
    d = Hss.diagonal()
    assert abs(Hss - sp.diags(d)).sum() < 1e-12 * abs(d).sum(), "slack block is not node-local"
    S = (Huu - Hus @ sp.diags(1.0 / d) @ Hus.T).tocsr()
    gs = g[:nu_] - Hus @ (g[nu_:] / d)
    return S, gs


def transfers(M):
    """Level transfers of the first state variable, fine -> coarse order (T[k]: level k+1 (coarser) -> level k)."""
    Ts = []
    L = len(M.R_fine)
    for l in range(L - 1, 0, -1):
        T = sp.csr_matrix(M.T[l - 1])
        r0, r1 = M.var_offsets[l][0], M.var_offsets[l][1]
        c0, c1 = M.var_offsets[l - 1][0], M.var_offsets[l - 1][1]
        Ts.append(T[r0:r1, c0:c1].tocsr())
    return Ts


class VCycle:
    def __init__(self, A, Ts, smoother="cheb", nu=2, ratio=8.0, gamma=1, coarse_max=128, lam="gershgorin"):
        self.smoother, self.nu, self.ratio, self.gamma = smoother, nu, ratio, gamma
        self.A, self.T = [A.tocsr()], []
        for T in Ts:
            if self.A[-1].shape[0] <= coarse_max:
                break
            if T.shape[0] == T.shape[1] and abs(T - sp.identity(T.shape[0])).sum() == 0:
                continue
            self.T.append(T)
            self.A.append((T.T @ self.A[-1] @ T).tocsr())
        self.bottom = np.linalg.pinv(self.A[-1].toarray()) if self.A[-1].shape[0] <= 4000 else None
        self.diag = [a.diagonal() for a in self.A]
        self.l1 = [np.asarray(abs(a).sum(axis=1)).ravel() for a in self.A]
        if lam == "gershgorin":
            self.lam = [float(np.max(l1 / d)) for l1, d in zip(self.l1, self.diag)]
        elif lam.startswith("power"):   # "power:<iterations>:<safety>": power iterations on D^-1 A from a fixed start vector
            _, nit, safety = (lam.split(":") + ["12", "1.1"])[:3] if lam.count(":") == 2 else ("power", "12", "1.1")
            self.lam = []
            for a, d in zip(self.A, self.diag):
                v = np.cos(0.7 * np.arange(a.shape[0]) ** 1.3) + 0.1
                nv = 1.0
                for _ in range(int(nit)):
                    v = (a @ v) / d
                    nv = np.linalg.norm(v)
                    v /= nv
                self.lam.append(float(safety) * nv)
        elif lam.startswith("scaled"):   # "scaled:<f>": Gershgorin bound times f (unsafe in general; shows the sensitivity)
            f = float(lam.split(":")[1])
            self.lam = [f * float(np.max(l1 / d)) for l1, d in zip(self.l1, self.diag)]
        elif lam == "exact":
            self.lam = [float(spla.eigsh(sp.diags(1 / np.sqrt(d)) @ a @ sp.diags(1 / np.sqrt(d)), k=1, which="LA", return_eigenvectors=False, tol=1e-3)[0])
                        if a.shape[0] > 3 else float(np.max(np.linalg.eigvalsh((a / np.sqrt(np.outer(d, d))).toarray() if sp.issparse(a) else a)))
                        for a, d in zip(self.A, self.diag)]
        self.mv = 0.0   # fine-level mat-vec equivalents

    def _mv(self, k, x):
        self.mv += self.A[k].nnz / self.A[0].nnz
        return self.A[k] @ x

    def smooth(self, k, b, x):
        A, d = self.A[k], self.diag[k]
        if self.smoother == "l1":
            for _ in range(self.nu):
                x = (b / self.l1[k]) if x is None else x + (b - self._mv(k, x)) / self.l1[k]
            return x
        if self.smoother == "sgs":   # symmetric Gauss-Seidel (sequential; a bound on what a point smoother can do)
            Lo = sp.tril(A, format="csr")
            Up = sp.triu(A, format="csr")
            for _ in range(max(1, self.nu // 2)):
                r = b if x is None else b - self._mv(k, x)
                x0 = 0.0 if x is None else x
                y = x0 + spla.spsolve_triangular(Lo, r, lower=True)
                r = b - self._mv(k, y)
                x = y + spla.spsolve_triangular(Up, r, lower=False)
            return x
        lam = self.lam[k]
        a_, b_ = lam / self.ratio, lam
        theta, delta = 0.5 * (a_ + b_), 0.5 * (b_ - a_)
        sigma = theta / delta
        rho = 1.0 / sigma
        dvec = None
        for it in range(self.nu):
            r = b if x is None else b - self._mv(k, x)
            if it == 0:
                dvec = r / d / theta
            else:
                rho_new = 1.0 / (2.0 * sigma - rho)
                dvec = rho_new * rho * dvec + (2.0 * rho_new / delta) * (r / d)
                rho = rho_new
            x = dvec if x is None else x + dvec
        return x

    def cycle(self, k, b):
        if k == len(self.A) - 1:
            if self.bottom is not None:
                return self.bottom @ b
            return self.smooth(k, b, None)
        x = self.smooth(k, b, None)
        for _ in range(self.gamma):
            r = b - self._mv(k, x)
            x = x + self.T[k] @ self.cycle(k + 1, self.T[k].T @ r)
        return self.smooth(k, b, x)

    def __call__(self, r):
        return self.cycle(0, r)


def pcg(A, b, Minv, rtol=1e-9, maxit=500):
    x = np.zeros_like(b)
    r = b.copy()
    z = Minv(r)
    p = z.copy()
    rz = r @ z
    bb = np.sqrt(b @ b)
    for it in range(1, maxit + 1):
        Ap = A @ p
        alpha = rz / (p @ Ap)
        x += alpha * p
        r -= alpha * Ap
        if np.sqrt(r @ r) <= rtol * bb:
            return it
        z = Minv(r)
        rz_new = r @ z
        p = z + (rz_new / rz) * p
        rz = rz_new
    return maxit


def main():
    case = sys.argv[1] if len(sys.argv) > 1 else "q1c12"
    if case.startswith("q1c"):
        prob = P.assemble(H.amg(G.structured_box(3, int(case[3:]), k=1)), p=1.0)
        kw = dict(t=0.01)
    else:
        prob = P.assemble(H.amg(G.subdivide(G.fem2d_P1(), int(case[3:]))), p=1.5)
        kw = {}
    M = prob.M[0]
    t0 = time.time()
    systems = record_systems(prob, kw)
    print("%s: %d systems recorded in %.0fs; fine unknowns %d, levels %s" % (case, len(systems), time.time() - t0, M.R_fine[-1].shape[1],
                                                                          [R.shape[1] for R in M.R_fine]), flush=True)
    Ts = transfers(M)
    variants = [
        ("cheb2 r8 V gershgorin (shipped)", dict(smoother="cheb", nu=2, ratio=8.0)),
        ("cheb2 r8 V exact lambda", dict(smoother="cheb", nu=2, ratio=8.0, lam="exact")),
        ("cheb2 r8 V power 12 x1.1", dict(smoother="cheb", nu=2, ratio=8.0, lam="power:12:1.1")),
        ("cheb2 r8 V power 6 x1.1", dict(smoother="cheb", nu=2, ratio=8.0, lam="power:6:1.1")),
        ("cheb2 r8 V power 6 x1.3", dict(smoother="cheb", nu=2, ratio=8.0, lam="power:6:1.3")),
        ("cheb2 r8 V power 3 x1.3", dict(smoother="cheb", nu=2, ratio=8.0, lam="power:3:1.3")),
        ("cheb2 r4 V power 6 x1.1", dict(smoother="cheb", nu=2, ratio=4.0, lam="power:6:1.1")),
        ("cheb2 r16 V power 6 x1.1", dict(smoother="cheb", nu=2, ratio=16.0, lam="power:6:1.1")),
        ("cheb3 r16 V power 6 x1.1", dict(smoother="cheb", nu=3, ratio=16.0, lam="power:6:1.1")),
        ("cheb2 r8 V gershgorin x0.7", dict(smoother="cheb", nu=2, ratio=8.0, lam="scaled:0.7")),
        ("cheb2 r8 V gershgorin x0.5", dict(smoother="cheb", nu=2, ratio=8.0, lam="scaled:0.5")),
        ("l1-Jacobi 2 V", dict(smoother="l1", nu=2)),
        ("sym. Gauss-Seidel V (sequential bound)", dict(smoother="sgs", nu=2)),
    ]
    V0 = VCycle(condense(*systems[len(systems) // 2][:2], M)[0], Ts)
    Vx = VCycle(condense(*systems[len(systems) // 2][:2], M)[0], Ts, lam="exact")
    print("  lambda_max(D^-1 A) per level, Gershgorin vs exact:", " ".join("%.2f/%.2f" % (a, b) for a, b in zip(V0.lam, Vx.lam)), flush=True)
    rows = []
    for name, opt in variants:
        its, mvs = [], []
        for Hm, g, tc in systems:
            S, gs = condense(Hm, g, M)
            V = VCycle(S, Ts, **opt)
            n_it = pcg(S, gs, V)
            its.append(n_it)
            mvs.append(V.mv / max(n_it, 1) + 1.0)
        rows.append((name, float(np.mean(its)), int(np.max(its)), float(np.mean(mvs))))
        print("  %-40s PCG its mean %6.1f max %4d | mat-vecs/it %5.2f | cost %7.1f" % (name, rows[-1][1], rows[-1][2], rows[-1][3], rows[-1][1] * rows[-1][3]),
              flush=True)


if __name__ == "__main__":
    main()
