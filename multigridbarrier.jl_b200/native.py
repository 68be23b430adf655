"""ctypes binding of the C ABI in include/mgbx.h (the same entry points a Julia `ccall` shim binds).

Only data marshalling lives here: numpy (C-order, 0-based) -> the column-major / int64 layouts of
the ABI.  There is no compute and no fallback: if libmgbx.so is missing or no CUDA device is
present the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional

import numpy as np
import scipy.sparse as sp

HERE = os.path.dirname(os.path.abspath(__file__))
LIBPATH = os.path.join(HERE, "libmgbx.so")

MAX_LEVELS, MAX_ND = 32, 12
OK, NOT_CONVERGED, NON_FINITE = 0, 1, 2
ERR_ARG, ERR_CUDA, ERR_ALLOC, ERR_UNSUPPORTED, ERR_INTERNAL = -1, -2, -3, -4, -5
MAIN, FEAS = 0, 1

c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)
c_f64p = C.POINTER(C.c_double)


class Csr(C.Structure):
    _fields_ = [("rows", C.c_int64), ("cols", C.c_int64), ("rowptr", c_i64p), ("colind", c_i64p),
                ("val", c_f64p)]


class Piece(C.Structure):
    _fields_ = [("kind", C.c_int32), ("ni", C.c_int32), ("nc", C.c_int32), ("idx", c_i32p),
                ("A", c_f64p), ("b", c_f64p), ("p", c_f64p), ("mu", c_f64p)]


class Convex(C.Structure):
    _fields_ = [("npieces", C.c_int32), ("pieces", C.POINTER(Piece)), ("select", c_f64p)]


class Amg(C.Structure):
    _fields_ = [("n", C.c_int64), ("N", C.c_int64), ("p", C.c_int32), ("nu", C.c_int32),
                ("nD", C.c_int32), ("L", C.c_int32), ("w", c_f64p), ("nops", C.c_int32),
                ("op_data", C.POINTER(c_f64p)), ("D_var", c_i32p), ("D_op", c_i32p),
                ("R_fine", C.POINTER(Csr)), ("T", C.POINTER(Csr)), ("var_offsets", c_i64p),
                ("n_global", C.c_int64), ("var_local", c_i32p)]


class Problem(C.Structure):
    _fields_ = [("amg", Amg * 2), ("f_grid", c_f64p), ("g_grid", c_f64p), ("Q", Convex),
                ("barrier_weights", c_f64p)]


class Config(C.Structure):
    _fields_ = [("dense_direct_max", C.c_int32), ("coarse_max", C.c_int32), ("pcg_maxit", C.c_int32),
                ("pcg_rtol", C.c_double), ("smoother_sweeps", C.c_int32), ("condense", C.c_int32),
                ("device", C.c_int32), ("verbose", C.c_int32), ("profile", C.c_int32),
                ("persistent", C.c_int32), ("tail_max", C.c_int32), ("pcg_rtol_final", C.c_double),
                ("fused", C.c_int32), ("smoother", C.c_int32), ("cheb_ratio", C.c_double),
                ("precond_fp32", C.c_int32), ("lambda_power", C.c_int32),
                ("pcg_fail_rtol", C.c_double), ("pcg_fail_etol", C.c_double), ("pcg_stall_window", C.c_int32), ("direct_fallback", C.c_int32), ("elem_bulk", C.c_int32), ("shard_solve", C.c_int32),
                ("shard_min_rows", C.c_int32), ("shard_min_nnz", C.c_int32), ("spectral_kron", C.c_int32), ("uncondensed_pcg", C.c_int32), ("analytic_schur", C.c_int32)]


class StepOpts(C.Structure):
    _fields_ = [("maxit", C.c_int32), ("max_newton", C.c_int32), ("initial_step", C.c_int32),
                ("stop_kind", C.c_int32), ("stop_lambda_tol", C.c_double), ("stop_theta", C.c_double),
                ("finalize", C.c_int32), ("finalize_theta", C.c_double), ("line_search", C.c_int32),
                ("ls_beta", C.c_double), ("ls_c1", C.c_double)]


class StepResult(C.Structure):
    _fields_ = [("converged", C.c_int32), ("its", C.c_int32 * MAX_LEVELS), ("y", C.c_double),
                ("gnorm", C.c_double), ("inc", C.c_double), ("f01_evals", C.c_int32),
                ("f2_evals", C.c_int32), ("linear_solves", C.c_int32), ("pcg_iters", C.c_int32),
                ("ms_f01", C.c_double), ("ms_f2", C.c_double), ("ms_solve", C.c_double),
                ("solve_failures", C.c_int32), ("its_finalize", C.c_int32), ("direct_fallbacks", C.c_int32)]


class ScalarsOut(C.Structure):
    _fields_ = [("c_dot_Dz", C.c_double), ("var_max", C.c_double * MAX_ND),
                ("var_absmax", C.c_double * MAX_ND), ("all_finite", C.c_int32)]


class SolverInfo(C.Structure):
    _fields_ = [("condensed", C.c_int32), ("nlev", C.c_int32), ("nbig", C.c_int32), ("bottom_dense", C.c_int32),
                ("grid", C.c_int32), ("threads", C.c_int32), ("m", C.c_int64 * MAX_LEVELS),
                ("nnz", C.c_int64 * MAX_LEVELS), ("nnzT", C.c_int64 * MAX_LEVELS), ("assembly_terms", C.c_int64),
                ("hblk_entries", C.c_int64), ("galerkin_terms", C.c_int64), ("dgemm_flops", C.c_double),
                ("nshard", C.c_int32), ("nranks", C.c_int32)]


EXPORTS = [
    "mgbx_default_config", "mgbx_default_step_opts", "mgbx_abi_version", "mgbx_device_count",
    "mgbx_create", "mgbx_destroy", "mgbx_last_error", "mgbx_step", "mgbx_scalars",
    "mgbx_nccl_unique_id", "mgbx_comm_init", "mgbx_comm_finalize",
    "mgbx_phase1_init", "mgbx_attach_feasibility", "mgbx_set_feasibility_box", "mgbx_reset_feasibility_state", "mgbx_handoff",
    "mgbx_matched_t", "mgbx_get_z", "mgbx_get_z_unfinalized", "mgbx_set_z", "mgbx_set_grids", "mgbx_level_size",
    "mgbx_barrier_eval", "mgbx_hessian_pattern", "mgbx_hessian_values", "mgbx_solve_newton_system",
    "mgbx_plan_pattern", "mgbx_recover_transfer", "mgbx_kron_factor", "mgbx_shard_row_range",
    "mgbx_rs_create", "mgbx_rs_levels", "mgbx_rs_get", "mgbx_rs_destroy", "mgbx_launch_count", "mgbx_memory_report", "mgbx_kernel_stats", "mgbx_set_profile", "mgbx_solver_info",
]

_lib = None


class MgbxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libmgbx error %d: %s" % (code, msg))
        self.code = code


def lib():
    """Load libmgbx.so (built in-tree by build.py).  Raises if it is missing: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIBPATH):
        raise ImportError("libmgbx.so has not been built: run `python -m mgbx.build` or "
                          "__graft_entry__.build() (nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(LIBPATH)
    H = C.c_void_p
    L.mgbx_default_config.argtypes = [C.POINTER(Config)]
    L.mgbx_default_config.restype = None
    L.mgbx_default_step_opts.argtypes = [C.POINTER(StepOpts), C.c_int64]
    L.mgbx_default_step_opts.restype = None
    L.mgbx_abi_version.restype = C.c_int
    L.mgbx_device_count.restype = C.c_int
    L.mgbx_create.argtypes = [C.POINTER(Problem), C.POINTER(Config), C.POINTER(H)]
    L.mgbx_nccl_unique_id.argtypes = [C.c_char_p]
    L.mgbx_comm_init.argtypes = [H, C.c_int, C.c_int, C.c_char_p]
    L.mgbx_destroy.argtypes = [H]
    L.mgbx_destroy.restype = None
    L.mgbx_last_error.argtypes = [H]
    L.mgbx_last_error.restype = C.c_char_p
    L.mgbx_step.argtypes = [H, C.c_int, C.c_double, C.POINTER(StepOpts), C.POINTER(StepResult)]
    L.mgbx_scalars.argtypes = [H, C.c_int, C.POINTER(ScalarsOut)]
    L.mgbx_phase1_init.argtypes = [H, c_i32p, c_f64p, c_f64p]
    L.mgbx_attach_feasibility.argtypes = [H, C.POINTER(Amg)]
    L.mgbx_set_feasibility_box.argtypes = [H, C.c_double, C.c_double]
    L.mgbx_reset_feasibility_state.argtypes = [H]
    L.mgbx_handoff.argtypes = [H]
    L.mgbx_matched_t.argtypes = [H, C.c_double, c_f64p, c_f64p]
    L.mgbx_get_z.argtypes = [H, C.c_int, c_f64p]
    L.mgbx_set_z.argtypes = [H, C.c_int, c_f64p]
    L.mgbx_get_z_unfinalized.argtypes = [H, C.c_int, c_f64p]
    L.mgbx_set_grids.argtypes = [H, c_f64p, c_f64p]
    L.mgbx_level_size.argtypes = [H, C.c_int, C.c_int]
    L.mgbx_level_size.restype = C.c_int64
    L.mgbx_barrier_eval.argtypes = [H, C.c_int, C.c_int, C.c_double, c_f64p, C.c_int, c_f64p]
    L.mgbx_hessian_pattern.argtypes = [H, C.c_int, C.c_int, c_i64p, c_i64p, c_i64p]
    L.mgbx_hessian_values.argtypes = [H, C.c_int, C.c_int, C.c_double, c_f64p, c_f64p]
    L.mgbx_solve_newton_system.argtypes = [H, C.c_int, C.c_int, C.c_double, c_f64p, c_f64p, c_f64p, c_i32p]
    L.mgbx_plan_pattern.argtypes = [C.POINTER(Csr), C.c_int64, C.c_int32, C.c_int32, C.c_int32, c_i32p,
                                    c_i64p, c_i64p, c_i64p]
    L.mgbx_rs_create.argtypes = [C.POINTER(Csr), C.c_int32, C.c_int32, C.c_double, C.POINTER(C.c_void_p)]
    L.mgbx_rs_levels.argtypes = [C.c_void_p]
    L.mgbx_rs_levels.restype = C.c_int32
    L.mgbx_rs_get.argtypes = [C.c_void_p, C.c_int32, c_i64p, c_i64p, c_i64p, c_i64p, c_i64p, c_f64p]
    L.mgbx_rs_destroy.argtypes = [C.c_void_p]
    L.mgbx_rs_destroy.restype = None
    L.mgbx_kron_factor.argtypes = [c_f64p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_f64p, c_f64p, C.POINTER(C.c_int32)]
    L.mgbx_shard_row_range.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_i64p, c_i64p]
    L.mgbx_recover_transfer.argtypes = [C.POINTER(Csr), C.POINTER(Csr), c_i64p, c_i64p, c_i64p, c_f64p]
    L.mgbx_memory_report.argtypes = [H, C.c_char_p, C.c_int64, c_i64p]
    L.mgbx_launch_count.argtypes = [H]
    L.mgbx_launch_count.restype = C.c_int64
    L.mgbx_kernel_stats.argtypes = [H, C.c_int, c_i32p, C.POINTER(C.c_char_p), c_i64p, c_f64p]
    L.mgbx_set_profile.argtypes = [H, C.c_int]
    L.mgbx_solver_info.argtypes = [H, C.c_int, C.POINTER(SolverInfo)]
    _lib = L
    return L


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a, t=c_f64p):
    return a.ctypes.data_as(t)


class _Keep:
    """Owns the numpy buffers a ctypes struct points into."""

    def __init__(self):
        self.bufs = []

    def f64(self, a):
        a = _f64(a)
        self.bufs.append(a)
        return _ptr(a)

    def colmajor(self, a):
        """(n, k) C-order grid -> column-major buffer (k contiguous columns of length n)."""
        a = np.asarray(a, dtype=np.float64)
        if a.ndim == 1:
            return self.f64(a)
        if a.flags.f_contiguous:      # already in the reference's own (Julia: column-major) layout -- no copy
            self.bufs.append(a)
            return _ptr(a)
        # cache-blocked transpose: about twice as fast as ascontiguousarray(a.T) on the 1.5 M-row grids of the bench
        n, k = a.shape
        b = np.empty((k, n), dtype=np.float64)
        for s in range(0, n, 8192):
            b[:, s:s + 8192] = a[s:s + 8192].T
        self.bufs.append(b)
        return _ptr(b)

    def i64(self, a):
        a = np.ascontiguousarray(a, dtype=np.int64)
        self.bufs.append(a)
        return _ptr(a, c_i64p)

    def i32(self, a):
        a = np.ascontiguousarray(a, dtype=np.int32)
        self.bufs.append(a)
        return _ptr(a, c_i32p)

    def csr(self, M) -> Csr:
        if not (sp.isspmatrix_csr(M) and M.has_canonical_format):
            M = sp.csr_matrix(M)
            M.sum_duplicates()
            M.sort_indices()
        return Csr(M.shape[0], M.shape[1], self.i64(M.indptr), self.i64(M.indices), self.f64(M.data))


def _pack_amg(keep: _Keep, M, recover_transfers=False) -> Amg:
    geom = M.geometry
    n, N, p = geom.n, geom.N, geom.V
    names, D_var, D_op = [], [], []
    # per geometry, computed once: which operators are the identity, and the operator blocks in the boundary's layout -- the
    # reference's BlockDiag.data is p x p x N column-major already (src/BlockMatrices.jl:17-44), so its shim passes it as it is
    cache = geom.__dict__.setdefault("_mgbx_abi_cache", {"ident": {}, "ops": {}})
    for (var, op) in M.D:
        if op not in cache["ident"]:
            blocks = geom.operators[op]
            eye = np.eye(p)
            cache["ident"][op] = bool(np.array_equal(blocks[0], eye) and np.array_equal(blocks, np.broadcast_to(eye, blocks.shape)))
        ident = cache["ident"][op]
        if ident:
            oid = -1
        else:
            if op not in names:
                names.append(op)
            oid = names.index(op)
        D_var.append(var)
        D_op.append(oid)
    ops = (c_f64p * max(1, len(names)))()
    for k, nm in enumerate(names):
        # numpy ops[e, r, c]  ->  BlockDiag.data[r, c, e] column-major == memory order [e][c][r]
        if nm not in cache["ops"]:
            cache["ops"][nm] = np.ascontiguousarray(geom.operators[nm].transpose(0, 2, 1), dtype=np.float64)
        ops[k] = keep.f64(cache["ops"][nm])
    keep.bufs.append(ops)
    L = len(M.R_fine)
    # only R_fine[L-1] crosses the boundary with data: the library composes the coarser ones from T (mgbx.h)
    if recover_transfers:
        # what a shim over the UNMODIFIED reference can provide (src/multigrid.jl:278-288: AMG keeps R_fine only):
        # every R_fine[l], no level transfers, no var_offsets -- the library recovers both (mgbx.h)
        Rs = (Csr * L)(*[keep.csr(R) for R in M.R_fine])
        Tp, voffp = None, None
        keep.bufs += [Rs]
    else:
        Rs = (Csr * L)(*([Csr(R.shape[0], R.shape[1], None, None, None) for R in M.R_fine[:-1]] + [keep.csr(M.R_fine[-1])]))
        Ts = (Csr * max(1, L - 1))(*[keep.csr(T) for T in M.T])
        keep.bufs += [Rs, Ts]
        Tp = C.cast(Ts, C.POINTER(Csr))
        voffp = keep.i64(np.asarray(M.var_offsets, dtype=np.int64).reshape(L, M.nu + 1))
    vl = getattr(M, "var_local", None)
    return Amg(n, N, p, M.nu, M.nD, L, keep.f64(M.w), len(names),
               C.cast(ops, C.POINTER(c_f64p)), keep.i32(D_var), keep.i32(D_op),
               C.cast(Rs, C.POINTER(Csr)), Tp, voffp,
               int(getattr(M, "n_global", 0)), keep.i32(vl) if vl is not None else None)


def _pack_convex(keep: _Keep, Q, n) -> Convex:
    K = len(Q.pieces)
    arr = (Piece * K)()
    for k, pc in enumerate(Q.pieces):
        arr[k].kind = pc.kind
        arr[k].ni = pc.ni
        arr[k].nc = pc.nc
        arr[k].idx = keep.i32(pc.idx) if pc.idx is not None else None
        arr[k].A = keep.colmajor(pc.A)
        arr[k].b = keep.colmajor(pc.b)
        arr[k].p = keep.f64(pc.p) if pc.p is not None else None
        arr[k].mu = keep.f64(pc.mu) if pc.mu is not None else None
    keep.bufs.append(arr)
    sel = keep.colmajor(Q.select) if Q.select is not None else None
    return Convex(K, C.cast(arr, C.POINTER(Piece)), sel)


def default_config(**kw) -> Config:
    cfg = Config()
    lib().mgbx_default_config(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise TypeError("unknown mgbx_config field %r" % k)
        setattr(cfg, k, v)
    return cfg


class Handle:
    """Device-resident problem (the result of native_to_device in the reference)."""

    def __init__(self, prob, barrier_weights=None, with_feasibility=True, comm=None, recover_transfers=False, **cfg):
        L = lib()
        keep = _Keep()
        P = Problem()
        self._recover = bool(recover_transfers)
        P.amg[0] = _pack_amg(keep, prob.M[0], self._recover)
        # the feasibility AMG is attached lazily, only when phase1_init reports that phase I must run
        self._feas_M = prob.M[1] if with_feasibility else None
        self._feas_attached = False
        n = prob.M[0].geometry.n
        P.f_grid = keep.colmajor(prob.f)
        P.g_grid = keep.colmajor(prob.g)
        P.Q = _pack_convex(keep, prob.Q, n)
        P.barrier_weights = keep.f64(barrier_weights) if barrier_weights is not None else None
        self.cfg = default_config(**cfg)
        self._h = C.c_void_p()
        rc = L.mgbx_create(C.byref(P), C.byref(self.cfg), C.byref(self._h))
        if rc != OK:
            raise MgbxError(rc, (L.mgbx_last_error(None) or b"").decode())
        if comm is not None:
            rank, world, uid = comm
            try:
                self._check(L.mgbx_comm_init(self._h, int(rank), int(world), uid))
            except Exception:
                self.close()      # the device handle exists already: do not leak it
                raise
        self.n = n
        self.nu = [prob.M[0].nu, prob.M[1].nu if prob.M[1] is not None else 0]
        self.nD = [prob.M[0].nD, prob.M[1].nD if prob.M[1] is not None else 0]
        self.L = [len(prob.M[0].R_fine), len(prob.M[1].R_fine) if prob.M[1] is not None else 0]

    def _check(self, rc, allow=()):
        if rc < 0 or (rc > 0 and rc not in allow):
            raise MgbxError(rc, (lib().mgbx_last_error(self._h) or b"").decode())
        return rc

    def close(self):
        if self._h:
            lib().mgbx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- hot path
    def step_opts(self, **kw) -> StepOpts:
        o = StepOpts()
        lib().mgbx_default_step_opts(C.byref(o), self.n)
        for k, v in kw.items():
            setattr(o, k, v)
        return o

    def step(self, which, t, opts: StepOpts):
        r = StepResult()
        rc = self._check(lib().mgbx_step(self._h, which, float(t), C.byref(opts), C.byref(r)),
                         allow=(NOT_CONVERGED, NON_FINITE))
        return rc, r

    def scalars(self, which=MAIN) -> ScalarsOut:
        out = ScalarsOut()
        self._check(lib().mgbx_scalars(self._h, which, C.byref(out)))
        return out

    # ---- phase I
    def attach_feasibility(self):
        if self._feas_attached:
            return
        if self._feas_M is None:
            raise MgbxError(ERR_ARG, "phase I needed but the problem carries no feasibility AMG")
        keep = _Keep()
        a = _pack_amg(keep, self._feas_M, self._recover)
        self._check(lib().mgbx_attach_feasibility(self._h, C.byref(a)))
        self._feas_attached = True

    def phase1_init(self):
        need, b, zmax = C.c_int32(), C.c_double(), C.c_double()
        self._check(lib().mgbx_phase1_init(self._h, C.byref(need), C.byref(b), C.byref(zmax)))
        if need.value and not self._feas_attached:
            self.attach_feasibility()
            self._check(lib().mgbx_phase1_init(self._h, C.byref(need), C.byref(b), C.byref(zmax)))
        return bool(need.value), b.value, zmax.value

    def set_feasibility_box(self, b, R):
        self._check(lib().mgbx_set_feasibility_box(self._h, float(b), float(R)))

    def reset_feasibility_state(self):
        self._check(lib().mgbx_reset_feasibility_state(self._h))

    def handoff(self):
        self._check(lib().mgbx_handoff(self._h))

    def matched_t(self, t_default):
        t, ts = C.c_double(), C.c_double()
        self._check(lib().mgbx_matched_t(self._h, float(t_default), C.byref(t), C.byref(ts)))
        return t.value, ts.value

    # ---- state
    def get_z(self, which=MAIN):
        z = np.empty(self.nu[which] * self.n)
        self._check(lib().mgbx_get_z(self._h, which, _ptr(z)))
        return z

    def get_z_unfinalized(self, which=MAIN):
        z = np.empty(self.nu[which] * self.n)
        self._check(lib().mgbx_get_z_unfinalized(self._h, which, _ptr(z)))
        return z

    def set_z(self, z, which=MAIN):
        z = _f64(z).reshape(-1)
        assert z.size == self.nu[which] * self.n
        self._check(lib().mgbx_set_z(self._h, which, _ptr(z)))

    def set_grids(self, f_grid=None, g_grid=None):
        keep = _Keep()
        self._check(lib().mgbx_set_grids(self._h, keep.colmajor(f_grid) if f_grid is not None else None,
                                         keep.colmajor(g_grid) if g_grid is not None else None))

    def memory_report(self):
        """(text, total bytes): device memory held by the handle, by category."""
        buf = C.create_string_buffer(8192)
        tot = C.c_int64()
        self._check(lib().mgbx_memory_report(self._h, buf, 8192, C.byref(tot)))
        return buf.value.decode(), tot.value

    def launch_count(self):
        return int(lib().mgbx_launch_count(self._h))

    def solver_info(self, which=MAIN):
        out = SolverInfo()
        self._check(lib().mgbx_solver_info(self._h, which, C.byref(out)))
        L = out.nlev
        return dict(condensed=bool(out.condensed), nlev=L, nbig=out.nbig, bottom_dense=bool(out.bottom_dense),
                    grid=out.grid, threads=out.threads, m=list(out.m[:L]), nnz=list(out.nnz[:L]), nnzT=list(out.nnzT[:L]),
                    assembly_terms=out.assembly_terms, hblk_entries=out.hblk_entries, galerkin_terms=out.galerkin_terms,
                    dgemm_flops=out.dgemm_flops, nshard=out.nshard, nranks=out.nranks)

    def set_profile(self, on):
        self._check(lib().mgbx_set_profile(self._h, int(on)))

    def kernel_stats(self, reset=False):
        """{class: (launches, device ms)}; ms are only accumulated while profiling is on."""
        nc = C.c_int32()
        names = (C.c_char_p * 32)()
        launches = np.zeros(32, np.int64)
        ms = np.zeros(32)
        self._check(lib().mgbx_kernel_stats(self._h, int(reset), C.byref(nc), names, _ptr(launches, c_i64p), _ptr(ms)))
        return {names[k].decode(): (int(launches[k]), float(ms[k])) for k in range(nc.value)}

    # ---- parity hooks
    def level_size(self, which, level):
        return int(lib().mgbx_level_size(self._h, which, level))

    def barrier_eval(self, which, level, t, s, order):
        s = _f64(s)
        out = np.empty(1 if order == 0 else s.size)
        self._check(lib().mgbx_barrier_eval(self._h, which, level, float(t), _ptr(s), order, _ptr(out)))
        return float(out[0]) if order == 0 else out

    def hessian_pattern(self, which, level):
        nnz = C.c_int64()
        self._check(lib().mgbx_hessian_pattern(self._h, which, level, C.byref(nnz), None, None))
        m = self.level_size(which, level)
        ptr = np.empty(m + 1, np.int64)
        ind = np.empty(nnz.value, np.int64)
        self._check(lib().mgbx_hessian_pattern(self._h, which, level, C.byref(nnz), _ptr(ptr, c_i64p),
                                               _ptr(ind, c_i64p)))
        return ptr, ind

    def hessian(self, which, level, t, s):
        ptr, ind = self.hessian_pattern(which, level)
        s = _f64(s)
        val = np.empty(ind.size)
        self._check(lib().mgbx_hessian_values(self._h, which, level, float(t), _ptr(s), _ptr(val)))
        m = ptr.size - 1
        return sp.csr_matrix((val, ind, ptr), shape=(m, m))

    def solve_newton_system(self, which, level, t, s, rhs):
        s, rhs = _f64(s), _f64(rhs)
        x = np.empty_like(rhs)
        it = C.c_int32()
        self._check(lib().mgbx_solve_newton_system(self._h, which, level, float(t), _ptr(s), _ptr(rhs),
                                                   _ptr(x), C.byref(it)))
        return x, it.value


def nccl_unique_id() -> bytes:
    """128-byte NCCL id (rank 0 creates it; broadcast it to the other ranks, e.g. with torch.distributed)."""
    buf = C.create_string_buffer(128)
    rc = lib().mgbx_nccl_unique_id(buf)
    if rc != OK:
        raise MgbxError(rc, (lib().mgbx_last_error(None) or b"").decode())
    return buf.raw


def plan_pattern(R, N, p, nu, D_var):
    """Host-only: reference assembly-plan pattern of R'HR (no GPU needed)."""
    keep = _Keep()
    Rc = keep.csr(R)
    nnz = C.c_int64()
    dv = np.ascontiguousarray(D_var, dtype=np.int32)
    rc = lib().mgbx_plan_pattern(C.byref(Rc), N, p, nu, len(dv), _ptr(dv, c_i32p), C.byref(nnz), None, None)
    if rc != OK:
        raise MgbxError(rc, (lib().mgbx_last_error(None) or b"").decode())
    ptr = np.empty(R.shape[1] + 1, np.int64)
    ind = np.empty(nnz.value, np.int64)
    rc = lib().mgbx_plan_pattern(C.byref(Rc), N, p, nu, len(dv), _ptr(dv, c_i32p), C.byref(nnz),
                                 _ptr(ptr, c_i64p), _ptr(ind, c_i64p))
    if rc != OK:
        raise MgbxError(rc, (lib().mgbx_last_error(None) or b"").decode())
    return ptr, ind


def ruge_stuben(K, max_coarse=2, max_levels=10, theta=0.25):
    """Host-only: prolongations finest -> coarsest of the classical Ruge-Stueben hierarchy of K (csrc/host_amg.hpp) -- the C++ twin of
    hierarchy.ruge_stuben, bitwise equal to it (src/amg_prolongators.jl:16-18 is the reference's call site)."""
    keep = _Keep()
    Kc = keep.csr(sp.csr_matrix(K, dtype=np.float64))
    h = C.c_void_p()
    rc = lib().mgbx_rs_create(C.byref(Kc), int(max_coarse), int(max_levels), float(theta), C.byref(h))
    if rc != OK:
        raise MgbxError(rc, (lib().mgbx_last_error(None) or b"").decode())
    try:
        Ps = []
        for l in range(lib().mgbx_rs_levels(h)):
            rows, cols, nnz = C.c_int64(), C.c_int64(), C.c_int64()
            lib().mgbx_rs_get(h, l, C.byref(rows), C.byref(cols), C.byref(nnz), None, None, None)
            ptr, ind, val = np.empty(rows.value + 1, np.int64), np.empty(nnz.value, np.int64), np.empty(nnz.value)
            rc = lib().mgbx_rs_get(h, l, C.byref(rows), C.byref(cols), C.byref(nnz), _ptr(ptr, c_i64p), _ptr(ind, c_i64p), _ptr(val))
            if rc != OK:
                raise MgbxError(rc, "mgbx_rs_get")
            Ps.append(sp.csr_matrix((val, ind, ptr), shape=(rows.value, cols.value)))
        return Ps
    finally:
        lib().mgbx_rs_destroy(h)


def kron_factor(M, r1, r2, c1, c2):
    """Host-only: (A, B) with M == kron(A, B) (A r1 x c1, B r2 x c2) or None -- the structure test behind the sum-factorised spectral
    assembly (csrc/engine.hpp kron_factor)."""
    M = np.ascontiguousarray(M, dtype=np.float64)
    assert M.shape == (r1 * r2, c1 * c2)
    A, B = np.zeros((r1, c1)), np.zeros((r2, c2))
    ok = C.c_int32(0)
    rc = lib().mgbx_kron_factor(_ptr(M), r1, r2, c1, c2, 0, _ptr(A), _ptr(B), C.byref(ok))
    if rc != OK:
        raise MgbxError(rc, (lib().mgbx_last_error(None) or b"").decode())
    return (A, B) if ok.value else None


def shard_row_range(rows, lanes_per_row, ctas_per_rank, nranks, rank):
    """Host-only: rows [r0, r1) of a level that `rank` owns in the row-sharded multi-GPU solve (csrc/pcg2.hpp)."""
    r0, r1 = C.c_int64(), C.c_int64()
    rc = lib().mgbx_shard_row_range(int(rows), int(lanes_per_row), int(ctas_per_rank), int(nranks), int(rank), C.byref(r0), C.byref(r1))
    if rc != OK:
        raise MgbxError(rc, "bad argument")
    return r0.value, r1.value


def recover_transfer(R_next, R_cur):
    """Host-only: T (scipy CSR) with R_next @ T = R_cur, as mgbx_create recovers the level transfers when none are given."""
    keep = _Keep()
    Rn, Rc = keep.csr(R_next), keep.csr(R_cur)
    nnz = C.c_int64()
    rc = lib().mgbx_recover_transfer(C.byref(Rn), C.byref(Rc), C.byref(nnz), None, None, None)
    if rc != OK:
        raise MgbxError(rc, (lib().mgbx_last_error(None) or b"").decode())
    ptr = np.empty(R_next.shape[1] + 1, np.int64)
    ind = np.empty(nnz.value, np.int64)
    val = np.empty(nnz.value, np.float64)
    rc = lib().mgbx_recover_transfer(C.byref(Rn), C.byref(Rc), C.byref(nnz), _ptr(ptr, c_i64p), _ptr(ind, c_i64p), _ptr(val))
    if rc != OK:
        raise MgbxError(rc, (lib().mgbx_last_error(None) or b"").decode())
    return sp.csr_matrix((val, ind, ptr), shape=(R_next.shape[1], R_cur.shape[1]))
