// mgbx.cu -- the C ABI (include/mgbx.h): argument checks, error reporting, the handle's life cycle, and the process-wide
// NCCL communicator.  The work behind each entry point is done by the Engine (engine.hpp); this unit launches no kernel.
// The t-ramp (mgb_core) and phase-I control flow (mgb_driver) stay on the host side of the ABI:
// they only exchange scalars with this library.
#include <dlfcn.h>

#include <numeric>

#include "engine.hpp"
#include "host_amg.hpp"

using namespace mgbx;

namespace {

thread_local std::string g_last_error;
const char *kKClassNames[KC_COUNT] = {"node_f01", "node_f2", "blockgrad", "blockhess", "csr_gather", "spmv", "spgemm",
                                             "vector", "condense", "dense", "pcg_persistent", "elem_f01", "elem_f2", "dgemm_dmma", "elem_generic_f01", "elem_generic_f2"};

// the AMG `which` refers to (1: the feasibility AMG, once attached)
Amg &amg_arg(mgbx_handle *h, int which, const char *prefix = "") {
  if (which < 0 || which > 1 || (which == 1 && !h->has_feas)) throw ArgError(std::string(prefix) + "no such AMG");
  return h->amg[which];
}
// ... and one of its levels
Amg &level_arg(mgbx_handle *h, int which, int level) {
  Amg &A = amg_arg(h, which);
  if (level < 0 || level >= A.L) throw ArgError("no such level");
  return A;
}

int guarded(mgbx_handle *h, const std::function<int()> &fn);

}  // namespace

// ------------------------------------------------------------------------------------------------
// NCCL, loaded on demand (multi-GPU runs only)
// ------------------------------------------------------------------------------------------------
NcclApi &mgbx::nccl_api() {
  static NcclApi api;
  if (api.lib) return api;
  const char *names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char *nm : names) {
    api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (api.lib) break;
  }
  if (!api.lib) throw std::runtime_error(std::string("cannot load NCCL (libnccl.so.2): ") + dlerror());
  auto sym = [&](const char *n) {
    void *p = dlsym(api.lib, n);
    if (!p) throw std::runtime_error(std::string("NCCL symbol missing: ") + n);
    return p;
  };
  api.GetUniqueId = (int (*)(NcclUniqueId *))sym("ncclGetUniqueId");
  api.CommInitRank = (int (*)(void **, int, NcclUniqueId, int))sym("ncclCommInitRank");
  api.CommDestroy = (int (*)(void *))sym("ncclCommDestroy");
  api.AllReduce = (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t))sym("ncclAllReduce");
  api.AllGather = (int (*)(const void *, void *, size_t, int, void *, cudaStream_t))sym("ncclAllGather");
  api.GroupStart = (int (*)())sym("ncclGroupStart");
  api.GroupEnd = (int (*)())sym("ncclGroupEnd");
  api.GetErrorString = (const char *(*)(int))sym("ncclGetErrorString");
  return api;
}

namespace {

int guarded(mgbx_handle *h, const std::function<int()> &fn) {
  try {
    // several handles (or torch) may have changed the calling thread's current device since this handle was created
    if (h && h->device >= 0) CK(cudaSetDevice(h->device));
    return fn();
  } catch (const ArgError &e) {
    if (h) h->err = e.what();
    g_last_error = e.what();
    return MGBX_ERR_ARG;
  } catch (const UnsupportedError &e) {
    if (h) h->err = e.what();
    g_last_error = e.what();
    return MGBX_ERR_UNSUPPORTED;
  } catch (const std::invalid_argument &e) {
    if (h) h->err = e.what();
    g_last_error = e.what();
    return MGBX_ERR_ARG;
  } catch (const std::bad_alloc &) {
    if (h) h->err = "host allocation failed";
    g_last_error = "host allocation failed";
    return MGBX_ERR_ALLOC;
  } catch (const std::exception &e) {
    if (h) h->err = e.what();
    g_last_error = e.what();
    const bool cuda = std::string(e.what()).find("CUDA") != std::string::npos || std::string(e.what()).find("cudaMalloc") != std::string::npos;
    return cuda ? MGBX_ERR_CUDA : MGBX_ERR_INTERNAL;
  }
}
}  // namespace

// -------------------------------------------------------------------------------------------------
// C ABI
// -------------------------------------------------------------------------------------------------
extern "C" {

void mgbx_default_config(mgbx_config *c) {
  c->dense_direct_max = 2048;
  c->coarse_max = 128;
  c->pcg_maxit = 400;
  c->pcg_rtol = 1e-7;
  c->smoother_sweeps = 2;
  c->condense = 1;
  c->device = -1;
  c->verbose = 0;
  c->profile = 0;
  c->persistent = 2;
  c->tail_max = 1200;
  c->pcg_rtol_final = 1e-15;
  c->fused = 1;
  c->smoother = 1;
  c->cheb_ratio = 8.0;
  c->precond_fp32 = 2;
  c->lambda_power = -1;
  c->pcg_fail_rtol = 1e-5;
  c->pcg_fail_etol = 1e-8;
  c->pcg_stall_window = 100;
  c->direct_fallback = 1;
  c->elem_bulk = 1;
  c->shard_solve = 1;
  c->shard_min_rows = 100000;
  c->shard_min_nnz = 4000000;
  c->spectral_kron = 1;
  c->uncondensed_pcg = 0;
  c->analytic_schur = 1;
}

void mgbx_default_step_opts(mgbx_step_opts *o, int64_t n) {
  o->maxit = 10000;
  o->max_newton = 8;   // ceil(log2(-log2(eps))) + 2 for Float64 (src/mgb.jl:101)
  o->initial_step = 0;
  o->stop_kind = 1;
  o->stop_lambda_tol = 0.25 / std::sqrt((double)n);
  o->stop_theta = 0.9;
  o->finalize = 0;
  o->finalize_theta = 0.9;
  o->line_search = 0;
  o->ls_beta = 0.5;
  o->ls_c1 = 0.1;
}

int mgbx_abi_version(void) { return MGBX_ABI_VERSION; }

int mgbx_device_count(void) {
  int c = 0;
  if (cudaGetDeviceCount(&c) != cudaSuccess) return 0;
  return c;
}

const char *mgbx_last_error(const mgbx_handle *h) { return h ? h->err.c_str() : g_last_error.c_str(); }

int mgbx_create(const mgbx_problem *prob, const mgbx_config *cfg, mgbx_handle **out) {
  if (!prob || !out) {
    g_last_error = "mgbx_create: null argument";
    return MGBX_ERR_ARG;
  }
  *out = nullptr;
  mgbx_handle *h = new mgbx_handle();
  if (cfg) h->cfg = *cfg;
  else mgbx_default_config(&h->cfg);
  if (h->cfg.dense_direct_max > kDenseMaxUnknowns) h->cfg.dense_direct_max = kDenseMaxUnknowns;
  if (h->cfg.coarse_max > kCoarseMaxDense) h->cfg.coarse_max = kCoarseMaxDense;
  if (h->cfg.coarse_max < 0) h->cfg.coarse_max = 0;
  h->last_tol = {h->cfg.pcg_rtol * h->cfg.pcg_rtol, 25};   // until the first Newton run: a window of 25, not cfg.pcg_stall_window
  int rc = guarded(h, [&]() -> int {
    if (h->cfg.persistent != 2) throw ArgError("mgbx_config.persistent must be 2 (the only solve kernel)");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
      throw std::runtime_error("CUDA device required: libmgbx has no CPU fallback (cudaGetDeviceCount: " +
                               std::string(cudaGetErrorString(e)) + ")");
    if (h->cfg.device >= 0) CK(cudaSetDevice(h->cfg.device));
    CK(cudaGetDevice(&h->device));
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    h->pool.stream = h->stream;
    {
      int dev = 0;
      CK(cudaGetDevice(&dev));
      cudaMemPool_t mp = nullptr;
      CK(cudaDeviceGetDefaultMemPool(&mp, dev));
      uint64_t keep = UINT64_MAX;   // freed blocks stay cached in the pool: the next handle reuses them without driver calls
      CK(cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep));
      h->pcg2_grid = pcg2_grid(dev);
      if (h->pcg2_grid == 0) throw std::runtime_error("CUDA device cannot run the cooperative solve kernel");
      solve_kernels_init();
    }
    h->partials = h->pool.zeros<double>((size_t)kRedBlocks * 8, h->stream);
    h->ticket = h->pool.zeros<unsigned int>(4, h->stream);
    h->dscal = h->pool.zeros<double>(kScalSlots, h->stream);
    CK(cudaMallocHost((void **)&h->hscal, sizeof(double) * kScalSlots));
    const mgbx_amg &a0 = prob->amg[0];
    create_amg(h, a0, h->amg[0]);
    Amg &A = h->amg[0];
    if (!prob->f_grid || !prob->g_grid) throw ArgError("f_grid / g_grid missing");
    CK(cudaMemcpyAsync(A.f, prob->f_grid, sizeof(double) * A.n * A.nD, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(A.z, prob->g_grid, sizeof(double) * A.n * A.nu, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(A.zinit, prob->g_grid, sizeof(double) * A.n * A.nu, cudaMemcpyHostToDevice, h->stream));
    if (prob->barrier_weights) A.bw = h->pool.upload<double>(prob->barrier_weights, A.n, h->stream);
    HostTimer tq;
    upload_convex(h, prob->Q, A.n, A.nD, A.cd);
    if (h->cfg.verbose > 0) fprintf(stderr, "[mgbx] convex set scanned + uploaded %.3fs\n", tq.lap());
    if (prob->amg[1].n > 0) attach_feasibility(h, prob->amg[1]);
    CK(cudaStreamSynchronize(h->stream));
    return MGBX_OK;
  });
  if (rc != MGBX_OK) {
    g_last_error = h->err;
    mgbx_destroy(h);
    return rc;
  }
  *out = h;
  return MGBX_OK;
}

// The communicator is process-wide: creating one costs about a second, so handles share it.  id != NULL creates
// (or replaces) it; id == NULL reuses the existing one for the same (rank, nranks).
static void *g_comm = nullptr;
static int g_comm_rank = -1, g_comm_nranks = 0;
static int g_comm_users = 0;   // live handles holding g_comm: it is neither replaced nor destroyed under them

void mgbx_destroy(mgbx_handle *h) {
  if (!h) return;
  if (h->device >= 0) cudaSetDevice(h->device);
  if (!h->prof_ns.empty()) {
    static const char *kinds[16] = {"first2", "pre", "resid", "restrict", "tail", "prolong", "post", "dense", "rz_sum", "pcg_matvec", "pcg_update", "init", "", "", "", ""};
    double tot = 0.0;
    for (double v : h->prof_ns) tot += v;
    fprintf(stderr, "[mgbx] phase profile of k_pcg2 (CTA 0's clock; each phase ends at its grid barrier), total %.3f ms\n", tot * 1e-6);
    for (size_t tag = 0; tag < h->prof_ns.size(); ++tag)
      if (h->prof_cnt[tag])
        fprintf(stderr, "[mgbx]   level %2d %-10s  n=%8lld  avg %7.2f us  total %8.3f ms  %5.1f %%\n", (int)(tag / 16), kinds[tag % 16], (long long)h->prof_cnt[tag],
                h->prof_ns[tag] * 1e-3 / h->prof_cnt[tag], h->prof_ns[tag] * 1e-6, 100.0 * h->prof_ns[tag] / tot);
  }
  if (h->comm && h->comm == g_comm && g_comm_users > 0) --g_comm_users;
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (int w = 0; w < 2; ++w)
    for (System *S : {h->amg[w].sys_cond.get(), h->amg[w].sys_coarse.get(), h->amg[w].sys_hook.get()})
      if (S)
        for (auto &kv : S->pplans2) {
          for (void *q : kv.second.peer)
            if (q) cudaIpcCloseMemHandle(q);
          if (kv.second.arena) cudaFree(kv.second.arena);
        }
  h->pool.release();
  if (h->hscal) cudaFreeHost(h->hscal);
  for (auto e : h->ev_free) cudaEventDestroy(e);
  for (auto &p : h->ev_pending) {
    cudaEventDestroy(p.a);
    cudaEventDestroy(p.b);
  }
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

int mgbx_nccl_unique_id(char id[128]) {
  if (!id) return MGBX_ERR_ARG;
  return guarded(nullptr, [&]() -> int {
    NcclUniqueId u;
    NCK(nccl_api().GetUniqueId(&u));
    memcpy(id, u.internal, 128);
    return MGBX_OK;
  });
}


int mgbx_comm_init(mgbx_handle *h, int rank, int nranks, const char id[128]) {
  if (!h || nranks < 1 || rank < 0 || rank >= nranks) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    if (h->comm) throw ArgError("mgbx_comm_init: communicator already initialised");
    if (nranks == 1) return MGBX_OK;
    for (int w = 0; w < 2; ++w)
      if (h->amg[w].sys_cond || h->amg[w].sys_coarse || h->amg[w].sys_hook) throw ArgError("mgbx_comm_init must precede the first solve");
    if (id) {
      NcclUniqueId u;
      memcpy(u.internal, id, 128);
      void *comm = nullptr;
      NCK(nccl_api().CommInitRank(&comm, nranks, u, rank));
      if (g_comm && g_comm_users > 0) {
        nccl_api().CommDestroy(comm);
        throw ArgError("mgbx_comm_init: live handles still use the process-wide communicator; destroy them before passing a new NCCL id");
      }
      if (g_comm) nccl_api().CommDestroy(g_comm);
      g_comm = comm;
      g_comm_rank = rank;
      g_comm_nranks = nranks;
    } else if (!g_comm || g_comm_rank != rank || g_comm_nranks != nranks) {
      throw ArgError("mgbx_comm_init: no process-wide communicator for this (rank, nranks); pass an NCCL id first");
    }
    h->comm = g_comm;
    ++g_comm_users;
    h->rank = rank;
    h->nranks = nranks;
    return MGBX_OK;
  });
}

int mgbx_comm_finalize(void) {
  if (g_comm && g_comm_users > 0) {
    g_last_error = "mgbx_comm_finalize: live handles still use the communicator";
    return MGBX_ERR_ARG;
  }
  if (g_comm) nccl_api().CommDestroy(g_comm);
  g_comm = nullptr;
  g_comm_rank = -1;
  g_comm_nranks = 0;
  return MGBX_OK;
}

int mgbx_step(mgbx_handle *h, int which, double t, const mgbx_step_opts *o, mgbx_step_result *r) {
  if (!h || !o || !r) return MGBX_ERR_ARG;
  const int rc = guarded(h, [&]() -> int {
    amg_arg(h, which, "mgbx_step: ");
    if (o->line_search != 0 && o->line_search != 1) throw ArgError("mgbx_step: line_search must be 0 (backtracking) or 1 (illinois)");
    Engine E(h);
    return E.step(which, t, *o, r);
  });
  h->res = nullptr;
  return rc;
}

int mgbx_scalars(mgbx_handle *h, int which, mgbx_scalars_out *out) {
  if (!h || !out) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &A = amg_arg(h, which, "mgbx_scalars: ");
    Engine E(h);
    memset(out, 0, sizeof(*out));
    // c_dot_Dz = sum_j dot(w .* f[:, j], D_j z): the linear part of f0 at t = 1, s = 0
    CK(cudaMemsetAsync(A.x, 0, sizeof(double) * A.m[A.L - 1], h->stream));
    EvalOut e = E.eval_f01(A, A.L - 1, 1.0, A.z, A.x, A.gn);
    out->c_dot_Dz = e.lin;
    out->all_finite = 1;
    for (int v = 0; v < A.nu; ++v) {
      const MaxAbs r = E.maxabs(A.n, A.z + (int64_t)v * A.n);
      out->var_max[v] = r.max;
      out->var_absmax[v] = r.absmax;
      if (r.nonfinite != 0.0) out->all_finite = 0;
    }
    return MGBX_OK;
  });
}

int mgbx_phase1_init(mgbx_handle *h, int32_t *needs_phase1, double *b, double *zabsmax) {
  if (!h || !needs_phase1 || !b || !zabsmax) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Engine E(h);
    Amg &A = h->amg[0];
    // feasibility probe: the barrier at every node of D*z0, ignoring barrier weights (src/mgb.jl:417-420)
    CK(cudaMemsetAsync(A.x, 0, sizeof(double) * A.m[A.L - 1], h->stream));
    EvalOut e = E.eval_f01(A, A.L - 1, 0.0, A.z, A.x, A.gn, /*use_bw=*/false);
    *needs_phase1 = (e.nonfinite_nodes > 0.0 || !std::isfinite(e.y)) ? 1 : 0;
    double zmax = 0.0;
    for (int v = 0; v < A.nu; ++v) zmax = std::max(zmax, E.maxabs(A.n, A.z + (int64_t)v * A.n).absmax);
    *zabsmax = zmax;
    *b = 0.0;
    if (*needs_phase1) {
      if (!h->has_feas) return MGBX_OK;   // the host attaches the feasibility AMG (mgbx_attach_feasibility) and calls again
      Amg &F = h->amg[1];
      // b = 2*max(1, max slack)   (src/mgb.jl:437-445)
      E.phase1_slack(A, F);
      *b = 2.0 * std::max(1.0, E.maxabs(A.n, F.zinit + (int64_t)A.nu * A.n).max);
    }
    return MGBX_OK;
  });
}

int mgbx_attach_feasibility(mgbx_handle *h, const mgbx_amg *feas) {
  if (!h || !feas) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    attach_feasibility(h, *feas);
    return MGBX_OK;
  });
}

int mgbx_set_feasibility_box(mgbx_handle *h, double b, double Rbox) {
  if (!h || !h->has_feas) return MGBX_ERR_ARG;
  h->amg[1].cd.fb = b;
  h->amg[1].cd.fR = Rbox;
  return MGBX_OK;
}

int mgbx_reset_feasibility_state(mgbx_handle *h) {
  if (!h || !h->has_feas) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &F = h->amg[1];
    CK(cudaMemcpyAsync(F.z, F.zinit, sizeof(double) * F.nu * F.n, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MGBX_OK;
  });
}

int mgbx_handoff(mgbx_handle *h) {
  if (!h || !h->has_feas) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &A = h->amg[0], &F = h->amg[1];
    CK(cudaMemcpyAsync(A.z, F.z, sizeof(double) * A.nu * A.n, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MGBX_OK;
  });
}

int mgbx_matched_t(mgbx_handle *h, double t_default, double *t_out, double *tstar_out) {
  if (!h || !t_out || !tstar_out) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Engine E(h);
    return E.matched_t(t_default, t_out, tstar_out);
  });
}

int mgbx_get_z(mgbx_handle *h, int which, double *z_host) {
  if (!h || !z_host || which < 0 || which > 1) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &A = h->amg[which];
    CK(cudaMemcpyAsync(z_host, A.z, sizeof(double) * A.nu * A.n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MGBX_OK;
  });
}

int mgbx_get_z_unfinalized(mgbx_handle *h, int which, double *z_host) {
  if (!h || !z_host || which < 0 || which > 1) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &A = h->amg[which];
    CK(cudaMemcpyAsync(z_host, A.zunfin, sizeof(double) * A.nu * A.n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MGBX_OK;
  });
}

int mgbx_set_z(mgbx_handle *h, int which, const double *z_host) {
  if (!h || !z_host || which < 0 || which > 1) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &A = h->amg[which];
    CK(cudaMemcpyAsync(A.z, z_host, sizeof(double) * A.nu * A.n, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MGBX_OK;
  });
}

int mgbx_set_grids(mgbx_handle *h, const double *f_grid, const double *g_grid) {
  if (!h) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &A = h->amg[0];
    if (f_grid) CK(cudaMemcpyAsync(A.f, f_grid, sizeof(double) * A.n * A.nD, cudaMemcpyHostToDevice, h->stream));
    if (g_grid) {
      CK(cudaMemcpyAsync(A.z, g_grid, sizeof(double) * A.n * A.nu, cudaMemcpyHostToDevice, h->stream));
      CK(cudaMemcpyAsync(A.zinit, g_grid, sizeof(double) * A.n * A.nu, cudaMemcpyHostToDevice, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return MGBX_OK;
  });
}

int64_t mgbx_launch_count(const mgbx_handle *h) { return h ? h->launches : 0; }

int mgbx_memory_report(mgbx_handle *h, char *buf, int64_t buflen, int64_t *total_bytes) {
  if (!h) return MGBX_ERR_ARG;
  std::string out;
  for (auto &kv : h->pool.by_cat) {
    char line[256];
    snprintf(line, sizeof(line), "%-52s %10.1f MB\n", kv.first.c_str(), kv.second / 1e6);
    out += line;
  }
  if (total_bytes) *total_bytes = (int64_t)h->pool.bytes;
  if (buf && buflen > 0) {
    const size_t nc = std::min<size_t>(out.size(), (size_t)buflen - 1);
    memcpy(buf, out.data(), nc);
    buf[nc] = 0;
  }
  return MGBX_OK;
}

int mgbx_solver_info(mgbx_handle *h, int which, mgbx_solver_info_t *out) {
  if (!h || !out || which < 0 || which > 1) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    memset(out, 0, sizeof(*out));
    out->dgemm_flops = h->dgemm_flops;
    Amg &A = h->amg[which];
    System *S = h->cfg.condense ? A.sys_cond.get() : A.sys_hook.get();
    if (!S) return MGBX_OK;   // no fine-level (sparse) system built yet
    out->condensed = S->condensed ? 1 : 0;
    out->assembly_terms = S->top.nterms;
    out->hblk_entries = S->hblk_size;
    auto it = S->pplans2.find(0);
    if (it != S->pplans2.end()) {
      const Pcg2Plan &P = it->second.host;
      out->nlev = P.nlev;
      out->nbig = P.nbig;
      out->bottom_dense = P.bottom_dense;
      out->grid = h->pcg2_grid;
      out->threads = kPcg2Threads;
      out->nshard = P.dist.nshard;
      out->nranks = P.dist.nranks;
      const std::vector<int> act = Engine(h).active_levels(*S, 0);
      for (int q = 0; q < P.nlev; ++q) {
        const SysLevel &Lv = S->lev[act[q]];
        out->m[q] = P.lev[q].m;
        out->nnz[q] = Lv.A.nnz;
        out->nnzT[q] = (q + 1 < P.nlev) ? Lv.T.nnz : 0;
      }
    }
    for (auto &Lv : S->lev) out->galerkin_terms += Lv.s1.nterms + Lv.s2.nterms;
    return MGBX_OK;
  });
}

int mgbx_kernel_stats(mgbx_handle *h, int reset, int32_t *nclasses, const char **names, int64_t *launches, double *ms) {
  if (!h || !nclasses) return MGBX_ERR_ARG;
  *nclasses = KC_COUNT;
  for (int k = 0; k < KC_COUNT; ++k) {
    if (names) names[k] = kKClassNames[k];
    if (launches) launches[k] = h->kc_launches[k];
    if (ms) ms[k] = h->kc_ms[k];
    if (reset) {
      h->kc_launches[k] = 0;
      h->kc_ms[k] = 0.0;
    }
  }
  return MGBX_OK;
}

int mgbx_set_profile(mgbx_handle *h, int on) {
  if (!h) return MGBX_ERR_ARG;
  cudaStreamSynchronize(h->stream);
  h->cfg.profile = on;
  return MGBX_OK;
}

int64_t mgbx_level_size(mgbx_handle *h, int which, int level) {
  if (!h || which < 0 || which > 1 || level < 0 || level >= h->amg[which].L) return -1;
  return h->amg[which].m[level];
}

int mgbx_barrier_eval(mgbx_handle *h, int which, int level, double t, const double *s, int order, double *out) {
  if (!h || !s || !out) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &A = level_arg(h, which, level);
    if (order != 0 && order != 1) throw ArgError("order must be 0 or 1 (use mgbx_hessian_values for f2)");
    Engine E(h);
    CK(cudaMemcpyAsync(A.xn, s, sizeof(double) * A.m[level], cudaMemcpyHostToDevice, h->stream));
    EvalOut e = E.eval_f01(A, level, t, A.z, A.xn, A.gn);
    if (order == 0) *out = e.y;
    else {
      CK(cudaMemcpyAsync(out, A.gn, sizeof(double) * A.m[level], cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
    }
    return MGBX_OK;
  });
}

int mgbx_hessian_pattern(mgbx_handle *h, int which, int level, int64_t *nnz, int64_t *rowptr, int64_t *colind) {
  if (!h || !nnz) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &A = level_arg(h, which, level);
    Engine E(h);
    if (!dense_mode(A) && !A.sys_hook) A.sys_hook = build_system(h, A, false, A.L - 1);
    SysLevel &Lv = dense_mode(A) ? E.system_for(A, level).lev[0] : A.sys_hook->lev[A.L - 1 - level];
    *nnz = Lv.A.nnz;
    if (rowptr) CK(cudaMemcpy(rowptr, Lv.A.ptr, sizeof(int64_t) * (Lv.m + 1), cudaMemcpyDeviceToHost));
    if (colind) {
      std::vector<int32_t> tmp(Lv.A.nnz);
      CK(cudaMemcpy(tmp.data(), Lv.A.idx, sizeof(int32_t) * Lv.A.nnz, cudaMemcpyDeviceToHost));
      for (int64_t k = 0; k < Lv.A.nnz; ++k) colind[k] = tmp[k];
    }
    return MGBX_OK;
  });
}

int mgbx_hessian_values(mgbx_handle *h, int which, int level, double t, const double *s, double *val) {
  if (!h || !s || !val) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &A = level_arg(h, which, level);
    Engine E(h);
    if (dense_mode(A)) {   // dense (spectral) systems are assembled directly at the requested level
      System &S = E.system_for(A, level);
      CK(cudaMemcpyAsync(A.xn, s, sizeof(double) * A.m[level], cudaMemcpyHostToDevice, h->stream));
      E.assemble(A, S, level, t, A.z, A.xn);
      CK(cudaMemcpyAsync(val, S.lev[0].A.val, sizeof(double) * S.lev[0].A.nnz, cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      return MGBX_OK;
    }
    if (!A.sys_hook) A.sys_hook = build_system(h, A, false, A.L - 1);
    System &S = *A.sys_hook;
    CK(cudaMemcpyAsync(A.xn, s, sizeof(double) * A.m[level], cudaMemcpyHostToDevice, h->stream));
    E.assemble_unfused(A, S, level, t, A.xn);
    const SysLevel &Lv = S.lev[A.L - 1 - level];
    CK(cudaMemcpyAsync(val, Lv.A.val, sizeof(double) * Lv.A.nnz, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MGBX_OK;
  });
}

int mgbx_solve_newton_system(mgbx_handle *h, int which, int level, double t, const double *s, const double *rhs, double *x,
                             int32_t *pcg_iters) {
  if (!h || !s || !rhs || !x) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    Amg &A = level_arg(h, which, level);
    Engine E(h);
    System &S = E.system_for(A, level);
    const int64_t m = A.m[level];
    CK(cudaMemcpyAsync(A.xn, s, sizeof(double) * m, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(A.gn, rhs, sizeof(double) * m, cudaMemcpyHostToDevice, h->stream));
    E.assemble(A, S, level, t, A.z, A.xn);
    const SolveResult r = E.solve(A, S, level, A.gn, A.dir, h->last_tol);
    if (pcg_iters) *pcg_iters = r.iters;
    CK(cudaMemcpyAsync(x, A.dir, sizeof(double) * m, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return MGBX_OK;
  });
}

int mgbx_plan_pattern(const mgbx_csr *R, int64_t N, int32_t p, int32_t nu, int32_t nD, const int32_t *D_var, int64_t *nnz,
                      int64_t *rowptr, int64_t *colind) {
  if (!R || !nnz || !D_var) return MGBX_ERR_ARG;
  return guarded(nullptr, [&]() -> int {
    const int64_t n = N * (int64_t)p;
    if (R->rows != (int64_t)nu * n) throw ArgError("mgbx_plan_pattern: R must have nu*p*N rows");
    HostCsr H = csr_from_abi(*R, false);
    std::vector<int> used;
    for (int v = 0; v < nu; ++v) {
      bool any = false;
      for (int j = 0; j < nD; ++j) any = any || (D_var[j] == v);
      if (any) used.push_back(v);
    }
    std::vector<int64_t> colmap(R->cols);
    std::iota(colmap.begin(), colmap.end(), (int64_t)0);
    HostCsr pat = plan_pattern(element_incidence(H, N, p, used, n, colmap, R->cols));
    *nnz = pat.nnz();
    if (rowptr) std::copy(pat.ptr.begin(), pat.ptr.end(), rowptr);
    if (colind)
      for (int64_t k = 0; k < pat.nnz(); ++k) colind[k] = pat.idx[k];
    return MGBX_OK;
  });
}

int mgbx_recover_transfer(const mgbx_csr *R_next, const mgbx_csr *R_cur, int64_t *nnz, int64_t *rowptr, int64_t *colind, double *val) {
  if (!R_next || !R_cur || !nnz) return MGBX_ERR_ARG;
  return guarded(nullptr, [&]() -> int {
    HostCsr T = recover_transfer(*R_next, *R_cur);
    *nnz = T.nnz();
    if (rowptr) std::copy(T.ptr.begin(), T.ptr.end(), rowptr);
    if (colind)
      for (int64_t k = 0; k < T.nnz(); ++k) colind[k] = T.idx[k];
    if (val) std::copy(T.val.begin(), T.val.end(), val);
    return MGBX_OK;
  });
}

// ---- classical Ruge-Stueben hierarchy on the host (csrc/host_amg.hpp)
struct mgbx_rs_hierarchy {
  std::vector<mgbx::AmgCsr> P;
};

int mgbx_rs_create(const mgbx_csr *K, int32_t max_coarse, int32_t max_levels, double theta, mgbx_rs_hierarchy **out) {
  if (!K || !out || !K->rowptr || K->rows != K->cols || K->rows < 0 || max_levels < 1 || max_coarse < 0) return MGBX_ERR_ARG;
  return guarded(nullptr, [&]() -> int {
    AmgCsr A;
    A.rows = K->rows;
    A.cols = K->cols;
    A.ptr.assign(K->rowptr, K->rowptr + K->rows + 1);
    const int64_t nz = A.ptr.back();
    A.idx.assign(K->colind, K->colind + nz);
    A.val.assign(K->val, K->val + nz);
    for (int64_t k = 0; k < nz; ++k)
      if (A.idx[k] < 0 || A.idx[k] >= A.cols) throw ArgError("mgbx_rs_create: column index out of range");
    auto H = std::make_unique<mgbx_rs_hierarchy>();
    H->P = amg_ruge_stuben(std::move(A), max_coarse, max_levels, theta);
    *out = H.release();
    return MGBX_OK;
  });
}

int32_t mgbx_rs_levels(const mgbx_rs_hierarchy *H) { return H ? (int32_t)H->P.size() : -1; }

int mgbx_rs_get(const mgbx_rs_hierarchy *H, int32_t level, int64_t *rows, int64_t *cols, int64_t *nnz, int64_t *rowptr, int64_t *colind, double *val) {
  if (!H || level < 0 || level >= (int32_t)H->P.size() || !rows || !cols || !nnz) return MGBX_ERR_ARG;
  const mgbx::AmgCsr &P = H->P[(size_t)level];
  *rows = P.rows;
  *cols = P.cols;
  *nnz = (int64_t)P.idx.size();
  if (rowptr) std::copy(P.ptr.begin(), P.ptr.end(), rowptr);
  if (colind) std::copy(P.idx.begin(), P.idx.end(), colind);
  if (val) std::copy(P.val.begin(), P.val.end(), val);
  return MGBX_OK;
}

void mgbx_rs_destroy(mgbx_rs_hierarchy *H) { delete H; }

int mgbx_kron_factor(const double *M, int32_t r1, int32_t r2, int32_t c1, int32_t c2, int32_t col_major, double *A, double *B, int32_t *is_kron) {
  if (!M || !A || !B || !is_kron || r1 < 1 || r2 < 1 || c1 < 1 || c2 < 1) return MGBX_ERR_ARG;
  return guarded(nullptr, [&]() -> int {
    const int64_t rows = (int64_t)r1 * r2, cols = (int64_t)c1 * c2;
    std::vector<double> a, b;
    const bool ok = kron_factor([&](int64_t r, int64_t c) { return col_major ? M[r + c * rows] : M[r * cols + c]; }, r1, r2, c1, c2, a, b);
    *is_kron = ok ? 1 : 0;
    if (ok) {
      std::copy(a.begin(), a.end(), A);
      std::copy(b.begin(), b.end(), B);
    }
    return MGBX_OK;
  });
}

int mgbx_shard_row_range(int64_t rows, int32_t lanes_per_row, int32_t ctas_per_rank, int32_t nranks, int32_t rank, int64_t *row_begin,
                         int64_t *row_end) {
  if (!row_begin || !row_end || rows < 0 || ctas_per_rank < 1 || nranks < 1 || rank < 0 || rank >= nranks) return MGBX_ERR_ARG;
  if (lanes_per_row != 1 && lanes_per_row != 2 && lanes_per_row != 4 && lanes_per_row != 8 && lanes_per_row != 16 && lanes_per_row != 32) return MGBX_ERR_ARG;
  pcg2_rank_rows(rows, lanes_per_row, ctas_per_rank, nranks, rank, *row_begin, *row_end);
  return MGBX_OK;
}

}  // extern "C"
