// engine.hpp -- the library's internal host types: error handling and launch accounting, the device memory pool, the
// linear-system and AMG state, the handle, and the Engine that runs evaluation, assembly, the linear solve and Newton.
// No kernel is defined or launched here.  Each unit owns the kernels it launches (device_common.cuh):
//   setup.cu         plans and systems, problem upload               setup_kernels.cuh
//   evaluate.cu      f0/f1, Hessian assembly, level chain, vectors    kernels.cuh, dense_kernels.cuh
//   linear_solve.cu  preconditioner setup, direct and PCG solves      solver_kernels.cuh, pcg2.hpp
//   newton.cu        Newton, mgb_step, matched t                      (host logic only)
//   mgbx.cu          NCCL loader, communicator and the C ABI         (host logic only)
#pragma once
#include <cuda_runtime.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "host_sparse.hpp"
#include "device_common.cuh"
#include "pcg2.hpp"

namespace mgbx {

#define CK(call)                                                                                      \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess)                                                                            \
      throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " + __FILE__ + ":" + \
                               std::to_string(__LINE__));                                             \
  } while (0)

// kernel classes for the optional per-class device timing (cfg.profile) and launch statistics
enum KClass { KC_NODE_F01 = 0, KC_NODE_F2, KC_BLOCKGRAD, KC_BLOCKHESS, KC_GATHER, KC_SPMV, KC_SPGEMM, KC_VEC, KC_COND,
              KC_DENSE, KC_PCG, KC_ELEM_F01, KC_ELEM_F2, KC_DGEMM, KC_ELEMG_F01, KC_ELEMG_F2, KC_COUNT };
enum { STAGE_F01 = -1, STAGE_F2 = -2, STAGE_SOLVE = -3 };
#define LAUNCH(kc, ...)   \
  do {                    \
    pre_launch(kc);       \
    __VA_ARGS__;          \
    post_launch(kc);      \
  } while (0)

struct UnsupportedError : std::runtime_error {
  explicit UnsupportedError(const std::string &m) : std::runtime_error(m) {}
};
struct ArgError : std::runtime_error {
  using std::runtime_error::runtime_error;
};

struct HostTimer {
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  double lap() {
    auto t1 = std::chrono::steady_clock::now();
    double s = std::chrono::duration<double>(t1 - t0).count();
    t0 = t1;
    return s;
  }
};

// at least one block: every kernel bounds-checks its index, and an empty level (e.g. no interior unknown) must not be a launch error
inline unsigned int nblk(int64_t work, int threads = 256) { return (unsigned int)std::max<int64_t>(1, (work + threads - 1) / threads); }

// ------------------------------------------------------------------------------------------------
// NCCL, loaded on demand (multi-GPU runs only, mgbx.cu): the few entry points used, declared here so that the
// library has no link-time dependency on NCCL.  Types follow nccl.h (2.x ABI).
// ------------------------------------------------------------------------------------------------
struct NcclUniqueId {
  char internal[128];
};
struct NcclApi {
  void *lib = nullptr;
  int (*GetUniqueId)(NcclUniqueId *) = nullptr;
  int (*CommInitRank)(void **, int, NcclUniqueId, int) = nullptr;
  int (*CommDestroy)(void *) = nullptr;
  int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
  int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
};
enum { kNcclInt64 = 4, kNcclUint64 = 5, kNcclFloat64 = 8, kNcclSum = 0, kNcclMax = 2 };
NcclApi &nccl_api();
#define NCK(call)                                                                                        \
  do {                                                                                                   \
    int r_ = (call);                                                                                     \
    if (r_ != 0) throw std::runtime_error(std::string("NCCL error: ") + nccl_api().GetErrorString(r_) + " at " + __FILE__ + ":" + \
                                          std::to_string(__LINE__));                                     \
  } while (0)

// ------------------------------------------------------------------------------------------------
// device memory pool (freed at destroy)
// ------------------------------------------------------------------------------------------------
struct Pool {
  std::vector<void *> ptrs;
  size_t bytes = 0;
  const char *cat = "problem";                 // category the next allocations are booked under (mgbx_memory_report)
  std::map<std::string, size_t> by_cat;
  cudaStream_t stream = nullptr;   // set at create: allocations are stream-ordered (cudaMallocAsync), cheap and reusable
  template <class T>
  T *alloc(size_t n) {
    if (n == 0) n = 1;
    void *p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, n * sizeof(T), stream);
    if (e != cudaSuccess) throw std::runtime_error(std::string("cudaMalloc failed: ") + cudaGetErrorString(e));
    ptrs.push_back(p);
    bytes += n * sizeof(T);
    by_cat[cat] += n * sizeof(T);
    return (T *)p;
  }
  template <class T>
  T *upload(const T *h, size_t n, cudaStream_t s) {
    T *d = alloc<T>(n);
    if (n) CK(cudaMemcpyAsync(d, h, n * sizeof(T), cudaMemcpyHostToDevice, s));
    return d;
  }
  template <class T>
  T *zeros(size_t n, cudaStream_t s) {
    T *d = alloc<T>(n);
    CK(cudaMemsetAsync(d, 0, (n ? n : 1) * sizeof(T), s));
    return d;
  }
  void release() {
    for (void *p : ptrs) cudaFreeAsync(p, stream);
    ptrs.clear();
    if (stream) cudaStreamSynchronize(stream);
  }
};

// stream-ordered scratch allocations for plan construction (no device-wide synchronisation, memory stays in the
// device's default pool between handles: its release threshold is raised at mgbx_create)
template <class T>
T *tmp_alloc(size_t n, cudaStream_t s) {
  void *p = nullptr;
  CK(cudaMallocAsync(&p, std::max<size_t>(n, 1) * sizeof(T), s));
  return (T *)p;
}
inline void tmp_free(void *p, cudaStream_t s) {
  if (p) cudaFreeAsync(p, s);
}

// ------------------------------------------------------------------------------------------------
// linear systems: top-level assembly plan + Galerkin hierarchy
// ------------------------------------------------------------------------------------------------
struct SysLevel {
  int64_t m = 0;
  DevCsr A;
  DevCsr T, Tt, AT;          // T: this level (rows) <- next coarser level (cols)
  // Galerkin gather plans: AT = A*T  and  A_coarse = T'*AT, one fixed-order sliced-ELL gather each
  SellPlan s1, s2;
  bool T_identity = false;
  float *val32 = nullptr;      // FP32 copy of A.val for the preconditioner passes (cfg.precond_fp32)
  double *dinv = nullptr, *diag = nullptr, *lam = nullptr;   // lam: Gershgorin bound of lambda_max(D^-1 A) (device scalar)
  double *pw = nullptr;       // power-iteration vector (kept across Newton iterations: warm start, cfg.lambda_power)
  double *b = nullptr, *x = nullptr, *x2 = nullptr, *r = nullptr;   // V-cycle work
  double *dense = nullptr, *dense_inv = nullptr, *dscale = nullptr;
  int spmv_group = 1;
  std::vector<int64_t> off;  // system offsets of the kept variables (+ end)
  // sliced-ELL copies for the solve kernel (pcg2.hpp): pattern built once, A's values refreshed
  // with every assembly, T / T' filled once
  SellBuild sA, sT, sTt;
  bool sell_A = false, sell_T = false;
};

struct System {
  bool condensed = false;
  int ltop = 0;                      // AMG level of lev[0]
  std::vector<int> kept, elim;       // state variable ids
  std::vector<SysLevel> lev;         // lev[k] <-> AMG level ltop-k
  PairList pl;
  int nK = 0, nE = 0;
  int Krow[MGBX_MAX_ND], Erow[MGBX_MAX_ND];
  SellPlan top;                      // element blocks -> top-level CSR values
  double *Hblk = nullptr;
  int64_t hblk_size = 0;
  int cut = -1;                      // V-cycle bottom (dense inverse) level index, -1: none
  // dense assembly path (spectral): R'HR by FP64 DMMA GEMMs into the (full) top matrix; no gather plan, no hierarchy
  bool dense = false;
  std::vector<double *> Rt;          // per kept variable: transposed dense prolongation block (m_q x n)
  double *Hd = nullptr, *Wt = nullptr;
  // sum-factorised assembly (tensor-product spectral discretisations, dense_kernels.cuh): one entry per block of kept variables
  struct KronPair {
    int c1a = 0, c2a = 0, c1b = 0, c2b = 0, ncombo = 0;
    int64_t offa = 0, offb = 0;
    const double *AA = nullptr;            // (c1a c1b) x (ncombo n1), constant
    const double *Qj[kKronMaxCombos], *Qk[kKronMaxCombos];
    int hidx[kKronMaxCombos];              // packed-symmetric index of the node sample h_jk
  };
  bool kron = false;
  // fine-level system with a slack-like variable (only :id rows) that could be eliminated neither node-locally nor element-locally:
  // its 1/slack^2 entries stay in the matrix, which the V-cycle PCG cannot solve reliably late in the t-ramp
  bool uncondensed_slack = false;
  // the eliminated variable is element-local (elem_schur.cuh, e.g. a slack in :broken_P1): elim == {that variable}, nE == 1
  bool elem_local = false;
  ElemLocal el{};
  std::vector<KronPair> kp;
  double *Wcat = nullptr;
  // PCG work at the largest size (sparse systems only)
  double *pc_r = nullptr, *pc_p = nullptr, *pc_p2 = nullptr, *pc_Ap = nullptr, *pc_x = nullptr, *pc_b = nullptr;
  double *pcg_partials = nullptr, *pcg_out = nullptr;
  unsigned int *pcg_bar = nullptr;
  // solve kernel: one plan per top level
  struct Pcg2Dev {
    Pcg2Plan host;
    Pcg2Plan *dev = nullptr;
    size_t smem = 0;
    // multi-GPU row-sharded solve: this rank's exchange arena (cudaMalloc, exported by CUDA IPC) and the peers' mappings
    char *arena = nullptr;
    void *peer[kPcg2MaxRanks] = {nullptr};
  };
  std::map<int, Pcg2Dev> pplans2;
};

struct Amg {
  int64_t n = 0, N = 0;
  int p = 0, nu = 0, nD = 0, L = 0, nops = 0;
  int D_var[MGBX_MAX_ND], D_op[MGBX_MAX_ND];
  double *w = nullptr, *f = nullptr, *bw = nullptr, *z = nullptr, *zsave = nullptr, *zinit = nullptr, *zunfin = nullptr;
  const double *ops[MGBX_MAX_OPS];
  // tensor-product structure of a dense discretisation (spectral2d): ops[o] = kron(kronA[o], kronB[o]), n1 x n1 row-major host
  // factors; kron_n1 == 0: none
  int kron_n1 = 0;
  std::vector<std::vector<double>> kronA, kronB;
  HostCsr hRL;
  std::vector<HostCsr> hT;
  DevCsr RL, RLt;
  std::vector<DevCsr> T, Tt;
  std::vector<std::vector<int64_t>> voff;   // L x (nu+1)
  std::vector<int64_t> m;
  ConvexDev cd;
  // work
  double *zf = nullptr, *G = nullptr, *gb = nullptr, *Hn = nullptr, *hEEinv = nullptr, *hKE = nullptr, *slack = nullptr;
  std::vector<double *> chain;              // per level work vector (m_l)
  std::vector<double *> chain2;
  double *x = nullptr, *xn = nullptr, *g = nullptr, *gn = nullptr, *dir = nullptr, *rhs = nullptr, *tmp = nullptr, *xbest = nullptr,
         *gbest = nullptr;
  std::unique_ptr<System> sys_cond, sys_coarse, sys_hook;   // fine-level (condensed), levels < L-1, parity hooks
  std::map<int, std::unique_ptr<System>> sys_dense;         // dense (spectral) discretisations: one directly assembled system per level
  double fb = 0.0, fR = 0.0;
  int64_t n_global = 0;              // nodes of the whole mesh (== n on a single rank)
  std::vector<char> var_local;       // per variable: node-local unknowns at the fine level (multi-GPU)
  bool any_local = false;
};

struct EvalOut {
  double y, gnorm;
  bool finite;
  double nonfinite_nodes, lin;
};
// f0 / f1 at a trial point, with |xn - x|^2 exactly as evaluated in floating point (zero: the step no longer moves x)
struct TrialOut : EvalOut {
  double step2;
};
struct Dot2 {
  double ab, aa, nonfinite;   // a.b, a.a, #non-finite entries of a
};
struct MaxAbs {
  double max, absmax, nonfinite;
};
// PCG stopping parameters: |r|^2 <= rtol2 |b|^2, or stagnation for `window` iterations without a new best residual
struct SolveTol {
  double rtol2;
  int window;
};

// Slots of the handle's device scalars dscal[kScalSlots] and of their pinned host mirror hscal.  The reduction kernels
// write fixed regions of dscal; evaluate.cu copies them to hscal and returns the values.  Successive calls reuse regions:
// each result is read before the next launch that writes its region.
// single GPU (fetched as the leading kScalSingle slots):
constexpr int kScalEval = 0;     // [0, 4) red_out of the f0 / f1 node and element kernels (and of k_node<NODE_SLACK> on every
                                 // path): sum bw F0 (or sum F0), sum w c.Dz, #non-finite F0, max slack (computed, never read)
constexpr int kScalMaxAbs = 0;   // [0, 3) k_maxabs: max, max|.|, #non-finite; reuses the evaluation slots, on every path
constexpr int kScalDot = 4;      // [4, 7) k_dot2: a.b, a.a, #non-finite(a)
constexpr int kScalTrial = 7;    // [7] k_trial: |xn - x|^2, read by the evaluation that follows the trial
constexpr int kScalSingle = 8;
// hscal only: readback of the solve kernel's result record (kPcg2Out*, pcg2.hpp)
constexpr int kScalPcgOut = 8;   // [8, 14)
// multi-GPU (the whole array is fetched); eval_f01 sums [kScalTrialSeg + 1, kScalDotSeg + 3) over the ranks in one all-reduce
constexpr int kScalTrialSeg = 38;   // [38] shared / [39] local part of |xn - x|^2 (k_trial_seg), zeroed by each evaluation
constexpr int kScalEvalDist = 40;   // [40, 44) red_out; the max slack is summed over the ranks here, not max-reduced
constexpr int kScalDotSeg = 44;     // [44, 50) k_dot2_seg: local part {a.b, a.a, #non-finite}, then shared part
constexpr int kScalDotSeg2 = 50;    // [50, 56) eval_f01's second k_dot2_seg, after the shared gradient entries were summed
constexpr int kScalSlots = 64;
static_assert(kScalEval + 4 <= kScalDot && kScalDot + 3 <= kScalTrial && kScalTrial + 1 <= kScalSingle &&
                  kScalSingle <= kScalPcgOut && kScalPcgOut + kPcg2OutCount <= kScalTrialSeg &&
                  kScalTrialSeg + 2 == kScalEvalDist && kScalEvalDist + 4 == kScalDotSeg &&   // contiguous for the all-reduce
                  kScalDotSeg + 6 <= kScalDotSeg2 && kScalDotSeg2 + 6 <= kScalSlots,
              "scalar slot regions overlap, break the all-reduced range or exceed dscal");

}  // namespace mgbx

struct mgbx_handle {
  mgbx::Pool pool;
  mgbx::Amg amg[2];
  std::string err;
  mgbx_config cfg;
  cudaStream_t stream = nullptr;
  bool has_feas = false;
  // reduction scratch
  double *partials = nullptr;
  unsigned int *ticket = nullptr;
  double *dscal = nullptr;   // device scalars, kScalSlots (layout above)
  double *hscal = nullptr;   // pinned host mirror
  // stats of the current step
  mgbx_step_result *res = nullptr;
  int64_t launches = 0;
  // per-class statistics; device time only when cfg.profile != 0
  int64_t kc_launches[mgbx::KC_COUNT] = {0};
  double kc_ms[mgbx::KC_COUNT] = {0};
  std::vector<cudaEvent_t> ev_free;
  struct Pending {
    int kc;
    cudaEvent_t a, b;
  };
  std::vector<Pending> ev_pending;
  cudaEvent_t ev_cur = nullptr;
  int pcg2_grid = 0;         // CTAs of the solve kernel k_pcg2
  double dgemm_flops = 0.0;   // FP64 tensor-core flops issued so far (spectral path)
  mgbx::SolveTol last_tol{};   // the last Newton run's tolerance (mgbx_create's before any), inherited by matched t and mgbx_solve_newton_system
  // multi-GPU
  int rank = 0, nranks = 1;
  void *comm = nullptr;
  int device = -1;           // CUDA device ordinal the handle lives on (made current at every ABI entry point)
  // phase profile of the solve kernel k_pcg2 (env MGBX_PCG_PROF=1): summed ns and counts per tag (level * 16 + kind)
  std::vector<double> prof_ns;
  std::vector<int64_t> prof_cnt;
  std::vector<unsigned long long> prof_host;
};
namespace mgbx {

// outcome of one linear solve (Engine::solve, solve_compact, pcg)
struct SolveResult {
  int iters = 0;       // PCG iterations, negative after a breakdown; 0 for a direct solve
  int status = 1;      // 1 converged / direct, 2 stagnated above the tolerance, 3 iteration limit, -1 breakdown
  double rel = 0.0;    // final relative residual |r| / |b| (0 for a direct solve)
  double erel = 0.0;   // share of the direction's energy b.x = |x|_A^2 gained in the last four PCG iterations
  Dot2 dg{};           // (dir, g) of Engine::solve: the Newton decrement g.dir, |dir|^2 and dir's non-finite entries
};

struct Engine {
  mgbx_handle *h;
  cudaStream_t s;
  explicit Engine(mgbx_handle *hh) : h(hh), s(hh->stream) {}

  // ---------------------------------------------------------------- streams, events, launch accounting
  void sync() {
    CK(cudaStreamSynchronize(s));
    if (!h->ev_pending.empty()) {
      for (auto &p : h->ev_pending) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, p.a, p.b);
        if (p.kc >= 0) h->kc_ms[p.kc] += ms;
        else if (h->res) {   // stage timers of the current mgbx_step
          if (p.kc == STAGE_F01) h->res->ms_f01 += ms;
          else if (p.kc == STAGE_F2) h->res->ms_f2 += ms;
          else if (p.kc == STAGE_SOLVE) h->res->ms_solve += ms;
        }
        h->ev_free.push_back(p.a);
        h->ev_free.push_back(p.b);
      }
      h->ev_pending.clear();
    }
  }
  // stage timing without extra host synchronisation: the event pair is resolved at the next sync()
  cudaEvent_t stage_begin() {
    cudaEvent_t e = get_event();
    cudaEventRecord(e, s);
    return e;
  }
  void stage_end(int stage, cudaEvent_t a) {
    cudaEvent_t b = get_event();
    cudaEventRecord(b, s);
    h->ev_pending.push_back({stage, a, b});
  }
  cudaEvent_t get_event() {
    if (!h->ev_free.empty()) {
      cudaEvent_t e = h->ev_free.back();
      h->ev_free.pop_back();
      return e;
    }
    cudaEvent_t e;
    CK(cudaEventCreate(&e));
    return e;
  }
  void pre_launch(int kc) {
    if (h->cfg.profile) {
      h->ev_cur = get_event();
      cudaEventRecord(h->ev_cur, s);
    }
  }
  void post_launch(int kc) {
    h->launches++;
    h->kc_launches[kc]++;
    if (h->cfg.profile) {
      cudaEvent_t b = get_event();
      cudaEventRecord(b, s);
      h->ev_pending.push_back({kc, h->ev_cur, b});
    }
    CK(cudaGetLastError());
  }
  void fetch(int count) {
    CK(cudaMemcpyAsync(h->hscal, h->dscal, sizeof(double) * count, cudaMemcpyDeviceToHost, s));
    sync();
  }
  void copy(double *dst, const double *src, int64_t m) {
    if (m) CK(cudaMemcpyAsync(dst, src, sizeof(double) * m, cudaMemcpyDeviceToDevice, s));
  }
  void zero(double *dst, int64_t m) {
    if (m) CK(cudaMemsetAsync(dst, 0, sizeof(double) * m, s));
  }
  unsigned int red_grid(int64_t work) {
    const int64_t b = (work + kRedThreads - 1) / kRedThreads;
    return (unsigned int)std::max<int64_t>(1, std::min<int64_t>(b, kRedBlocks));
  }

  // ---------------------------------------------------------------- multi-GPU helpers
  bool dist() const { return h->nranks > 1; }
  void allreduce(double *buf, int64_t count, int op = kNcclSum) {
    if (count > 0) NCK(nccl_api().AllReduce(buf, buf, (size_t)count, kNcclFloat64, op, h->comm, s));
  }
  SegList seglist(Amg &A, int J);
  void allreduce_shared(Amg &A, int J, double *v, double *extra = nullptr, int64_t nextra = 0);

  // ---------------------------------------------------------------- evaluation and vectors (evaluate.cu)
  static int group_for(const DevCsr &A) {
    const double avg = A.rows ? (double)A.nnz / (double)A.rows : 0.0;
    return avg > 48.0 ? 32 : (avg > 6.0 ? 4 : 1);
  }
  void spmv(const DevCsr &A, const double *x, const double *y0, double alpha, double *y, int G = 0);
  void axpby(int64_t m, double a, const double *x, double b, const double *y, double *out);
  void prolong_to_fine(Amg &A, int J, const double *x, const double *zbase, double *zf);
  void restrict_from_fine(Amg &A, int J, const double *gb, double *gJ);
  Dot2 dot2(Amg &A, int J, const double *a, const double *b);
  MaxAbs maxabs(int64_t n, const double *v);
  TrialOut eval_trial(Amg &A, int J, double t, double sigma);
  void phase1_slack(Amg &A, Amg &F);
  void blockgrad(Amg &A, const ElemParams &E);
  NodeParams node_params(Amg &A, double t);
  ElemParams elem_params(Amg &A);
  bool elem_fused_setup(Amg &A, const NodeParams &NP, int nex, ElemFused &Q, size_t &smem, unsigned int &grid);
  int plap_dim(const Amg &A) const;
  bool plap_setup(Amg &A, int dim, double t, bool use_bw, PlapParams &Q, size_t &smem, unsigned int &grid, bool cond = true);
  EvalOut eval_f01(Amg &A, int J, double t, const double *zbase, const double *x, double *gout, bool use_bw = true,
                   double *step2 = nullptr);

  // ---------------------------------------------------------------- system assembly (evaluate.cu; system_for: setup.cu)
  System &system_for(Amg &A, int J);
  void assemble(Amg &A, System &S, int J, double t, const double *zbase, const double *x);
  void assemble_unfused(Amg &A, System &S, int J, double t, const double *x);
  void galerkin(System &S, int kend);
  void schur_masks(const Amg &A, const System &S, unsigned &pieces, unsigned &elim) const;
  void assemble_dense(Amg &A, System &S, const NodeParams &P);
  void dgemm_nt(int M, int N, int K, const double *Am, int64_t lda, const double *Bm, int64_t ldb, const double *sc, double *C, int64_t ldc, bool acc, double alpha = 1.0);

  // ---------------------------------------------------------------- linear solve (linear_solve.cu)
  bool precond_fp32(const System &S) const;
  int lambda_power_its(const System &S) const;
  bool use_direct(const System &S, const SysLevel &Lv) const;
  std::vector<int> active_levels(const System &S, int ktop) const;
  void setup_hierarchy(Amg &A, System &S, int ktop);
  void dense_factor(SysLevel &Lv);
  void dense_apply(SysLevel &Lv, const double *b, double *x);      // x = A^{-1} b via factor (direct)
  void direct_solve(SysLevel &Lv, const double *b, double *x);
  SellBuild make_sell(const DevCsr &A, int64_t nthreads);
  void sell_prepare(System &S, int ktop);
  System::Pcg2Dev &pcg2_plan(System &S, int ktop);
  void pcg2_setup_dist(System::Pcg2Dev &D, int nshard);
  SolveResult pcg(System &S, int ktop, const double *b, double *x, const SolveTol &tol);
  SolveResult solve_compact(System &S, int ktop, const double *b, double *x, const SolveTol &tol);
  SolveResult solve(Amg &A, System &S, int J, const double *g, double *dir, const SolveTol &tol);

  // ---------------------------------------------------------------- Newton (newton.cu)
  struct NewtonOut {
    bool converged;
    int k;
    int status;   // MGBX_OK or MGBX_NON_FINITE
    double y, gnorm, inc;
  };
  NewtonOut newton(Amg &A, int J, double t, int maxit, int stop_kind, double lambda_tol, double theta, const mgbx_step_opts &o);
  int step(int which, double t, const mgbx_step_opts &o, mgbx_step_result *r);
  int matched_t(double t_default, double *t_out, double *tstar_out);
};

// raise the dynamic shared-memory limits of the kernels that need more than 48 KB (linear_solve.cu; evaluate.cu)
void solve_kernels_init();
void kron_w_init(size_t smem);

inline bool dense_mode(const Amg &A) { return A.N == 1 && A.p > 64; }

// M = kron(A, B) with A r1 x c1 and B r2 x c2 (row-major outputs)?  M(r, c) is any accessor.  The factors are fixed up to a
// scalar by taking B as the block through the entry of largest magnitude; the product is verified entry by entry.
template <class F>
bool kron_factor(F M, int r1, int r2, int c1, int c2, std::vector<double> &A, std::vector<double> &B) {
  const int64_t rows = (int64_t)r1 * r2, cols = (int64_t)c1 * c2;
  double best = 0.0;
  int64_t pr = 0, pc = 0;
  for (int64_t r = 0; r < rows; ++r)
    for (int64_t c = 0; c < cols; ++c) {
      const double v = std::fabs(M(r, c));
      if (v > best) {
        best = v;
        pr = r;
        pc = c;
      }
    }
  if (!(best > 0.0) || !std::isfinite(best)) return false;
  const int a0 = (int)(pr / r2), b0 = (int)(pr % r2), g0 = (int)(pc / c2), d0 = (int)(pc % c2);
  A.assign((size_t)r1 * c1, 0.0);
  B.assign((size_t)r2 * c2, 0.0);
  for (int b = 0; b < r2; ++b)
    for (int d = 0; d < c2; ++d) B[(size_t)b * c2 + d] = M((int64_t)a0 * r2 + b, (int64_t)g0 * c2 + d);
  const double piv = B[(size_t)b0 * c2 + d0];
  for (int a = 0; a < r1; ++a)
    for (int g = 0; g < c1; ++g) A[(size_t)a * c1 + g] = M((int64_t)a * r2 + b0, (int64_t)g * c2 + d0) / piv;
  const double tol = 1e-12 * best;
  for (int64_t r = 0; r < rows; ++r)
    for (int64_t c = 0; c < cols; ++c)
      if (std::fabs(M(r, c) - A[(size_t)(r / r2) * c1 + (c / c2)] * B[(size_t)(r % r2) * c2 + (c % c2)]) > tol) return false;
  return true;
}
inline int isqrt_exact(int64_t v) {
  const int r = (int)std::llround(std::sqrt((double)v));
  return ((int64_t)r * r == v) ? r : 0;
}

std::unique_ptr<System> build_system(mgbx_handle *h, Amg &A, bool condensed, int ltop);
void upload_convex(mgbx_handle *h, const mgbx_convex &Q, int64_t n, int nD_user, ConvexDev &cd);
void create_amg(mgbx_handle *h, const mgbx_amg &in, Amg &A);
void attach_feasibility(mgbx_handle *h, const mgbx_amg &a1);

}  // namespace mgbx
