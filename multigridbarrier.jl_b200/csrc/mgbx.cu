// mgbx.cu -- handle, setup plans, device-resident Newton / line search / mgb_step, and the C ABI.
//
// Reference behaviour implemented here (paths under /root/reference/src):
//   newton.jl:227-287          newton          -> Engine::newton
//   newton.jl:35-50,139-154    backtracking    -> Engine::newton (inlined trial loop)
//   newton.jl:187,222-225      stopping rules  -> Engine::stop_test
//   mgb.jl:10-82               divide_and_conquer / mgb_step -> Engine::step
//   mgb.jl:307-330             _matched_t      -> Engine::matched_t
//   convex.jl:155-202          f0 / f1 / f2    -> Engine::eval_f01 / assemble
//   BlockMatrices.jl:322-555   assembly plan   -> build_system (once; plans built on the device) + k_elem*/k_sell_gather
//   utils.jl:142-145           solve           -> Engine::solve (dense Cholesky or V-cycle PCG)
// The t-ramp (mgb_core) and phase-I control flow (mgb_driver) stay on the host side of the ABI:
// they only exchange scalars with this library.
#include <cuda_runtime.h>
#include <dlfcn.h>

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
#include "kernels.cuh"
#include "solver_kernels.cuh"
#include "setup_kernels.cuh"
#include "dense_kernels.cuh"
#include "pcg2.hpp"
#include "host_amg.hpp"

using namespace mgbx;

#define CK(call)                                                                                      \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess)                                                                            \
      throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " + __FILE__ + ":" + \
                               std::to_string(__LINE__));                                             \
  } while (0)

static thread_local std::string g_last_error;

// kernel classes for the optional per-class device timing (cfg.profile) and launch statistics
enum KClass { KC_NODE_F01 = 0, KC_NODE_F2, KC_BLOCKGRAD, KC_BLOCKHESS, KC_GATHER, KC_SPMV, KC_SPGEMM, KC_VEC, KC_COND,
              KC_DENSE, KC_PCG, KC_ELEM_F01, KC_ELEM_F2, KC_DGEMM, KC_ELEMG_F01, KC_ELEMG_F2, KC_COUNT };
static const char *kKClassNames[KC_COUNT] = {"node_f01", "node_f2", "blockgrad", "blockhess", "csr_gather", "spmv", "spgemm",
                                             "vector", "condense", "dense", "pcg_persistent", "elem_f01", "elem_f2", "dgemm_dmma", "elem_generic_f01", "elem_generic_f2"};
enum { STAGE_F01 = -1, STAGE_F2 = -2, STAGE_SOLVE = -3 };
#define LAUNCH(kc, ...)   \
  do {                    \
    pre_launch(kc);       \
    __VA_ARGS__;          \
    post_launch(kc);      \
  } while (0)
#define E_LAUNCH(kc, ...) \
  do {                    \
    E.pre_launch(kc);     \
    __VA_ARGS__;          \
    E.post_launch(kc);    \
  } while (0)

namespace {

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
// NCCL, loaded on demand (multi-GPU runs only): the few entry points used, declared here so that the
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
NcclApi &nccl_api() {
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

DevCsr upload_csr(Pool &pool, const HostCsr &H, cudaStream_t s, bool with_values = true) {
  DevCsr D;
  D.rows = H.rows;
  D.cols = H.cols;
  D.nnz = H.nnz();
  D.ptr = pool.upload<int64_t>(H.ptr.data(), H.ptr.size(), s);
  D.idx = pool.upload<int32_t>(H.idx.data(), H.idx.size(), s);
  if (with_values && !H.val.empty()) D.val = pool.upload<double>(H.val.data(), H.val.size(), s);
  else D.val = pool.zeros<double>(H.idx.size(), s);
  return D;
}


// temporary device CSR (plan construction only), freed explicitly
struct TempCsr {
  DevCsr d;
  cudaStream_t s = nullptr;
  void free_all() {
    if (d.ptr) cudaFreeAsync(d.ptr, s);
    if (d.idx) cudaFreeAsync(d.idx, s);
    if (d.val) cudaFreeAsync(d.val, s);
    d = DevCsr();
  }
};
TempCsr upload_csr_temp(const HostCsr &H, cudaStream_t s, bool with_values) {
  TempCsr T;
  T.s = s;
  T.d.rows = H.rows;
  T.d.cols = H.cols;
  T.d.nnz = H.nnz();
  CK(cudaMallocAsync((void **)&T.d.ptr, sizeof(int64_t) * (H.rows + 1), s));
  CK(cudaMallocAsync((void **)&T.d.idx, sizeof(int32_t) * std::max<int64_t>(1, H.nnz()), s));
  CK(cudaMemcpyAsync(T.d.ptr, H.ptr.data(), sizeof(int64_t) * (H.rows + 1), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(T.d.idx, H.idx.data(), sizeof(int32_t) * H.nnz(), cudaMemcpyHostToDevice, s));
  if (with_values && !H.val.empty()) {
    CK(cudaMallocAsync((void **)&T.d.val, sizeof(double) * std::max<int64_t>(1, H.nnz()), s));
    CK(cudaMemcpyAsync(T.d.val, H.val.data(), sizeof(double) * H.nnz(), cudaMemcpyHostToDevice, s));
  }
  CK(cudaStreamSynchronize(s));
  return T;
}

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

// (row << 32 | col) keys (unsorted, duplicates allowed) -> CSR pattern with sorted columns; consumes `keys`.
// drop_sentinel: keys equal to ~0 (padding of the multi-GPU all-gather) are discarded.
DevCsr csr_from_keys(Pool &pool, unsigned long long *keys, int64_t total, int64_t rows, int64_t cols, bool drop_sentinel, cudaStream_t s) {
  DevCsr C;
  C.rows = rows;
  C.cols = cols;
  if (total > INT32_MAX) throw std::runtime_error("csr_from_keys: more than 2^31 candidate entries");
  unsigned long long *keys2 = tmp_alloc<unsigned long long>(total, s);
  int *nsel = tmp_alloc<int>(1, s);
  int nnz = 0;
  if (total > 0) {
    size_t tmp_bytes = 0;
    const int end_bit = 64;
    CK(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, keys, keys2, (int)total, 0, end_bit, s));
    char *tmp = tmp_alloc<char>(tmp_bytes, s);
    CK(cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, keys, keys2, (int)total, 0, end_bit, s));
    tmp_free(tmp, s);
    CK(cub::DeviceSelect::Unique(nullptr, tmp_bytes, keys2, keys, nsel, (int)total, s));
    tmp = tmp_alloc<char>(tmp_bytes, s);
    CK(cub::DeviceSelect::Unique(tmp, tmp_bytes, keys2, keys, nsel, (int)total, s));
    tmp_free(tmp, s);
    CK(cudaMemcpyAsync(&nnz, nsel, sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (drop_sentinel && nnz > 0) {
      unsigned long long last = 0;
      CK(cudaMemcpyAsync(&last, keys + (nnz - 1), sizeof(last), cudaMemcpyDeviceToHost, s));
      CK(cudaStreamSynchronize(s));
      if (last == ~0ull) --nnz;
    }
  }
  C.nnz = nnz;
  C.ptr = pool.alloc<int64_t>(C.rows + 1);
  C.idx = pool.alloc<int32_t>(C.nnz);
  C.val = pool.zeros<double>(C.nnz, s);
  k_sym_finish<<<nblk(std::max<int64_t>(C.nnz, C.rows + 1)), 256, 0, s>>>(keys, C.nnz, C.rows, C.ptr, C.idx);
  CK(cudaGetLastError());
  tmp_free(keys, s);
  tmp_free(keys2, s);
  tmp_free(nsel, s);
  CK(cudaStreamSynchronize(s));
  return C;
}

// Multi-GPU: the union over the ranks of the local top-level patterns (each rank sees only its elements), so that
// every rank assembles into the SAME CSR structure and the values can be all-reduced.
DevCsr global_pattern(int nranks, void *comm, Pool &pool, const HostCsr &pat, cudaStream_t s) {
  NcclApi &N = nccl_api();
  const int64_t nloc = pat.nnz();
  std::vector<unsigned long long> hk(nloc);
  for (int64_t i = 0; i < pat.rows; ++i)
    for (int64_t k = pat.ptr[i]; k < pat.ptr[i + 1]; ++k) hk[k] = ((unsigned long long)i << 32) | (unsigned int)pat.idx[k];
  int64_t *dcnt = tmp_alloc<int64_t>(nranks + 1, s);
  CK(cudaMemcpyAsync(dcnt + nranks, &nloc, sizeof(int64_t), cudaMemcpyHostToDevice, s));
  NCK(N.AllGather(dcnt + nranks, dcnt, 1, kNcclInt64, comm, s));
  std::vector<int64_t> cnt(nranks);
  CK(cudaMemcpyAsync(cnt.data(), dcnt, sizeof(int64_t) * nranks, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  tmp_free(dcnt, s);
  const int64_t maxc = *std::max_element(cnt.begin(), cnt.end());
  unsigned long long *send = tmp_alloc<unsigned long long>(maxc, s);
  unsigned long long *all = tmp_alloc<unsigned long long>(maxc * nranks, s);
  CK(cudaMemsetAsync(send, 0xff, sizeof(unsigned long long) * std::max<int64_t>(1, maxc), s));
  CK(cudaMemcpyAsync(send, hk.data(), sizeof(unsigned long long) * nloc, cudaMemcpyHostToDevice, s));
  NCK(N.AllGather(send, all, (size_t)maxc, kNcclUint64, comm, s));
  CK(cudaStreamSynchronize(s));
  tmp_free(send, s);
  return csr_from_keys(pool, all, maxc * nranks, pat.rows, pat.cols, true, s);
}

// Sparsity pattern of A*B on the device: candidate keys (row << 32 | col) -> radix sort -> unique -> CSR.
DevCsr device_symbolic(Pool &pool, const DevCsr &A, const DevCsr &B, cudaStream_t s) {
  if (A.cols != B.rows) throw std::runtime_error("device_symbolic: inner dimensions differ");
  DevCsr C;
  C.rows = A.rows;
  C.cols = B.cols;
  int64_t *cand = tmp_alloc<int64_t>(A.rows + 1, s), *offs = tmp_alloc<int64_t>(A.rows + 1, s);
  k_sym_count<<<nblk(A.rows + 1), 256, 0, s>>>(A, B, cand);
  CK(cudaGetLastError());
  size_t tmp_bytes = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, cand, offs, (int)(A.rows + 1), s));
  char *tmp = tmp_alloc<char>(tmp_bytes, s);
  CK(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, cand, offs, (int)(A.rows + 1), s));
  int64_t total = 0;
  CK(cudaMemcpyAsync(&total, offs + A.rows, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  tmp_free(tmp, s);
  if (total > INT32_MAX) {
    tmp_free(cand, s);
    tmp_free(offs, s);
    throw std::runtime_error("device_symbolic: more than 2^31 candidate entries");
  }
  unsigned long long *keys = tmp_alloc<unsigned long long>(total, s);
  if (total > 0) {
    k_sym_fill<<<nblk(A.rows), 256, 0, s>>>(A, B, offs, keys);
    CK(cudaGetLastError());
  }
  tmp_free(cand, s);
  tmp_free(offs, s);
  return csr_from_keys(pool, keys, total, C.rows, C.cols, false, s);
}

// two-pass sliced-ELL construction shared by the device plan builders: COUNT(P, width) then FILL(P)
template <class CountFn, class FillFn>
SellPlan build_sell_two_pass(Pool &pool, int64_t nout, bool with_weights, cudaStream_t s, CountFn count, FillFn fill) {
  SellPlan P;
  P.nout = nout;
  P.nslices = (nout + 31) / 32;
  if (nout == 0) return P;
  int32_t *width = tmp_alloc<int32_t>(P.nslices, s);
  P.cnt = pool.alloc<int32_t>(nout);
  count(P, width);
  CK(cudaGetLastError());
  std::vector<int32_t> hwid(P.nslices);
  CK(cudaMemcpyAsync(hwid.data(), width, sizeof(int32_t) * P.nslices, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  std::vector<int64_t> sptr(P.nslices + 1, 0);
  for (int64_t sl = 0; sl < P.nslices; ++sl) sptr[sl + 1] = sptr[sl] + 32 * (int64_t)hwid[sl];
  P.nterms = sptr[P.nslices];
  P.sptr = pool.upload<int64_t>(sptr.data(), sptr.size(), s);
  P.src = pool.zeros<int32_t>(P.nterms, s);
  P.w = with_weights ? pool.zeros<double>(P.nterms, s) : nullptr;
  fill(P, width);
  CK(cudaGetLastError());
  tmp_free(width, s);
  CK(cudaStreamSynchronize(s));
  return P;
}

// Term list of the sparse product C = Lm * Rm, built on the device (one thread per non-zero of C; two passes).
SellPlan device_product_plan(Pool &pool, const DevCsr &Lm, const DevCsr &Rm, const DevCsr &C, bool variable_left, cudaStream_t s) {
  if (Lm.nnz > INT32_MAX || Rm.nnz > INT32_MAX || C.rows > INT32_MAX) throw std::runtime_error("product plan: index exceeds 32 bits");
  if (C.nnz == 0) return SellPlan();
  int32_t *rowof = tmp_alloc<int32_t>(C.nnz, s);
  k_csr_rows<<<nblk(C.rows), 256, 0, s>>>(C, rowof);
  const unsigned int g = nblk(((C.nnz + 31) / 32) * 32);
  const int vl = variable_left ? 1 : 0;
  SellPlan P = build_sell_two_pass(
      pool, C.nnz, true, s, [&](SellPlan &Q, int32_t *width) { k_prod_plan<0><<<g, 256, 0, s>>>(Lm, Rm, C, rowof, vl, Q, width); },
      [&](SellPlan &Q, int32_t *width) { k_prod_plan<1><<<g, 256, 0, s>>>(Lm, Rm, C, rowof, vl, Q, width); });
  tmp_free(rowof, s);
  return P;
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
  bool has_coarser = false, T_identity = false;
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
  bool dense_elements = false;       // spectral-type geometry (one dense "element"): small systems are solved directly
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
  // fine-level system with a slack-like variable (only :id rows) that could NOT be eliminated node-locally (e.g. a slack in
  // :broken_P1): its 1/slack^2 entries stay in the matrix, which the V-cycle PCG cannot solve reliably late in the t-ramp
  bool uncondensed_slack = false;
  std::vector<KronPair> kp;
  double *Wcat = nullptr;
  // PCG work at the largest size
  double *pc_r = nullptr, *pc_p = nullptr, *pc_Ap = nullptr, *pc_x = nullptr, *pc_b = nullptr;
  // solve kernel: one plan per top level
  struct Pcg2Dev {
    Pcg2Plan host;
    Pcg2Plan *dev = nullptr;
    size_t smem = 0;
    // multi-GPU row-sharded solve: this rank's exchange arena (cudaMalloc, exported by CUDA IPC) and the peers' mappings
    char *arena = nullptr;
    size_t arena_bytes = 0;
    void *peer[kPcg2MaxRanks] = {nullptr};
  };
  std::map<int, Pcg2Dev> pplans2;
  double *pc_p2 = nullptr, *pcg_partials = nullptr, *pcg_out = nullptr;
  unsigned int *pcg_bar = nullptr;
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

}  // namespace

struct mgbx_handle {
  std::string err;
  mgbx_config cfg;
  cudaStream_t stream = nullptr;
  Pool pool;
  Amg amg[2];
  bool has_feas = false;
  // reduction scratch
  double *partials = nullptr;
  unsigned int *ticket = nullptr;
  double *dscal = nullptr;   // device scalars
  double *hscal = nullptr;   // pinned host mirror
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // stats of the current step
  mgbx_step_result *res = nullptr;
  mgbx_step_result scratch_res;
  int64_t launches = 0;
  // per-class statistics; device time only when cfg.profile != 0
  int64_t kc_launches[KC_COUNT] = {0};
  double kc_ms[KC_COUNT] = {0};
  std::vector<cudaEvent_t> ev_free;
  struct Pending {
    int kc;
    cudaEvent_t a, b;
  };
  std::vector<Pending> ev_pending;
  cudaEvent_t ev_cur = nullptr;
  int pcg2_grid = 0;         // CTAs of the solve kernel k_pcg2
  double dgemm_flops = 0.0;   // FP64 tensor-core flops issued so far (spectral path)
  double cur_rtol2 = 1e-22;
  int cur_window = 25;       // PCG stagnation window (iterations without a new best residual)
  int last_solve_status = 1;       // 1 converged / direct, 2 stagnated above the tolerance, 3 iteration limit, -1 breakdown
  double last_solve_rel = 0.0;     // final relative residual |r| / |b| of the last PCG solve (0 for a direct solve)
  double last_solve_erel = 0.0;    // share of the direction's energy b.x = |x|_A^2 gained in the last four PCG iterations
  // multi-GPU
  int rank = 0, nranks = 1;
  void *comm = nullptr;
  int device = -1;           // CUDA device ordinal the handle lives on (made current at every ABI entry point)
  // phase profile of the solve kernel k_pcg2 (env MGBX_PCG_PROF=1): summed ns and counts per tag (level * 16 + kind)
  std::vector<double> prof_ns;
  std::vector<int64_t> prof_cnt;
  std::vector<unsigned long long> prof_host;
};

namespace {


// per-node kernel, instantiated for array bounds NDT in {4, 6, 8, 12}
template <int MODE>
void launch_node(const NodeParams &P, unsigned int grid, cudaStream_t s) {
  if (P.nD <= 4) k_node<MODE, 4><<<grid, kRedThreads, 0, s>>>(P);
  else if (P.nD <= 6) k_node<MODE, 6><<<grid, kRedThreads, 0, s>>>(P);
  else if (P.nD <= 8) k_node<MODE, 8><<<grid, kRedThreads, 0, s>>>(P);
  else k_node<MODE, MGBX_MAX_ND><<<grid, kRedThreads, 0, s>>>(P);
}

// fused element kernel (k_elem), same NDT dispatch; the dynamic shared-memory limit is raised once per instantiation
template <int MODE, int NDT>
void launch_elem_inst(const ElemFused &Q, unsigned int grid, size_t smem, cudaStream_t s) {
  static bool attr_done = false;
  static int nsm = 0;
  if (!attr_done) {
    CK(cudaFuncSetAttribute(k_elem<MODE, NDT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    int dev = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
    attr_done = true;
  }
  int occ = 1;   // one wave of resident CTAs walking the tiles
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_elem<MODE, NDT>, 256, smem));
  const unsigned int wave = (unsigned int)std::min(std::max(1, occ) * nsm, kRedBlocks);
  k_elem<MODE, NDT><<<std::min(grid, wave), 256, smem, s>>>(Q);
}
template <int MODE>
void launch_elem(const ElemFused &Q, unsigned int grid, size_t smem, cudaStream_t s) {
  if (Q.np.nD <= 4) launch_elem_inst<MODE, 4>(Q, grid, smem, s);
  else if (Q.np.nD <= 6) launch_elem_inst<MODE, 6>(Q, grid, smem, s);
  else if (Q.np.nD <= 8) launch_elem_inst<MODE, 8>(Q, grid, smem, s);
  else launch_elem_inst<MODE, MGBX_MAX_ND>(Q, grid, smem, s);
}

// specialised fused kernel of the default problem family (k_elem_plap)
template <int MODE, int DIM, bool COND>
void launch_plap_inst(const PlapParams &Q, unsigned int grid, size_t smem, cudaStream_t s) {
  static bool attr_done = false;
  static int nsm = 0;
  if (!attr_done) {
    CK(cudaFuncSetAttribute(k_elem_plap<MODE, DIM, COND>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    int dev = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
    attr_done = true;
  }
  // persistent tiles: exactly one wave of resident CTAs (grid = SMs x occupancy), never more than the reduction slots
  int occ = 1;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_elem_plap<MODE, DIM, COND>, 256, smem));
  const unsigned int wave = (unsigned int)std::min(std::max(1, occ) * nsm, kRedBlocks);
  k_elem_plap<MODE, DIM, COND><<<std::min(grid, wave), 256, smem, s>>>(Q);
}
template <int MODE>
void launch_plap(int dim, bool cond, const PlapParams &Q, unsigned int grid, size_t smem, cudaStream_t s) {
  if (cond || MODE == NODE_F01) {
    if (dim == 1) launch_plap_inst<MODE, 1, true>(Q, grid, smem, s);
    else if (dim == 2) launch_plap_inst<MODE, 2, true>(Q, grid, smem, s);
    else launch_plap_inst<MODE, 3, true>(Q, grid, smem, s);
  } else {
    if (dim == 1) launch_plap_inst<NODE_F2, 1, false>(Q, grid, smem, s);
    else if (dim == 2) launch_plap_inst<NODE_F2, 2, false>(Q, grid, smem, s);
    else launch_plap_inst<NODE_F2, 3, false>(Q, grid, smem, s);
  }
}

struct Engine {
  mgbx_handle *h;
  cudaStream_t s;
  explicit Engine(mgbx_handle *hh) : h(hh), s(hh->stream) {}

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

  // ---------------------------------------------------------------- sparse helpers
  static int group_for(const DevCsr &A) {
    const double avg = A.rows ? (double)A.nnz / (double)A.rows : 0.0;
    return avg > 48.0 ? 32 : (avg > 6.0 ? 4 : 1);
  }
  void spmv(const DevCsr &A, const double *x, const double *y0, double alpha, double *y, int G = 0) {
    if (A.rows == 0) return;
    if (G == 0) G = group_for(A);
    pre_launch(KC_SPMV);
    if (G == 32) k_spmv<32><<<nblk(A.rows * 32), 256, 0, s>>>(A, x, y0, alpha, y);
    else if (G == 4) k_spmv<4><<<nblk(A.rows * 4), 256, 0, s>>>(A, x, y0, alpha, y);
    else k_spmv<1><<<nblk(A.rows), 256, 0, s>>>(A, x, y0, alpha, y);
    post_launch(KC_SPMV);
  }
  void copy(double *dst, const double *src, int64_t m) {
    if (m) CK(cudaMemcpyAsync(dst, src, sizeof(double) * m, cudaMemcpyDeviceToDevice, s));
  }
  void zero(double *dst, int64_t m) {
    if (m) CK(cudaMemsetAsync(dst, 0, sizeof(double) * m, s));
  }

  // ---------------------------------------------------------------- level chain
  // zf = z + R_L * T_{L-2} ... T_J * x
  void prolong_to_fine(Amg &A, int J, const double *x, const double *zbase, double *zf) {
    const double *v = x;
    for (int l = J; l < A.L - 1; ++l) {
      spmv(A.T[l], v, nullptr, 1.0, A.chain[l + 1]);
      v = A.chain[l + 1];
    }
    spmv(A.RL, v, zbase, 1.0, zf);
  }
  // g_J = T_J' ... T_{L-2}' R_L' gb
  void restrict_from_fine(Amg &A, int J, const double *gb, double *gJ) {
    if (J == A.L - 1) {
      spmv(A.RLt, gb, nullptr, 1.0, gJ);
      return;
    }
    spmv(A.RLt, gb, nullptr, 1.0, A.chain2[A.L - 1]);
    const double *v = A.chain2[A.L - 1];
    for (int l = A.L - 2; l >= J; --l) {
      double *out = (l == J) ? gJ : A.chain2[l];
      spmv(A.Tt[l], v, nullptr, 1.0, out);
      v = out;
    }
  }


  // ---------------------------------------------------------------- multi-GPU helpers
  bool dist() const { return h->nranks > 1; }
  SegList seglist(Amg &A, int J) {
    SegList S;
    memset(&S, 0, sizeof(S));
    if (J == A.L - 1) {
      S.n = A.nu;
      for (int v = 0; v < A.nu; ++v) {
        S.off[v] = A.voff[J][v];
        S.local[v] = A.var_local[v];
      }
      S.off[A.nu] = A.voff[J][A.nu];
    } else {
      S.n = 1;
      S.off[0] = 0;
      S.off[1] = A.m[J];
    }
    return S;
  }
  void allreduce(double *buf, int64_t count, int op = kNcclSum) {
    if (count > 0) NCK(nccl_api().AllReduce(buf, buf, (size_t)count, kNcclFloat64, op, h->comm, s));
  }
  // sum the shared segments of a level-J vector over the ranks (the local segments are already complete)
  void allreduce_shared(Amg &A, int J, double *v, double *extra = nullptr, int64_t nextra = 0) {
    const SegList S = seglist(A, J);
    NCK(nccl_api().GroupStart());
    for (int q = 0; q < S.n; ++q)
      if (!S.local[q]) allreduce(v + S.off[q], S.off[q + 1] - S.off[q]);
    if (extra) allreduce(extra, nextra);
    NCK(nccl_api().GroupEnd());
  }
  // hscal[4..6] = {a.b, a.a, #non-finite(a)} over a level-J vector (all ranks obtain the same values)
  void dot2_fetch(Amg &A, int J, const double *a, const double *b) {
    const int64_t m = A.m[J];
    if (!dist()) {
      LAUNCH(KC_VEC, k_dot2<<<red_grid(m), kRedThreads, 0, s>>>(m, a, b, h->partials, h->ticket, h->dscal + 4));
      fetch(8);
      return;
    }
    LAUNCH(KC_VEC, k_dot2_seg<<<red_grid(m), kRedThreads, 0, s>>>(seglist(A, J), m, a, b, h->partials, h->ticket, h->dscal + 44));
    allreduce(h->dscal + 44, 3);
    fetch(64);
    for (int k = 0; k < 3; ++k) h->hscal[4 + k] = h->hscal[44 + k] + h->hscal[47 + k];
  }

  NodeParams node_params(Amg &A, double t) {
    NodeParams P;
    memset(&P, 0, sizeof(P));
    P.n = A.n;
    P.p = A.p;
    P.nu = A.nu;
    P.nD = A.nD;
    for (int j = 0; j < A.nD; ++j) {
      P.D_var[j] = A.D_var[j];
      P.D_op[j] = A.D_op[j];
    }
    for (int o = 0; o < A.nops; ++o) P.ops[o] = A.ops[o];
    P.zf = A.zf;
    P.w = A.w;
    P.f = A.f;
    P.bw = A.bw;
    P.t = t;
    P.inv_n = 1.0 / (double)A.n_global;
    P.cd = A.cd;
    P.G = A.G;
    P.partials = h->partials;
    P.ticket = h->ticket;
    P.red_out = h->dscal;
    P.slack = A.slack;
    return P;
  }
  ElemParams elem_params(Amg &A) {
    ElemParams P;
    memset(&P, 0, sizeof(P));
    P.n = A.n;
    P.N = A.N;
    P.p = A.p;
    P.nD = A.nD;
    for (int j = 0; j < A.nD; ++j) {
      P.D_var[j] = A.D_var[j];
      P.D_op[j] = A.D_op[j];
    }
    for (int o = 0; o < A.nops; ++o) P.ops[o] = A.ops[o];
    P.nK = A.nD;
    for (int j = 0; j < A.nD; ++j) P.Krow[j] = j;
    return P;
  }

  // tile geometry of the fused element kernel; false: fall back to the separate node / block kernels
  // (operator blocks too large for shared memory, e.g. the dense spectral "element")
  bool elem_fused_setup(Amg &A, const NodeParams &NP, int nex, ElemFused &Q, size_t &smem, unsigned int &grid) {
    if (!h->cfg.fused || A.p > 256) return false;
    memset(&Q, 0, sizeof(Q));
    Q.np = NP;
    Q.N = A.N;
    Q.nops = A.nops;
    Q.p1 = A.p | 1;
    Q.ES = (A.p * Q.p1) | 1;
    Q.nex = nex;
    int epb = std::max(1, 256 / A.p);
    const size_t cap = 216 * 1024;
    while (epb > 1 && elem_fused_smem(A.nops, epb, Q.ES, A.nu, nex, A.p) > cap) epb = (epb + 1) / 2;
    smem = elem_fused_smem(A.nops, epb, Q.ES, A.nu, nex, A.p);
    if (smem > cap) return false;
    Q.epb = epb;
    const int64_t ntiles = (A.N + epb - 1) / epb;
    grid = (unsigned int)std::max<int64_t>(1, std::min<int64_t>(ntiles, kRedBlocks));
    return true;
  }

  // The default problem family (state (u, s), D = [u:id; u:d_1..d_dim; s:id], one Euclidean-power cone on rows 1..dim+1
  // with identity A, zero b, uniform p and mu): returns dim (1..3) if the specialised kernel applies, else 0.
  int plap_dim(const Amg &A) const {
    if (h->cfg.fused != 1 || A.nu != 2 || A.p >= 256) return 0;
    const int dim = A.nD - 2;
    if (dim < 1 || dim > 3) return 0;
    const int vu = A.D_var[0], vs = A.D_var[dim + 1];
    if (vu == vs || A.D_op[0] >= 0 || A.D_op[dim + 1] >= 0) return 0;
    for (int a = 1; a <= dim; ++a)
      if (A.D_var[a] != vu || A.D_op[a] < 0) return 0;
    const ConvexDev &cd = A.cd;
    if (cd.feas || cd.npieces != 1 || cd.select) return 0;
    const PieceDev &pc = cd.pc[0];
    if (pc.kind != MGBX_PIECE_EP || pc.ni != dim + 1 || pc.nc != dim + 1 || pc.A || pc.b || pc.p || pc.mu) return 0;
    for (int c = 0; c <= dim; ++c)
      if (pc.idx[c] != c + 1) return 0;
    return dim;
  }
  bool plap_setup(Amg &A, int dim, double t, bool use_bw, PlapParams &Q, size_t &smem, unsigned int &grid, bool cond = true) {
    memset(&Q, 0, sizeof(Q));
    Q.n = A.n;
    Q.N = A.N;
    Q.p = A.p;
    Q.p1 = A.p | 1;
    Q.ES = (A.p * Q.p1) | 1;
    // bulk staging (cfg.elem_bulk): operator slabs and node columns arrive by cp.async.bulk instead of one 8-byte cp.async per
    // double.  Odd p: the padded layout already equals the contiguous one (p1 == p, ES == p*p) -> one copy per operator slab;
    // even p: columns are padded to p + 2 (16-byte aligned, conflict-free transposed reads) -> one copy per block column.
    Q.bulk = 0;
    if (h->cfg.elem_bulk) {
      if (A.p & 1) {
        if (Q.p1 == A.p && Q.ES == A.p * A.p) Q.bulk = 1;
      } else {
        Q.p1 = A.p + 2;
        Q.ES = A.p * Q.p1;
        if (Q.ES % 16 == 0) Q.ES += 8;
        Q.bulk = 2;
      }
    }
    int epb = std::max(1, 256 / A.p);
    const size_t cap = 216 * 1024, want = 72 * 1024;   // aim at 3 resident CTAs per SM (double-buffered tiles)
    while (epb > 1 && elem_plap_smem(dim, epb, Q.ES, A.p, cond) > want && epb * A.p > 128) epb = (epb + 1) / 2;
    while (epb > 1 && elem_plap_smem(dim, epb, Q.ES, A.p, cond) > cap) epb = (epb + 1) / 2;
    if (Q.bulk && (epb & 1) && epb > 1) --epb;         // even tiles keep every slab a multiple of 16 bytes and 16-byte aligned
    if (Q.bulk && (epb & 1) && (A.p & 1)) Q.bulk = 0;  // a one-element tile of an odd element cannot be bulk-copied
    smem = elem_plap_smem(dim, epb, Q.ES, A.p, cond);
    if (smem > cap) return false;
    Q.epb = epb;
    Q.dp = make_fastdiv((unsigned int)A.p);
    Q.dpp = make_fastdiv((unsigned int)(A.p * A.p));
    for (int a = 0; a < dim; ++a) Q.ops[a] = A.ops[A.D_op[a + 1]];
    Q.zu = A.zf + (int64_t)A.D_var[0] * A.n;
    Q.zs = A.zf + (int64_t)A.D_var[dim + 1] * A.n;
    Q.w = A.w;
    Q.f = A.f;
    Q.bw = use_bw ? A.bw : nullptr;
    Q.t = t;
    Q.inv_n = 1.0 / (double)A.n_global;
    Q.pexp = A.cd.pc[0].p_uniform;
    Q.mu = A.cd.pc[0].mu_uniform;
    Q.partials = h->partials;
    Q.ticket = h->ticket;
    Q.red_out = dist() ? h->dscal + 40 : h->dscal;
    if (Q.bulk) {   // bulk copies need 16-byte aligned sources: every base pointer, and the column stride n of f / the state blocks
      auto al16 = [](const void *q) { return q == nullptr || ((uintptr_t)q & 15) == 0; };
      bool ok = al16(Q.zu) && al16(Q.zs) && al16(Q.w) && al16(Q.bw) && al16(Q.f) && (A.n % 2 == 0);
      for (int a = 0; a < dim; ++a) ok = ok && al16(Q.ops[a]);
      if (!ok) {   // fall back to the per-double staging with its own padding
        Q.bulk = 0;
        Q.p1 = A.p | 1;
        Q.ES = (A.p * Q.p1) | 1;
        smem = elem_plap_smem(dim, epb, Q.ES, A.p, cond);
        if (smem > cap) return false;
      }
    }
    const int64_t ntiles = (A.N + epb - 1) / epb;
    grid = (unsigned int)std::max<int64_t>(1, std::min<int64_t>(ntiles, kRedBlocks));
    return true;
  }
  unsigned int red_grid(int64_t work) {
    const int64_t b = (work + kRedThreads - 1) / kRedThreads;
    return (unsigned int)std::max<int64_t>(1, std::min<int64_t>(b, kRedBlocks));
  }

  // ---------------------------------------------------------------- f0 + f1 at level J
  // zbase: broken state the level correction is added to; x: level-J coefficients; gout: level-J gradient
  EvalOut eval_f01(Amg &A, int J, double t, const double *zbase, const double *x, double *gout, bool use_bw = true) {
    cudaEvent_t st = stage_begin();
    prolong_to_fine(A, J, x, zbase, A.zf);
    NodeParams P = node_params(A, t);
    if (!use_bw) P.bw = nullptr;
    if (dist()) P.red_out = h->dscal + 40;
    ElemFused Q;
    PlapParams PQ;
    size_t smem = 0;
    unsigned int grid = 0;
    const int pdim = plap_dim(A);
    if (pdim && plap_setup(A, pdim, t, use_bw, PQ, smem, grid)) {
      PQ.gbu = A.gb + (int64_t)A.D_var[0] * A.n;
      PQ.gbs = A.gb + (int64_t)A.D_var[pdim + 1] * A.n;
      LAUNCH(KC_ELEM_F01, launch_plap<NODE_F01>(pdim, true, PQ, grid, smem, s));
    } else if (elem_fused_setup(A, P, A.nD, Q, smem, grid)) {
      Q.gb = A.gb;
      LAUNCH(KC_ELEMG_F01, launch_elem<NODE_F01>(Q, grid, smem, s));
    } else {
      LAUNCH(KC_NODE_F01, launch_node<NODE_F01>(P, red_grid(A.n), s));
      ElemParams E = elem_params(A);
      LAUNCH(KC_BLOCKGRAD, k_blockgrad<<<nblk((int64_t)A.nu * A.n), 256, 0, s>>>(E, A.G, A.gb, A.nu));
    }
    restrict_from_fine(A, J, A.gb, gout);
    if (!dist()) {
      LAUNCH(KC_VEC, k_dot2<<<red_grid(A.m[J]), kRedThreads, 0, s>>>(A.m[J], gout, nullptr, h->partials, h->ticket, h->dscal + 4));
      stage_end(STAGE_F01, st);
      fetch(8);
    } else {
      // partial sums over this rank's elements -> all ranks: the shared part of R'g, the objective scalars, and the
      // local-part norms (one grouped all-reduce); the shared-part norm is then formed identically on every rank
      const SegList SG = seglist(A, J);
      LAUNCH(KC_VEC, k_dot2_seg<<<red_grid(A.m[J]), kRedThreads, 0, s>>>(SG, A.m[J], gout, nullptr, h->partials, h->ticket, h->dscal + 44));
      allreduce_shared(A, J, gout, h->dscal + 39, 8);   // [39] trial norm (local part), [40..43] node sums, [44..46] local dot
      LAUNCH(KC_VEC, k_dot2_seg<<<red_grid(A.m[J]), kRedThreads, 0, s>>>(SG, A.m[J], gout, nullptr, h->partials, h->ticket, h->dscal + 50));
      stage_end(STAGE_F01, st);
      fetch(64);
      for (int k = 0; k < 4; ++k) h->hscal[k] = h->hscal[40 + k];
      for (int k = 0; k < 3; ++k) h->hscal[4 + k] = h->hscal[44 + k] + h->hscal[53 + k];
      h->hscal[7] = h->hscal[38] + h->hscal[39];
      CK(cudaMemsetAsync(h->dscal + 38, 0, 2 * sizeof(double), s));   // the trial norms are consumed
    }
    if (h->res) h->res->f01_evals++;
    EvalOut o;
    const double bar = (use_bw && A.bw) ? h->hscal[0] : h->hscal[0] * (1.0 / (double)A.n_global);
    o.lin = h->hscal[1];
    o.y = bar + h->hscal[1];
    o.nonfinite_nodes = h->hscal[2];
    o.gnorm = std::sqrt(h->hscal[5]);
    o.finite = std::isfinite(o.y) && (h->hscal[6] == 0.0) && std::isfinite(h->hscal[5]);
    return o;
  }

  // ---------------------------------------------------------------- system assembly
  System &system_for(Amg &A, int J);
  // Systems with at most dense_direct_max unknowns are solved directly (shared-memory solve with pivoted fallback up to
  // 128, blocked DMMA Cholesky above): faster than PCG at these sizes and robust for the systems that could not be
  // condensed (e.g. a :broken_P1 slack), whose 1/slack^2 entries make them too ill-conditioned for an iterative solve.
  // FP32 copies of the level matrices for the preconditioner passes: on, off, or (2) automatic -- only when the top matrix
  // is far larger than the L2 cache, i.e. when the V-cycle is HBM-bound (measured -12% per PCG iteration at 26 M non-zeros,
  // neutral at 2 M)
  bool precond_fp32(const System &S) const {
    if (h->cfg.precond_fp32 != 2) return h->cfg.precond_fp32 == 1;
    int64_t tot = 0;                       // automatic: the level matrices together (12 B per entry) no longer fit the 126 MB L2
    for (const SysLevel &Lv : S.lev) tot += Lv.A.nnz;
    return tot >= 10000000;
  }
  // power iterations per level and assembly for lambda_max(D^-1 A): cfg.lambda_power, or automatic (-1): 6 when the top
  // matrix has long rows (3-D stencils: the Gershgorin bound overestimates 1.3-2.5x there and misplaces the Chebyshev
  // interval -- measured on fem3d 32^3: 14 194 -> 8 294 PCG iterations per solve), none on 2-D meshes (bound within 4 %)
  int lambda_power_its(const System &S) const {
    if (h->cfg.lambda_power >= 0) return h->cfg.lambda_power;
    if (S.lev.empty() || S.lev[0].A.rows == 0) return 0;
    return ((double)S.lev[0].A.nnz / (double)S.lev[0].A.rows > 16.0) ? 6 : 0;
  }
  bool use_direct(const System &S, const SysLevel &Lv) const {
    return S.dense || Lv.m <= h->cfg.dense_direct_max;   // dense (spectral) systems have no hierarchy: always direct
  }
  void assemble(Amg &A, System &S, int J, double t, const double *zbase, const double *x);
  void schur_masks(const Amg &A, const System &S, unsigned &pieces, unsigned &elim) const;
  void assemble_dense(Amg &A, System &S, const NodeParams &P);
  void dgemm_nt(int M, int N, int K, const double *Am, int64_t lda, const double *Bm, int64_t ldb, const double *sc, double *C, int64_t ldc, bool acc, double alpha = 1.0);
  void setup_hierarchy(Amg &A, System &S, int ktop);
  void dense_factor(System &S, SysLevel &Lv, bool want_inverse);
  void dense_apply(SysLevel &Lv, const double *b, double *x);      // x = A^{-1} b via factor (direct)
  // ---- solve kernel (pcg2.hpp)
  std::vector<int> active_levels(const System &S, int ktop) const {
    const int nlev = (int)S.lev.size();
    const int kend = (S.cut >= 0) ? std::max(S.cut, ktop) : nlev - 1;
    std::vector<int> act;
    for (int k = ktop; k <= kend; ++k) {
      if (k < kend && S.lev[k].T_identity) continue;   // same matrix as the next level
      act.push_back(k);
    }
    return act;
  }
  SellBuild make_sell(const DevCsr &A, int64_t nthreads);
  void sell_prepare(System &S, int ktop);
  System::Pcg2Dev &pcg2_plan(System &S, int ktop);
  void pcg2_setup_dist(System::Pcg2Dev &D, int nshard);
  int pcg(System &S, int ktop, const double *b, double *x);
  int solve_compact(System &S, int ktop, const double *b, double *x);
  int solve(Amg &A, System &S, int J, const double *g, double *dir);

  // ---------------------------------------------------------------- Newton
  struct NewtonOut {
    bool converged;
    int k;
    int status;   // MGBX_OK or MGBX_NON_FINITE
    double y, gnorm, inc;
  };
  bool stop_test(int kind, double lambda_tol, double theta, double ymin, double ynext, double gmin, double gnext, double ndec) {
    const bool ex = (ynext >= ymin) && (gnext >= theta * gmin);
    if (kind == 0) return ex;
    return (ndec < lambda_tol) || ex;
  }
  NewtonOut newton(Amg &A, int J, double t, int maxit, int stop_kind, double lambda_tol, double theta, const mgbx_step_opts &o);
  int step(int which, double t, const mgbx_step_opts &o, mgbx_step_result *r);
  int matched_t(double t_default, double *t_out, double *tstar_out);
};

// -------------------------------------------------------------------------------------------------
// host-side plan construction
// -------------------------------------------------------------------------------------------------
// Build the index plans of one linear-system family.  ltop: the AMG level the top matrix lives on.  The top
// matrix is assembled directly from the element blocks with R_top = R_fine[ltop] (= R_fine[L-1] * T[L-2] ... T[ltop]),
// every coarser level by Galerkin gather plans.
// spectral discretisations: one dense "element" (N == 1) with more nodes than a finite element ever has
inline bool dense_mode(const Amg &A) { return A.N == 1 && A.p > 64; }
constexpr int kDenseMaxUnknowns = 8192;   // blocked Cholesky: the triangular solve keeps the right-hand side in shared memory (64 KB)

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

std::unique_ptr<System> build_system(mgbx_handle *h, Amg &A, bool condensed, int ltop) {
  auto S = std::make_unique<System>();
  Pool &pool = h->pool;
  pool.cat = "system: patterns, gather plans, level vectors";
  cudaStream_t s = h->stream;
  const int L = ltop + 1;            // levels 0..ltop take part
  S->condensed = condensed;
  S->ltop = ltop;
  S->dense_elements = A.p > 64;
  if (condensed && ltop != A.L - 1) throw std::runtime_error("internal: condensation only at the fine level");
  // prolongation from the top level of this system to the broken fine space
  HostCsr Rtop_store;
  const HostCsr *Rtop_p = &A.hRL;
  if (ltop != A.L - 1) {
    Rtop_store = A.hRL;
    for (int l = A.L - 2; l >= ltop; --l) Rtop_store = spgemm_numeric_host(Rtop_store, A.hT[l]);
    Rtop_p = &Rtop_store;
  }
  const HostCsr &Rtop = *Rtop_p;
  // which variables can be eliminated node-locally at the fine level: R block == identity and every D row is :id
  std::vector<char> is_elim(A.nu, 0);
  if (condensed) {
    for (int v = 0; v < A.nu; ++v) {
      const int64_t c0 = A.voff[L - 1][v], c1 = A.voff[L - 1][v + 1];
      if (c1 - c0 != A.n) continue;
      bool idonly = true, any = false;
      for (int j = 0; j < A.nD; ++j)
        if (A.D_var[j] == v) {
          any = true;
          if (A.D_op[j] >= 0) idonly = false;
        }
      if (!any || !idonly) continue;
      HostCsr blk = submatrix(Rtop, (int64_t)v * A.n, (int64_t)(v + 1) * A.n, c0, c1);
      if (is_identity(blk)) is_elim[v] = 1;
    }
    int ne = 0;
    for (int v = 0; v < A.nu; ++v) ne += is_elim[v];
    if (ne > 4) {   // keep at most 4 eliminated variables (register budget of the node kernel)
      for (int v = A.nu - 1; v >= 0 && ne > 4; --v)
        if (is_elim[v]) {
          is_elim[v] = 0;
          --ne;
        }
    }
    if (ne == A.nu) is_elim[0] = 0;   // keep at least one variable in the reduced system
  }
  for (int v = 0; v < A.nu; ++v) (is_elim[v] ? S->elim : S->kept).push_back(v);
  S->nE = (int)S->elim.size();
  if (condensed)
    for (int v = 0; v < A.nu; ++v) {
      bool idonly = true, any = false;
      for (int j = 0; j < A.nD; ++j)
        if (A.D_var[j] == v) {
          any = true;
          if (A.D_op[j] >= 0) idonly = false;
        }
      if (any && idonly && !is_elim[v] && A.nu > 1) S->uncondensed_slack = true;
    }
  // row classification
  S->nK = 0;
  for (int j = 0; j < A.nD; ++j) {
    S->Erow[j] = -1;
    for (int e = 0; e < S->nE; ++e)
      if (S->elim[e] == A.D_var[j]) S->Erow[j] = e;
    if (S->Erow[j] < 0) S->Krow[S->nK++] = j;
  }
  // variables of the kept set that own at least one D row form the block pairs
  std::vector<int> used;
  for (int v : S->kept) {
    bool any = false;
    for (int j = 0; j < A.nD; ++j) any = any || (A.D_var[j] == v);
    if (any) used.push_back(v);
  }
  if ((int)(used.size() * used.size()) > 16) throw ArgError("too many coupled state variables (max 4 kept variables)");
  S->pl.npairs = 0;
  for (int a : used)
    for (int b : used) {
      S->pl.va[S->pl.npairs] = a;
      S->pl.vb[S->pl.npairs] = b;
      S->pl.npairs++;
    }
  // levels
  const int nlev = L;
  S->lev.resize(nlev);
  for (int k = 0; k < nlev; ++k) {
    const int l = L - 1 - k;
    SysLevel &Lv = S->lev[k];
    Lv.off.assign(1, 0);
    for (int v : S->kept) Lv.off.push_back(Lv.off.back() + (A.voff[l][v + 1] - A.voff[l][v]));
    Lv.m = Lv.off.back();
  }
  if (dense_mode(A)) {
    // ---- dense (spectral) system: full m x m matrix assembled by GEMMs, solved directly; no plans, no hierarchy
    S->dense = true;
    S->lev.resize(1);
    SysLevel &Lv = S->lev[0];
    const int64_t m = Lv.m;
    if (m > kDenseMaxUnknowns) throw std::runtime_error("dense (spectral) Newton systems are limited to 8192 unknowns in this build");
    HostCsr full;
    full.rows = full.cols = m;
    full.ptr.resize(m + 1);
    full.idx.resize((size_t)m * m);
    for (int64_t i = 0; i <= m; ++i) full.ptr[i] = i * m;
    for (int64_t i = 0; i < m; ++i)
      for (int64_t j = 0; j < m; ++j) full.idx[i * m + j] = (int32_t)j;
    Lv.A = upload_csr(pool, full, s, false);
    Lv.spmv_group = 32;
    Lv.dinv = pool.alloc<double>(m);
    Lv.diag = pool.alloc<double>(m);
    Lv.lam = pool.zeros<double>(1, s);
    Lv.b = pool.alloc<double>(m);
    Lv.x = pool.alloc<double>(m);
    Lv.x2 = pool.alloc<double>(m);
    Lv.r = pool.alloc<double>(m);
    TempCsr rt = upload_csr_temp(Rtop, s, true);
    int64_t mvmax = 1;
    for (size_t q = 0; q < S->kept.size(); ++q) {
      const int v = S->kept[q];
      const int64_t mv = Lv.off[q + 1] - Lv.off[q];
      mvmax = std::max(mvmax, mv);
      double *d = pool.zeros<double>((size_t)mv * A.n, s);
      k_csr_block_to_dense_t<<<nblk(A.n), 256, 0, s>>>(rt.d, (int64_t)v * A.n, (int)A.n, A.voff[L - 1][v], (int)mv, d);
      CK(cudaGetLastError());
      S->Rt.push_back(d);
    }
    CK(cudaStreamSynchronize(s));
    rt.free_all();
    S->Hd = pool.alloc<double>((size_t)A.n * A.n);
    S->Wt = pool.alloc<double>((size_t)mvmax * A.n);
    S->cut = -1;
    // ---- sum-factorised assembly when every operator and every prolongation block is a Kronecker product
    if (h->cfg.spectral_kron && A.kron_n1 > 0 && S->nE == 0) {
      const int n1 = A.kron_n1;
      const size_t nk = S->kept.size();
      std::vector<std::vector<double>> R1a(nk), R1b(nk);
      std::vector<int> cq(nk, 0);
      bool ok = true;
      for (size_t q = 0; q < nk && ok; ++q) {
        const int v = S->kept[q];
        const int64_t mv = Lv.off[q + 1] - Lv.off[q];
        const int c = isqrt_exact(mv);
        if (c <= 0 || c > n1) {
          ok = false;
          break;
        }
        std::vector<double> dense((size_t)A.n * mv, 0.0);
        const int64_t c0 = A.voff[L - 1][v];
        for (int64_t i = 0; i < A.n; ++i)
          for (int64_t k = Rtop.ptr[(int64_t)v * A.n + i]; k < Rtop.ptr[(int64_t)v * A.n + i + 1]; ++k) {
            const int64_t cc = Rtop.idx[k] - c0;
            if (cc >= 0 && cc < mv) dense[(size_t)i * mv + cc] = Rtop.val[k];
          }
        cq[q] = c;
        ok = kron_factor([&](int64_t r, int64_t cc) { return dense[(size_t)r * mv + cc]; }, n1, n1, c, c, R1a[q], R1b[q]);
      }
      if (ok) {
        // per D row j: P_j = A_j R1a_v, Q_j = B_j R1b_v  (n1 x c_v); identity operators have A_j = B_j = I
        std::vector<std::vector<double>> Pj(S->nK), Qj(S->nK);
        std::vector<const double *> Qdev(S->nK, nullptr);
        std::vector<int> qof(S->nK, -1);
        auto mul = [&](const std::vector<double> *F, const std::vector<double> &Rm, int c) {
          if (!F) return Rm;
          std::vector<double> out((size_t)n1 * c, 0.0);
          for (int e = 0; e < n1; ++e)
            for (int g = 0; g < n1; ++g) {
              const double f = (*F)[(size_t)e * n1 + g];
              if (f != 0.0)
                for (int i = 0; i < c; ++i) out[(size_t)e * c + i] += f * Rm[(size_t)g * c + i];
            }
          return out;
        };
        for (int a = 0; a < S->nK; ++a) {
          const int j = S->Krow[a], v = A.D_var[j], o = A.D_op[j];
          for (size_t q = 0; q < nk; ++q)
            if (S->kept[q] == v) qof[a] = (int)q;
          if (qof[a] < 0) continue;
          Pj[a] = mul(o >= 0 ? &A.kronA[o] : nullptr, R1a[qof[a]], cq[qof[a]]);
          Qj[a] = mul(o >= 0 ? &A.kronB[o] : nullptr, R1b[qof[a]], cq[qof[a]]);
          Qdev[a] = pool.upload<double>(Qj[a].data(), Qj[a].size(), s);
        }
        size_t wmax = 0;
        for (size_t qa = 0; qa < nk && ok; ++qa)
          for (size_t qb = 0; qb < nk && ok; ++qb) {
            System::KronPair kp;
            kp.c1a = kp.c2a = cq[qa];
            kp.c1b = kp.c2b = cq[qb];
            kp.offa = Lv.off[qa];
            kp.offb = Lv.off[qb];
            std::vector<std::pair<int, int>> combos;
            for (int ja = 0; ja < S->nK; ++ja)
              for (int kb = 0; kb < S->nK; ++kb)
                if (qof[ja] == (int)qa && qof[kb] == (int)qb) combos.push_back({ja, kb});
            if (combos.empty()) continue;
            if ((int)combos.size() > kKronMaxCombos) {
              ok = false;
              break;
            }
            kp.ncombo = (int)combos.size();
            const int64_t Mr = (int64_t)kp.c1a * kp.c1b, K = (int64_t)kp.ncombo * n1;
            std::vector<double> AA((size_t)Mr * K);
            for (int c = 0; c < kp.ncombo; ++c) {
              const int ja = combos[c].first, kb = combos[c].second;
              const int lo = std::min(ja, kb), hi = std::max(ja, kb);
              kp.hidx[c] = lo * S->nK - (lo * (lo - 1)) / 2 + (hi - lo);
              kp.Qj[c] = Qdev[ja];
              kp.Qk[c] = Qdev[kb];
              for (int i = 0; i < kp.c1a; ++i)
                for (int l = 0; l < kp.c1b; ++l)
                  for (int e = 0; e < n1; ++e)
                    AA[((size_t)i * kp.c1b + l) * K + (size_t)c * n1 + e] = Pj[ja][(size_t)e * kp.c1a + i] * Pj[kb][(size_t)e * kp.c1b + l];
            }
            kp.AA = pool.upload<double>(AA.data(), AA.size(), s);
            wmax = std::max(wmax, (size_t)kp.c2a * kp.c2b * (size_t)K);
            S->kp.push_back(kp);
          }
        if (ok && !S->kp.empty()) {
          S->Wcat = pool.alloc<double>(wmax);
          S->kron = true;
          const size_t smem = sizeof(double) * ((size_t)n1 + 2 * (size_t)n1 * n1);
          CK(cudaFuncSetAttribute(k_kron_w, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        } else {
          S->kp.clear();
        }
      }
      if (h->cfg.verbose > 0) fprintf(stderr, "[mgbx] build_system(dense, level %d): sum-factorised (Kronecker) assembly %s\n", ltop, S->kron ? "on" : "not applicable");
    }
    S->pc_r = pool.alloc<double>(m);
    S->pc_p = pool.alloc<double>(m);
    S->pc_p2 = pool.alloc<double>(m);
    S->pc_Ap = pool.alloc<double>(m);
    S->pc_x = pool.alloc<double>(m);
    S->pc_b = pool.alloc<double>(m);
    S->pcg_partials = pool.zeros<double>(3 * (size_t)kPcg2MaxGrid, s);
    S->pcg_out = pool.zeros<double>(8, s);
    S->pcg_bar = pool.zeros<unsigned int>(4, s);
    CK(cudaStreamSynchronize(s));
    if (h->cfg.verbose > 0) fprintf(stderr, "[mgbx] build_system(dense, level %d): m=%lld, n=%lld\n", ltop, (long long)m, (long long)A.n);
    return S;
  }
  // top pattern = reference plan pattern restricted to the kept variables
  const int64_t mtop = S->lev[0].m;
  std::vector<int64_t> colmap(A.m[L - 1], -1);
  for (size_t q = 0; q < S->kept.size(); ++q) {
    const int v = S->kept[q];
    for (int64_t c = A.voff[L - 1][v]; c < A.voff[L - 1][v + 1]; ++c) colmap[c] = S->lev[0].off[q] + (c - A.voff[L - 1][v]);
  }
  HostTimer tm;
  const bool vb = h->cfg.verbose > 0;
  HostCsr Einc = element_incidence(Rtop, A.N, A.p, used, A.n, colmap, mtop);
  HostCsr pat = plan_pattern(Einc);
  if (vb) fprintf(stderr, "[mgbx] build_system(cond=%d): pattern m=%lld nnz=%lld %.3fs\n", (int)condensed, (long long)mtop, (long long)pat.nnz(), tm.lap());   // (local pattern on a multi-GPU rank)
  // gather plan, built on the device: for each nz of the pattern, the Hblk entries (and weights) that sum into it
  const int p = A.p;
  const int64_t pp = (int64_t)p * p;
  S->hblk_size = (int64_t)S->pl.npairs * A.N * pp;
  if (S->hblk_size > INT32_MAX) throw std::runtime_error("element block array exceeds 32-bit gather indices");
  // multi-GPU: each rank sees only its own elements; the CSR structure is the union over the ranks
  S->lev[0].A = (h->nranks > 1) ? global_pattern(h->nranks, h->comm, pool, pat, s) : upload_csr(pool, pat, s, false);
  const int64_t top_nnz = S->lev[0].A.nnz;
  {
    bool unit = true;
    for (double v : Rtop.val)
      if (v != 1.0) {
        unit = false;
        break;
      }
    TempCsr einct = upload_csr_temp(transpose(Einc), s, false);
    TempCsr rtmp;
    TopPlanParams Q;
    memset(&Q, 0, sizeof(Q));
    if (ltop == A.L - 1) Q.R = A.RL;
    else {
      rtmp = upload_csr_temp(Rtop, s, true);
      Q.R = rtmp.d;
    }
    Q.EincT = einct.d;
    Q.pat = S->lev[0].A;
    Q.n = A.n;
    Q.N = A.N;
    Q.p = p;
    Q.unit = unit ? 1 : 0;
    Q.nkept = (int)S->kept.size();
    for (int q = 0; q < Q.nkept; ++q) {
      Q.kept[q] = S->kept[q];
      Q.off[q] = S->lev[0].off[q];
      Q.rcol0[q] = A.voff[L - 1][S->kept[q]];
    }
    Q.off[Q.nkept] = S->lev[0].off[Q.nkept];
    for (int qa = 0; qa < Q.nkept; ++qa)
      for (int qb = 0; qb < Q.nkept; ++qb) {
        int pr = -1;
        for (int k = 0; k < S->pl.npairs; ++k)
          if (S->pl.va[k] == S->kept[qa] && S->pl.vb[k] == S->kept[qb]) pr = k;
        Q.pair_of[qa * Q.nkept + qb] = pr;
      }
    int32_t *rowof = tmp_alloc<int32_t>(top_nnz, s);
    k_csr_rows<<<nblk(pat.rows), 256, 0, s>>>(S->lev[0].A, rowof);
    Q.rowof = rowof;
    const unsigned int g = nblk(((top_nnz + 31) / 32) * 32);
    S->top = build_sell_two_pass(
        pool, top_nnz, !unit, s, [&](SellPlan &P, int32_t *width) { k_top_plan<0><<<g, 256, 0, s>>>(Q, P, width); },
        [&](SellPlan &P, int32_t *width) { k_top_plan<1><<<g, 256, 0, s>>>(Q, P, width); });
    tmp_free(rowof, s);
    einct.free_all();
    if (rtmp.d.ptr) rtmp.free_all();
  }
  pool.cat = "system: element block Hessians";
  S->Hblk = pool.alloc<double>(S->hblk_size);
  pool.cat = "system: Galerkin patterns and term lists";
  if (vb) fprintf(stderr, "[mgbx]   gather plan (%lld padded terms) %.3fs\n", (long long)S->top.nterms, tm.lap());
  // hierarchy patterns (device symbolic products) and Galerkin gather plans
  for (int k = 0; k < nlev; ++k) {
    SysLevel &Lv = S->lev[k];
    const int l = L - 1 - k;
    Lv.spmv_group = Engine::group_for(Lv.A);
    Lv.dinv = pool.alloc<double>(Lv.m);
    Lv.diag = pool.alloc<double>(Lv.m);
    Lv.lam = pool.zeros<double>(1, s);
    Lv.b = pool.alloc<double>(Lv.m);
    Lv.x = pool.alloc<double>(Lv.m);
    Lv.x2 = pool.alloc<double>(Lv.m);
    Lv.r = pool.alloc<double>(Lv.m);
    if (k + 1 < nlev) {
      // transfer from level l-1 to level l restricted to the kept variables
      std::vector<HostCsr> blocks;
      for (int v : S->kept)
        blocks.push_back(submatrix(A.hT[l - 1], A.voff[l][v], A.voff[l][v + 1], A.voff[l - 1][v], A.voff[l - 1][v + 1]));
      HostCsr Tk = block_diag(blocks);
      Lv.has_coarser = true;
      Lv.T_identity = is_identity(Tk);
      HostCsr Ttk = transpose(Tk);
      Lv.T = upload_csr(pool, Tk, s);
      Lv.Tt = upload_csr(pool, Ttk, s);
      if (Lv.T_identity) {
        S->lev[k + 1].A = Lv.A;   // same matrix: the coarser level aliases this one
      } else {
        const double t_host = tm.lap();
        Lv.AT = device_symbolic(pool, Lv.A, Lv.T, s);
        S->lev[k + 1].A = device_symbolic(pool, Lv.Tt, Lv.AT, s);
        const double t_sym = tm.lap();
        Lv.s1 = device_product_plan(pool, Lv.A, Lv.T, Lv.AT, true, s);
        Lv.s2 = device_product_plan(pool, Lv.Tt, Lv.AT, S->lev[k + 1].A, false, s);
        if (vb)
          fprintf(stderr, "[mgbx]   level %d: m=%lld -> %lld, nnz(A_c)=%lld, plan entries %lld + %lld, host %.3fs symbolic %.3fs plans %.3fs\n", k,
                  (long long)Lv.m, (long long)S->lev[k + 1].m, (long long)S->lev[k + 1].A.nnz, (long long)Lv.s1.nterms, (long long)Lv.s2.nterms,
                  t_host, t_sym, tm.lap());
      }
    }
  }
  // V-cycle cut: the first level small enough for the shared-memory dense inverse
  S->cut = -1;
  for (int k = 0; k < nlev; ++k)
    if (S->lev[k].m <= h->cfg.coarse_max) {
      S->cut = k;
      break;
    }
  const int64_t mx = S->lev[0].m;
  S->pc_r = pool.alloc<double>(mx);
  S->pc_p = pool.alloc<double>(mx);
  S->pc_p2 = pool.alloc<double>(mx);
  S->pc_Ap = pool.alloc<double>(mx);
  S->pc_x = pool.alloc<double>(mx);
  S->pc_b = pool.alloc<double>(mx);
  S->pcg_partials = pool.zeros<double>(3 * (size_t)kPcg2MaxGrid, s);
  S->pcg_out = pool.zeros<double>(8, s);
  S->pcg_bar = pool.zeros<unsigned int>(4, s);
  CK(cudaStreamSynchronize(s));
  return S;
}

System &Engine::system_for(Amg &A, int J) {
  if (dense_mode(A)) {
    auto &p = A.sys_dense[J];
    if (!p) p = build_system(h, A, false, J);
    return *p;
  }
  const bool fine = (J == A.L - 1);
  if (fine) {
    if (h->cfg.condense) {
      if (!A.sys_cond) A.sys_cond = build_system(h, A, true, A.L - 1);
      return *A.sys_cond;
    }
    if (!A.sys_hook) A.sys_hook = build_system(h, A, false, A.L - 1);
    return *A.sys_hook;
  }
  // coarse Newton levels (the recovery path of mgb_step): assembled directly at level L-2, Galerkin below
  if (!A.sys_coarse) A.sys_coarse = build_system(h, A, false, A.L - 2);
  return *A.sys_coarse;
}

// Which Euclidean-power pieces can be condensed analytically (node_barrier.cuh piece_eval): identity A, not under the phase-I
// wrapper, the piece's slack row belongs to a node-locally eliminated variable that has no other D row and that no other piece
// (nor another input of this piece) touches, and none of its q rows is eliminated.  Then H_EE is diagonal in that variable and its
// Schur complement is the piece's own.
void Engine::schur_masks(const Amg &A, const System &S, unsigned &pieces, unsigned &elim) const {
  pieces = elim = 0u;
  if (!h->cfg.analytic_schur || S.nE == 0 || A.cd.feas) return;
  const ConvexDev &cd = A.cd;
  for (int k = 0; k < cd.npieces && k < 32; ++k) {
    const PieceDev &pc = cd.pc[k];
    if (pc.kind != MGBX_PIECE_EP || pc.A != nullptr || pc.nc < 2 || pc.ni != pc.nc) continue;
    const int nq = pc.nc - 1, js = pc.idx[nq];
    if (js < 0 || js >= A.nD) continue;
    const int ev = S.Erow[js];
    if (ev < 0) continue;
    bool ok = true;
    for (int r = 0; r < nq; ++r) ok = ok && pc.idx[r] != js && S.Erow[pc.idx[r]] < 0;
    for (int j = 0; j < A.nD; ++j) ok = ok && (j == js || S.Erow[j] != ev);          // the variable's only row
    for (int k2 = 0; k2 < cd.npieces; ++k2)
      if (k2 != k)
        for (int c = 0; c < cd.pc[k2].ni; ++c) ok = ok && cd.pc[k2].idx[c] != js;     // no other piece reads it
    if (ok) {
      pieces |= 1u << k;
      elim |= 1u << ev;
    }
  }
}

// Evaluate the node Hessians at zbase + R_J x and fill the system matrices from the top level down to
// level index ktop (= L-1-J), then the preconditioner hierarchy below it.
void Engine::assemble(Amg &A, System &S, int J, double t, const double *zbase, const double *x) {
  cudaEvent_t st = stage_begin();
  prolong_to_fine(A, J, x, zbase, A.zf);
  NodeParams P = node_params(A, t);
  P.nK = S.nK;
  P.nE = S.nE;
  for (int j = 0; j < MGBX_MAX_ND; ++j) {
    P.Krow[j] = S.Krow[j];
    P.Erow[j] = S.Erow[j];
  }
  P.Hn = A.Hn;
  P.hEEinv = A.hEEinv;
  P.hKE = A.hKE;
  schur_masks(A, S, P.schur_pieces, P.schur_elim);
  if (S.dense) {
    assemble_dense(A, S, P);
    stage_end(STAGE_F2, st);
    if (h->res) h->res->f2_evals++;
    return;
  }
  ElemFused Q;
  PlapParams PQ;
  size_t smem = 0;
  unsigned int grid = 0;
  const int pdim = plap_dim(A);
  // the specialised kernel needs exactly: s eliminated node-locally, u kept with all of its rows
  const bool plap_ok = pdim && S.nE == 1 && S.kept.size() == 1 && S.kept[0] == A.D_var[0] && S.elim[0] == A.D_var[pdim + 1] &&
                       S.nK == pdim + 1 && S.pl.npairs == 1 && plap_setup(A, pdim, t, true, PQ, smem, grid);
  // ... or nothing eliminated and the four pairs (u,u), (u,s), (s,u), (s,s) in this order (coarse-level systems)
  const bool plap_unc = !plap_ok && pdim && S.nE == 0 && S.kept.size() == 2 && S.nK == pdim + 2 && S.pl.npairs == 4 &&
                        S.pl.va[0] == A.D_var[0] && S.pl.vb[0] == A.D_var[0] && S.pl.va[1] == A.D_var[0] && S.pl.vb[1] == A.D_var[pdim + 1] &&
                        S.pl.va[2] == A.D_var[pdim + 1] && S.pl.vb[2] == A.D_var[0] && S.pl.va[3] == A.D_var[pdim + 1] &&
                        S.pl.vb[3] == A.D_var[pdim + 1] && plap_setup(A, pdim, t, true, PQ, smem, grid, false);
  if (plap_ok || plap_unc) {
    PQ.hEEinv = A.hEEinv;
    PQ.hKE = A.hKE;
    PQ.Hblk = S.Hblk;
    LAUNCH(KC_ELEM_F2, launch_plap<NODE_F2>(pdim, plap_ok, PQ, grid, smem, s));
  } else if (elem_fused_setup(A, P, std::max(A.nD, S.nK * (S.nK + 1) / 2), Q, smem, grid)) {
    Q.pl = S.pl;
    Q.Hblk = S.Hblk;
    LAUNCH(KC_ELEMG_F2, launch_elem<NODE_F2>(Q, grid, smem, s));
  } else {
    LAUNCH(KC_NODE_F2, launch_node<NODE_F2>(P, red_grid(A.n), s));
    ElemParams E = elem_params(A);
    E.nK = S.nK;
    for (int j = 0; j < S.nK; ++j) E.Krow[j] = S.Krow[j];
    LAUNCH(KC_BLOCKHESS, k_blockhess<<<nblk(S.hblk_size), 256, 0, s>>>(E, S.pl, A.Hn, S.Hblk));
  }
  SysLevel &top = S.lev[0];
  LAUNCH(KC_GATHER, k_sell_gather<<<nblk(top.A.nnz), 256, 0, s>>>(S.top, S.Hblk, top.A.val));
  if (dist()) allreduce(top.A.val, top.A.nnz);   // sum of the ranks' element contributions (identical pattern on every rank)
  const int ktop = S.ltop - J;
  setup_hierarchy(A, S, ktop);
  stage_end(STAGE_F2, st);
  if (h->res) h->res->f2_evals++;
}


void Engine::dgemm_nt(int M, int N, int K, const double *Am, int64_t lda, const double *Bm, int64_t ldb, const double *sc, double *C, int64_t ldc,
                      bool acc, double alpha) {
  if (M <= 0 || N <= 0) return;
  dim3 grid((N + kGemmBN - 1) / kGemmBN, (M + kGemmBM - 1) / kGemmBM);
  LAUNCH(KC_DGEMM, k_dgemm_nt<<<grid, 128, 0, s>>>(M, N, K, Am, lda, Bm, ldb, sc, C, ldc, acc ? 1 : 0, alpha));
  h->dgemm_flops += 2.0 * M * (double)N * K;
}

// Dense (spectral) assembly: per pair of state variables  Hd = sum_jk D_j' diag(h_jk) D_k  (n x n),  then
// A_top[a-block, b-block] = R_a' Hd R_b  by two GEMMs, written straight into the full row-major top matrix.
void Engine::assemble_dense(Amg &A, System &S, const NodeParams &P) {
  LAUNCH(KC_NODE_F2, launch_node<NODE_F2>(P, red_grid(A.n), s));
  SysLevel &top = S.lev[0];
  const int64_t m = top.m;
  const int n = (int)A.n, nK = S.nK;
  zero(top.A.val, m * m);
  if (S.kron) {
    // sum-factorised: per block of kept variables one small contraction over the fast index (k_kron_w), ONE DMMA GEMM over
    // (operator pair, slow index) against the constant factor table, and the index permutation into the system matrix
    const int n1 = A.kron_n1;
    for (const System::KronPair &kp : S.kp) {
      KronWArgs W;
      memset(&W, 0, sizeof(W));
      W.n1 = n1;
      W.c2a = kp.c2a;
      W.c2b = kp.c2b;
      W.ncombo = kp.ncombo;
      W.K = kp.ncombo * n1;
      for (int c = 0; c < kp.ncombo; ++c) {
        W.c[c].Qj = kp.Qj[c];
        W.c[c].Qk = kp.Qk[c];
        W.c[c].h = A.Hn + (int64_t)kp.hidx[c] * A.n;
      }
      const size_t smem = sizeof(double) * ((size_t)n1 + (size_t)n1 * kp.c2a + (size_t)n1 * kp.c2b);
      LAUNCH(KC_DENSE, k_kron_w<<<kp.ncombo * n1, 256, smem, s>>>(W, S.Wcat));
      const int Mr = kp.c1a * kp.c1b, Nc = kp.c2a * kp.c2b;
      dgemm_nt(Mr, Nc, W.K, kp.AA, W.K, S.Wcat, W.K, nullptr, S.Hd, Nc, false);
      LAUNCH(KC_DENSE, k_kron_scatter<<<nblk((int64_t)Mr * Nc), 256, 0, s>>>(kp.c1a, kp.c2a, kp.c1b, kp.c2b, S.Hd, top.A.val, m, kp.offa, kp.offb));
    }
    setup_hierarchy(A, S, 0);
    return;
  }
  for (size_t qa = 0; qa < S.kept.size(); ++qa)
    for (size_t qb = 0; qb < S.kept.size(); ++qb) {
      const int va = S.kept[qa], vb = S.kept[qb];
      bool any = false;
      zero(S.Hd, (int64_t)n * n);
      for (int ja = 0; ja < nK; ++ja) {
        const int j = S.Krow[ja];
        if (A.D_var[j] != va) continue;
        for (int kb = 0; kb < nK; ++kb) {
          const int k = S.Krow[kb];
          if (A.D_var[k] != vb) continue;
          any = true;
          const int a = std::min(ja, kb), b = std::max(ja, kb);
          const double *hv = A.Hn + (int64_t)(a * nK - (a * (a - 1)) / 2 + (b - a)) * A.n;
          const int oj = A.D_op[j], ok = A.D_op[k];
          if (oj < 0 && ok < 0) LAUNCH(KC_DENSE, k_dense_hess_ident<<<nblk(n), 256, 0, s>>>(n, 0, hv, nullptr, S.Hd));
          else if (oj < 0) LAUNCH(KC_DENSE, k_dense_hess_ident<<<nblk((int64_t)n * n), 256, 0, s>>>(n, 1, hv, A.ops[ok], S.Hd));
          else if (ok < 0) LAUNCH(KC_DENSE, k_dense_hess_ident<<<nblk((int64_t)n * n), 256, 0, s>>>(n, 2, hv, A.ops[oj], S.Hd));
          else dgemm_nt(n, n, n, A.ops[oj], n, A.ops[ok], n, hv, S.Hd, n, true);
        }
      }
      if (!any) continue;
      const int ma = (int)(top.off[qa + 1] - top.off[qa]), mb = (int)(top.off[qb + 1] - top.off[qb]);
      dgemm_nt(mb, n, n, S.Rt[qb], n, S.Hd, n, nullptr, S.Wt, n, false);                                   // Wt = (Hd R_b)'
      dgemm_nt(ma, mb, n, S.Rt[qa], n, S.Wt, n, nullptr, top.A.val + top.off[qa] * m + top.off[qb], m, false);   // R_a' Hd R_b
    }
  setup_hierarchy(A, S, 0);
}

void Engine::setup_hierarchy(Amg &A, System &S, int ktop) {
  const int nlev = (int)S.lev.size();
  SysLevel &Ltop = S.lev[ktop];
  const bool direct = use_direct(S, Ltop);
  int kend = ktop;
  if (!direct) kend = (S.cut >= 0) ? std::max(S.cut, ktop) : nlev - 1;
  for (int k = 0; k < kend; ++k) {
    SysLevel &Lv = S.lev[k];
    SysLevel &Lc = S.lev[k + 1];
    if (!Lv.T_identity) {   // an identity transfer aliases the same matrix
      LAUNCH(KC_SPGEMM, k_sell_gather<<<nblk(Lv.AT.nnz), 256, 0, s>>>(Lv.s1, Lv.A.val, Lv.AT.val));
      LAUNCH(KC_SPGEMM, k_sell_gather<<<nblk(Lc.A.nnz), 256, 0, s>>>(Lv.s2, Lv.AT.val, Lc.A.val));
    }
  }
  if (direct) {
    if (Ltop.m > kCoarseMaxDense) dense_factor(S, Ltop, false);   // tiny systems are factorised inside k_dense_solve_small
    return;
  }
  for (int k = ktop; k <= kend; ++k) {
    SysLevel &Lv = S.lev[k];
    CK(cudaMemsetAsync(Lv.lam, 0, sizeof(double), s));
    LAUNCH(KC_VEC, k_l1diag<<<nblk(Lv.m), 256, 0, s>>>(Lv.A, Lv.dinv, Lv.diag, (unsigned long long *)Lv.lam));
    if (precond_fp32(S)) {
      if (!Lv.val32) Lv.val32 = h->pool.alloc<float>(Lv.A.nnz);
      LAUNCH(KC_VEC, k_f64_to_f32<<<nblk(Lv.A.nnz), 256, 0, s>>>(Lv.A.nnz, Lv.A.val, Lv.val32));
    }
  }
  if (S.cut >= 0 && S.cut >= ktop) {
    SysLevel &Lc = S.lev[S.cut];
    const int m = (int)Lc.m;
    if (!Lc.dense_inv) Lc.dense_inv = h->pool.alloc<double>((size_t)m * m);
    LAUNCH(KC_DENSE, k_coarse_inverse<<<1, 1024, coarse_inverse_smem(m), s>>>(Lc.A, Lc.dense_inv));
  }
  sell_prepare(S, ktop);
  if (lambda_power_its(S) > 0) {   // all levels' power iterations in one cooperative launch
    System::Pcg2Dev &D = pcg2_plan(S, ktop);
    if ((int64_t)D.host.nlev * h->pcg2_grid > 3 * (int64_t)kPcg2MaxGrid) throw std::runtime_error("internal: too many levels for the power-iteration kernel");
    LAUNCH(KC_VEC, CK(pcg2_lambda_power(D.dev, h->pcg2_grid, lambda_power_its(S), 1.2, s)));
  }
}

void Engine::dense_factor(System &S, SysLevel &Lv, bool want_inverse) {
  (void)S;
  (void)want_inverse;
  const int m = (int)Lv.m;
  if (m == 0) return;
  const int npan = (m + kCholNB - 1) / kCholNB;
  if (!Lv.dense) {
    Lv.dense = h->pool.alloc<double>((size_t)m * m);
    Lv.dscale = h->pool.alloc<double>(m);
    Lv.dense_inv = h->pool.alloc<double>((size_t)npan * kCholNB * kCholNB);   // inverses of the diagonal blocks
  }
  zero(Lv.dense, (int64_t)m * m);
  LAUNCH(KC_DENSE, k_dense_scale_diag<<<nblk(m), 256, 0, s>>>(Lv.A, Lv.dscale));
  LAUNCH(KC_DENSE, k_csr_to_dense<<<nblk(m), 256, 0, s>>>(Lv.A, Lv.dscale, Lv.dense));
  // blocked right-looking Cholesky, panel width 64: diagonal block in shared memory, panel and trailing update as DMMA GEMMs
  for (int p = 0; p < npan; ++p) {
    const int k0 = p * kCholNB, nb = std::min(kCholNB, m - k0), rem = m - k0 - nb;
    double *Li = Lv.dense_inv + (size_t)p * kCholNB * kCholNB;
    LAUNCH(KC_DENSE, k_chol_diag_inv<<<1, 1024, kCholDiagSmem, s>>>(Lv.dense, m, k0, Li));
    if (rem > 0) {
      double *A21 = Lv.dense + (size_t)(k0 + nb) * m + k0;
      dgemm_nt(rem, nb, nb, A21, m, Li, kCholNB, nullptr, A21, m, false);                                   // L21 = A21 inv(L11)' (in place: one tile column)
      dgemm_nt(rem, rem, nb, A21, m, A21, m, nullptr, Lv.dense + (size_t)(k0 + nb) * m + k0 + nb, m, true, -1.0);   // A22 -= L21 L21'
    }
  }
}

// x = A^{-1} b through the scaled Cholesky factor (one right-hand side), uses Lv.r as scratch
void Engine::dense_apply(SysLevel &Lv, const double *b, double *x) {
  const int m = (int)Lv.m;
  LAUNCH(KC_DENSE, k_chol_solve_blocked<<<1, 1024, sizeof(double) * m, s>>>(Lv.dense, m, Lv.dense_inv, Lv.dscale, b, x));
}

// sliced-ELL copy of a device CSR pattern (32 rows per slice, slices-per-CTA for the grid the kernel is launched with)
SellBuild Engine::make_sell(const DevCsr &A, int64_t nthreads) {
  SellBuild B;
  h->pool.cat = "solve kernel: sliced-ELL level matrices";
  if (A.rows >= INT32_MAX / 2) throw std::runtime_error("persistent solve kernel: a level matrix exceeds 32-bit indexing");
  // lanes per row: widen while the level leaves at least half of the threads that share its phases idle and the rows
  // still give every lane two entries (measured, tools/micro/bench_spmv_phase: one lane per row wins on the two finest
  // levels of C2, four lanes on the 32 k-row level)
  int lpr = 1;
  const double avg = A.rows ? (double)A.nnz / (double)A.rows : 0.0;
  // up to a whole warp per row: the near-dense coarse Galerkin levels of 3-D hierarchies (fem3d 64^3: 544 rows of ~500 entries)
  // otherwise leave 8 lanes walking 60+ dependent rounds each -- 141 us per PCG iteration on a 544-row level
  // (profiles/r02h_pcg2_phase_profile_fem3d_64cubed.txt)
  while (lpr < 32 && A.rows * (int64_t)lpr * 2 <= nthreads && avg / lpr >= 2.0) lpr *= 2;
  const int rps = 32 / lpr;
  const int nsl = (int)((A.rows + rps - 1) / rps);
  B.M.rows = (int)A.rows;
  B.M.lpr = lpr;
  B.M.nslices = nsl;
  B.M.spc = pcg2_slices_per_cta(nsl, std::max(1, h->pcg2_grid));
  if (nsl == 0) return B;
  int *width = tmp_alloc<int>(nsl, s);
  CK(sell_slice_widths(A.rows, lpr, A.ptr, width, s));
  std::vector<int> hw(nsl);
  CK(cudaMemcpyAsync(hw.data(), width, sizeof(int) * nsl, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  tmp_free(width, s);
  std::vector<int> soff(nsl + 1, 0);
  int64_t tot = 0;
  for (int q = 0; q < nsl; ++q) {
    tot += 32 * (int64_t)hw[q];
    if (tot > INT32_MAX) throw std::runtime_error("persistent solve kernel: sliced-ELL level matrix exceeds 32-bit indexing");
    soff[q + 1] = (int)tot;
  }
  B.M.entries = (int)tot;
  B.soff = h->pool.upload<int>(soff.data(), soff.size(), s);
  B.idx = h->pool.alloc<int>((size_t)tot);
  B.src = h->pool.alloc<int>((size_t)tot);
  B.val = h->pool.alloc<double>((size_t)tot);
  B.valf = h->pool.alloc<float>((size_t)tot);
  CK(sell_fill_pattern(A.rows, lpr, A.ptr, A.idx, B.soff, B.idx, B.src, s));
  h->launches += 2;
  B.M.soff = B.soff;
  B.M.idx = B.idx;
  B.M.val = B.val;
  B.M.valf = nullptr;
  CK(cudaStreamSynchronize(s));   // soff (host vector) has been consumed
  return B;
}

// Build (once) the sliced-ELL structures of the active levels below lev[ktop] and refresh the values of the level matrices.
// Called from setup_hierarchy after every assembly, i.e. before every solve.
void Engine::sell_prepare(System &S, int ktop) {
  const std::vector<int> act = active_levels(S, ktop);
  const int64_t grid_threads = (int64_t)h->pcg2_grid * kPcg2Threads;
  for (size_t q = 0; q < act.size(); ++q) {
    SysLevel &Lv = S.lev[act[q]];
    // threads that share this level's phases: the whole grid, or CTA 0 alone for the tail (q > 0 and small)
    const int64_t nthr = (q > 0 && Lv.m <= h->cfg.tail_max) ? kPcg2Threads : grid_threads;
    if (!Lv.sell_A) {
      Lv.sA = make_sell(Lv.A, nthr);
      Lv.sell_A = true;
    }
    if (Lv.sA.M.entries) LAUNCH(KC_VEC, CK(sell_fill_values(Lv.sA.M.entries, Lv.sA.src, Lv.A.val, Lv.sA.val, Lv.sA.valf, s)));
    if (q + 1 < act.size() && !Lv.sell_T) {
      const int64_t nthr_c = (S.lev[act[q + 1]].m <= h->cfg.tail_max) ? kPcg2Threads : grid_threads;
      Lv.sT = make_sell(Lv.T, nthr);
      Lv.sTt = make_sell(Lv.Tt, nthr_c);
      if (Lv.sT.M.entries) LAUNCH(KC_VEC, CK(sell_fill_values(Lv.sT.M.entries, Lv.sT.src, Lv.T.val, Lv.sT.val, Lv.sT.valf, s)));
      if (Lv.sTt.M.entries) LAUNCH(KC_VEC, CK(sell_fill_values(Lv.sTt.M.entries, Lv.sTt.src, Lv.Tt.val, Lv.sTt.val, Lv.sTt.valf, s)));
      Lv.sell_T = true;
    }
  }
}

System::Pcg2Dev &Engine::pcg2_plan(System &S, int ktop) {
  auto it = S.pplans2.find(ktop);
  if (it != S.pplans2.end()) return it->second;
  System::Pcg2Dev &D = S.pplans2[ktop];
  Pcg2Plan &P = D.host;
  P = Pcg2Plan();
  const std::vector<int> act = active_levels(S, ktop);
  if ((int)act.size() > kPcg2MaxLevels) throw std::runtime_error("persistent solve kernel: too many levels");
  P.nlev = (int)act.size();
  P.bottom_dense = (S.cut >= 0 && act.back() == S.cut) ? 1 : 0;
  P.nu = std::max(1, h->cfg.smoother_sweeps);
  P.nu_bottom = 30;
  P.smoother = h->cfg.smoother;
  P.cheb_ratio = h->cfg.cheb_ratio > 1.0 ? h->cfg.cheb_ratio : 8.0;
  const bool f32 = precond_fp32(S);
  for (int q = 0; q < P.nlev; ++q) {
    SysLevel &Lv = S.lev[act[q]];
    Pcg2Level &pl = P.lev[q];
    if (Lv.m > INT32_MAX / 2) throw std::runtime_error("persistent solve kernel: level exceeds 32-bit indexing");
    pl.m = (int)Lv.m;
    pl.A = Lv.sA.M;
    pl.A.valf = Lv.sA.valf;       // narrowed below for the grid-wide levels
    if (q + 1 < P.nlev) {
      pl.T = Lv.sT.M;
      pl.T.valf = Lv.sT.valf;
      pl.Tt = Lv.sTt.M;
      pl.Tt.valf = Lv.sTt.valf;
    }
    pl.idiag = Lv.diag;
    pl.dinv = Lv.dinv;
    pl.lam = Lv.lam;
    pl.b = Lv.b;
    pl.x = Lv.x;
    pl.x2 = Lv.x2;
    pl.r = Lv.r;
    if (!Lv.pw) {   // power-iteration vector (warm-started across Newton iterations)
      Lv.pw = h->pool.alloc<double>(Lv.m);
      LAUNCH(KC_VEC, k_pw_init<<<nblk(Lv.m), 256, 0, s>>>(Lv.m, Lv.pw));
    }
    pl.pw = Lv.pw;
  }
  // the tail [nbig, nlev): levels with <= tail_max unknowns, as many as fit into CTA 0's shared memory
  int dev = 0;
  CK(cudaGetDevice(&dev));
  const size_t cap = pcg2_max_tail_bytes(dev);
  P.nbig = 0;
  for (int q = 0; q < P.nlev; ++q)
    if (S.lev[act[q]].m > h->cfg.tail_max) P.nbig = q + 1;
  P.nbig = std::max(P.nbig, 1);
  while (P.nbig < P.nlev && (pcg2_tail_bytes(P) > cap || P.nlev - P.nbig > 12)) P.nbig++;
  D.smem = (P.nbig < P.nlev) ? pcg2_tail_bytes(P) : 0;
  P.tail_smem_bytes = (int)D.smem;
  for (int q = 0; q < P.nbig; ++q) {   // grid-wide levels read FP32 values only when the FP32 preconditioner is on
    if (!f32) P.lev[q].A.valf = P.lev[q].T.valf = P.lev[q].Tt.valf = nullptr;
  }
  P.dense_inv = P.bottom_dense ? S.lev[S.cut].dense_inv : nullptr;
  P.r = S.pc_r;
  P.p = S.pc_p;
  P.p2 = S.pc_p2;
  P.Ap = S.pc_Ap;
  P.x = S.pc_x;
  P.b = S.pc_b;
  P.partials = S.pcg_partials;
  P.bar = S.pcg_bar;
  P.out = S.pcg_out;
  if (getenv("MGBX_PCG_PROF")) P.prof = h->pool.zeros<unsigned long long>(1 + 2 * (size_t)kPcg2ProfCap, s);
  if (dist() && h->cfg.shard_solve && P.nlev >= 2) {
    // multi-GPU: the leading levels with at least shard_min_rows unknowns are row-sharded over the ranks (pcg2.hpp)
    // A cross-GPU barrier costs several microseconds more than the local grid barrier, so a level is sharded only when a phase
    // over it is long enough to pay for that: T (1 - 1/N) > B with T ~ 12 B nnz / 3 TB/s and B ~ 10 us (measured on 2 GPUs:
    // profiles/r02f_*), i.e. nnz (1 - 1/N) >= shard_min_nnz (default 4 M).  C2's 2-D levels (1.8 M non-zeros) stay replicated.
    int nshard = 0;
    const std::vector<int> act = active_levels(S, ktop);
    for (int q = 0; q < P.nbig && q < P.nlev - 1; ++q) {
      const double nnzq = (double)S.lev[act[q]].A.nnz * (1.0 - 1.0 / (double)h->nranks);
      if (P.lev[q].m < h->cfg.shard_min_rows || nnzq < (double)h->cfg.shard_min_nnz) break;
      nshard = q + 1;
    }
    if (nshard > 0) pcg2_setup_dist(D, nshard);
  }
  D.dev = h->pool.upload<Pcg2Plan>(&P, 1, s);
  CK(cudaStreamSynchronize(s));
  if (h->cfg.verbose > 0)
    fprintf(stderr, "[mgbx] persistent PCG plan: %d levels (%d grid-wide, %d in CTA 0 from %zu bytes of shared memory), dense bottom %d, grid %d x %d\n",
            P.nlev, P.nbig, P.nlev - P.nbig, D.smem, P.bottom_dense, h->pcg2_grid, kPcg2Threads);
  return D;
}

// Exchange arena of one sharded solve plan: every vector a peer writes into (the work vectors of the sharded levels, p, x, the
// partial-sum slots, the barrier flags) is carved out of ONE cudaMalloc block with the same layout on every rank; the blocks
// are exported with CUDA IPC, the handles all-gathered with NCCL, and each rank maps its peers' blocks.
void Engine::pcg2_setup_dist(System::Pcg2Dev &D, int nshard) {
  Pcg2Plan &P = D.host;
  const int nr = h->nranks;
  if (nr > kPcg2MaxRanks) throw std::runtime_error("row-sharded solve: more than 8 ranks");
  if ((int64_t)nr * h->pcg2_grid > kPcg2MaxGrid) throw std::runtime_error("row-sharded solve: too many CTAs for the partial-sum slots");
  size_t bytes = 0;
  auto take = [&](size_t n) {
    const size_t off = bytes;
    bytes += (n + 255) & ~(size_t)255;
    return off;
  };
  const size_t o_flags = take(sizeof(unsigned long long) * kPcg2MaxRanks), o_arr = take(sizeof(unsigned int)), o_rel = take(sizeof(unsigned long long));
  const size_t o_part = take(sizeof(double) * 3 * (size_t)kPcg2MaxGrid);
  const size_t m0 = (size_t)P.lev[0].m;
  const size_t o_p = take(8 * m0), o_p2 = take(8 * m0), o_x = take(8 * m0);
  std::vector<size_t> o_lev(4 * (size_t)nshard);
  for (int q = 0; q < nshard; ++q)
    for (int v = 0; v < 4; ++v) o_lev[4 * q + v] = take(8 * (size_t)P.lev[q].m);
  CK(cudaMalloc((void **)&D.arena, bytes));
  D.arena_bytes = bytes;
  CK(cudaMemsetAsync(D.arena, 0, bytes, s));
  // export / all-gather / import
  cudaIpcMemHandle_t mine;
  CK(cudaIpcGetMemHandle(&mine, D.arena));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  char *dsend = tmp_alloc<char>(64, s), *dall = tmp_alloc<char>(64 * (size_t)nr, s);
  CK(cudaMemcpyAsync(dsend, &mine, 64, cudaMemcpyHostToDevice, s));
  NCK(nccl_api().AllGather(dsend, dall, 8, kNcclInt64, h->comm, s));
  std::vector<cudaIpcMemHandle_t> all(nr);
  CK(cudaMemcpyAsync(all.data(), dall, 64 * (size_t)nr, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  tmp_free(dsend, s);
  tmp_free(dall, s);
  P.dist = Pcg2Dist();
  P.dist.nranks = nr;
  P.dist.rank = h->rank;
  P.dist.nshard = nshard;
  for (int q = 0; q < nr; ++q) {
    if (q == h->rank) {
      P.dist.peer_off[q] = 0;
      continue;
    }
    CK(cudaIpcOpenMemHandle(&D.peer[q], all[q], cudaIpcMemLazyEnablePeerAccess));
    P.dist.peer_off[q] = (long long)((char *)D.peer[q] - D.arena);
  }
  P.dist.flags = (unsigned long long *)(D.arena + o_flags);
  P.dist.xarrive = (unsigned int *)(D.arena + o_arr);
  P.dist.xrelease = (unsigned long long *)(D.arena + o_rel);
  P.partials = (double *)(D.arena + o_part);
  P.p = (double *)(D.arena + o_p);
  P.p2 = (double *)(D.arena + o_p2);
  P.x = (double *)(D.arena + o_x);
  const int64_t gcta = (int64_t)nr * h->pcg2_grid;
  auto respc = [&](SellMat &M) { M.spc = pcg2_slices_per_cta(M.nslices, gcta); };
  for (int q = 0; q < nshard; ++q) {
    Pcg2Level &pl = P.lev[q];
    pl.x = (double *)(D.arena + o_lev[4 * q + 0]);
    pl.x2 = (double *)(D.arena + o_lev[4 * q + 1]);
    pl.r = (double *)(D.arena + o_lev[4 * q + 2]);
    pl.b = (double *)(D.arena + o_lev[4 * q + 3]);
    respc(pl.A);              // rows of level q: owned by the CTAs of all ranks together
    respc(pl.T);
    if (q > 0) respc(P.lev[q - 1].Tt);
  }
  if (h->cfg.verbose > 0)
    fprintf(stderr, "[mgbx] rank %d: row-sharded solve over %d ranks, %d of %d levels sharded, exchange arena %.1f MB\n", h->rank, nr, nshard, P.nlev, bytes / 1e6);
}

// Preconditioned CG on lev[ktop], the whole solve in one cooperative launch of k_pcg2; returns the iteration count
// (negative: breakdown)
int Engine::pcg(System &S, int ktop, const double *b, double *x) {
  SysLevel &Lv = S.lev[ktop];
  const int64_t m = Lv.m;
  System::Pcg2Dev &D = pcg2_plan(S, ktop);
  if (b != S.pc_b) copy(S.pc_b, b, m);
  pre_launch(KC_PCG);
  CK(pcg2_launch(D.dev, h->pcg2_grid, D.smem, h->cur_rtol2, h->cfg.pcg_maxit, h->cur_window, D.host.dist.nshard > 0, s));
  post_launch(KC_PCG);
  if (D.host.prof) {   // debugging aid: accumulate the per-phase durations of this launch
    h->prof_host.resize(1 + 2 * (size_t)kPcg2ProfCap);
    CK(cudaMemcpyAsync(h->prof_host.data(), D.host.prof, sizeof(unsigned long long) * h->prof_host.size(), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (h->prof_ns.empty()) {
      h->prof_ns.assign(kPcg2MaxLevels * 16, 0.0);
      h->prof_cnt.assign(kPcg2MaxLevels * 16, 0);
    }
    const size_t nrec = (size_t)h->prof_host[0];
    for (size_t q = 1; q < nrec; ++q) {
      const int tag = (int)h->prof_host[1 + 2 * q];
      if (tag < 0 || tag >= kPcg2MaxLevels * 16) continue;
      h->prof_ns[tag] += (double)(h->prof_host[2 + 2 * q] - h->prof_host[2 + 2 * (q - 1)]);
      h->prof_cnt[tag]++;
    }
  }
  CK(cudaMemcpyAsync(h->hscal + 8, S.pcg_out, sizeof(double) * 6, cudaMemcpyDeviceToHost, s));
  sync();
  const int it = (int)h->hscal[8];
  const double status = h->hscal[10];
  h->last_solve_status = (int)status;
  h->last_solve_rel = (h->hscal[11] > 0.0) ? std::sqrt(h->hscal[9] / h->hscal[11]) : 0.0;
  h->last_solve_erel = (h->hscal[12] > 0.0) ? h->hscal[13] / h->hscal[12] : 0.0;
  if (status == -3.0) throw std::runtime_error("row-sharded solve: a peer rank never arrived at a cross-GPU barrier (ranks out of step?)");
  if (x != D.host.x) copy(x, D.host.x, m);
  return status < 0 ? -std::max(it, 1) : it;
}

int Engine::solve_compact(System &S, int ktop, const double *b, double *x) {
  SysLevel &Lv = S.lev[ktop];
  if (use_direct(S, Lv)) {
    h->last_solve_status = 1;
    h->last_solve_rel = 0.0;
    h->last_solve_erel = 0.0;
    const bool small = Lv.m <= kCoarseMaxDense;
    auto apply = [&](const double *rhs, double *out) {
      if (small) LAUNCH(KC_DENSE, k_dense_solve_small<<<1, 1024, dense_solve_small_smem((int)Lv.m), s>>>(Lv.A, rhs, out, nullptr));
      else dense_apply(Lv, rhs, out);
    };
    apply(b, x);
    // one step of iterative refinement against the CSR operator
    spmv(Lv.A, x, b, -1.0, Lv.r, Lv.spmv_group);
    apply(Lv.r, Lv.x2);
    LAUNCH(KC_VEC, k_axpby<<<nblk(Lv.m), 256, 0, s>>>(Lv.m, 1.0, x, 1.0, Lv.x2, x));
    return 0;
  }
  // Loud, not slow: an un-condensable slack above the dense fallback size would grind through thousands of failing PCG solves
  // (kappa -> sqrt(kappa) ~50 times per barrier step) before mgb_core gives up.  The reference's direct solve has no such
  // regime; refuse it up front unless the caller opts in (cfg.uncondensed_pcg).
  if (S.uncondensed_slack && !h->cfg.uncondensed_pcg && Lv.m > kDenseMaxUnknowns)
    throw UnsupportedError("Newton system with a slack variable that cannot be eliminated node-locally (e.g. a slack in :broken_P1) and " +
                           std::to_string((long long)Lv.m) + " unknowns: above the dense direct solver's size (8192) only the V-cycle PCG is available, "
                           "which is not reliable for these systems (set cfg.uncondensed_pcg = 1 to try anyway)");
  const int it = pcg(S, ktop, b, x);
  // PCG first, direct second: a solve that broke down or stayed inexact is redone by the dense Cholesky when the system is
  // small enough to hold as a dense matrix (the un-condensable families, the last steps of a parabolic ramp)
  const bool bad = h->last_solve_status < 0 || (h->last_solve_rel > h->cfg.pcg_fail_rtol && h->last_solve_erel > h->cfg.pcg_fail_etol);
  if (bad && h->cfg.direct_fallback && Lv.m <= kDenseMaxUnknowns) {
    if (h->cfg.verbose > 0)
      fprintf(stderr, "[mgbx] PCG on %lld unknowns ended with status %d, |r|/|b| = %.3g: falling back to the dense direct solve\n", (long long)Lv.m,
              h->last_solve_status, h->last_solve_rel);
    const bool small = Lv.m <= kCoarseMaxDense;
    if (!small) dense_factor(S, Lv, false);
    auto apply = [&](const double *rhs, double *out) {
      if (small) LAUNCH(KC_DENSE, k_dense_solve_small<<<1, 1024, dense_solve_small_smem((int)Lv.m), s>>>(Lv.A, rhs, out, nullptr));
      else dense_apply(Lv, rhs, out);
    };
    apply(b, x);
    spmv(Lv.A, x, b, -1.0, Lv.r, Lv.spmv_group);
    apply(Lv.r, Lv.x2);
    LAUNCH(KC_VEC, k_axpby<<<nblk(Lv.m), 256, 0, s>>>(Lv.m, 1.0, x, 1.0, Lv.x2, x));
    h->last_solve_status = 1;
    h->last_solve_rel = 0.0;
    h->last_solve_erel = 0.0;
    if (h->res) h->res->direct_fallbacks++;
  }
  return it;
}

// dir = H_J^{-1} g  (full level-J vectors).  With a condensed system the node-local variables are
// eliminated exactly first and recovered by back-substitution.
int Engine::solve(Amg &A, System &S, int J, const double *g, double *dir) {
  cudaEvent_t st = stage_begin();
  const int ktop = S.ltop - J;
  SysLevel &Lv = S.lev[ktop];
  int iters = 0;
  if (S.nE == 0) {
    iters = solve_compact(S, ktop, g, dir);
  } else {
    // (only at the fine level)  rhs_K = g_K + R_K' sum_j D_j' gt_j
    CondParams C;
    memset(&C, 0, sizeof(C));
    C.n = A.n;
    C.nD = A.nD;
    C.nK = S.nK;
    C.nE = S.nE;
    for (int j = 0; j < S.nK; ++j) C.Krow[j] = S.Krow[j];
    for (int e = 0; e < S.nE; ++e) C.Eoff[e] = A.voff[A.L - 1][S.elim[e]];
    C.hEEinv = A.hEEinv;
    C.hKE = A.hKE;
    LAUNCH(KC_COND, k_condense_rhs<<<nblk(A.n), 256, 0, s>>>(C, g, A.G));
    ElemParams E = elem_params(A);
    E.nK = S.nK;
    for (int j = 0; j < S.nK; ++j) E.Krow[j] = S.Krow[j];
    LAUNCH(KC_BLOCKGRAD, k_blockgrad<<<nblk((int64_t)A.nu * A.n), 256, 0, s>>>(E, A.G, A.gb, A.nu));
    if (!dist()) {
      spmv(A.RLt, A.gb, g, 1.0, A.tmp);               // tmp = g + R' gb   (entries of eliminated variables unused)
    } else {
      spmv(A.RLt, A.gb, nullptr, 1.0, A.tmp);         // this rank's part of R' gb, summed over the ranks, then + g
      allreduce_shared(A, J, A.tmp);
      LAUNCH(KC_VEC, k_axpby<<<nblk(A.m[J]), 256, 0, s>>>(A.m[J], 1.0, A.tmp, 1.0, g, A.tmp));
    }
    for (size_t q = 0; q < S.kept.size(); ++q)
      copy(S.pc_b + Lv.off[q], A.tmp + A.voff[A.L - 1][S.kept[q]], Lv.off[q + 1] - Lv.off[q]);
    iters = solve_compact(S, ktop, S.pc_b, S.pc_x);
    zero(dir, A.m[A.L - 1]);
    for (size_t q = 0; q < S.kept.size(); ++q)
      copy(dir + A.voff[A.L - 1][S.kept[q]], S.pc_x + Lv.off[q], Lv.off[q + 1] - Lv.off[q]);
    // broken image of the kept part, then back-substitution
    spmv(A.RL, dir, nullptr, 1.0, A.gb);
    NodeParams NP = node_params(A, 0.0);
    NP.zf = A.gb;
    LAUNCH(KC_COND, k_backsubst<<<nblk(A.n), 256, 0, s>>>(C, NP, g, dir));
  }
  stage_end(STAGE_SOLVE, st);
  // inc = g . dir, finiteness of dir
  dot2_fetch(A, J, dir, g);
  if (h->res) {
    h->res->linear_solves++;
    h->res->pcg_iters += iters > 0 ? iters : -iters;
  }
  return iters;
}

Engine::NewtonOut Engine::newton(Amg &A, int J, double t, int maxit, int stop_kind, double lambda_tol, double theta,
                                 const mgbx_step_opts &o) {
  NewtonOut out{false, 0, MGBX_OK, 0.0, 0.0, 0.0};
  const int64_t m = A.m[J];
  System &S = system_for(A, J);
  if (dist() && J == A.L - 1)
    for (int v : S.kept)
      if (A.var_local[v]) throw std::runtime_error("multi-GPU: a node-local state variable could not be condensed out of the Newton system");
  // the finalize pass stops on floating-point stagnation (stopping_exact): give it directions converged to the
  // attainable accuracy so that it stagnates where a direct solve would
  const double rt = (stop_kind == 0) ? std::min(h->cfg.pcg_rtol, h->cfg.pcg_rtol_final) : h->cfg.pcg_rtol;
  h->cur_rtol2 = rt * rt;
  h->cur_window = (stop_kind == 0) ? 6 : std::max(1, h->cfg.pcg_stall_window);   // finalize: iterate to the attainable accuracy, detected quickly
  zero(A.x, m);
  EvalOut e0 = eval_f01(A, J, t, A.z, A.x, A.g);
  if (!e0.finite) {
    if (h->cfg.verbose > 0)
      fprintf(stderr, "[mgbx] newton J=%d: starting point outside the domain (y=%g, non-finite nodes=%g, |g|=%g)\n", J, e0.y, e0.nonfinite_nodes, e0.gnorm);
    out.status = MGBX_NON_FINITE;
    out.y = e0.y;
    return out;
  }
  double y = e0.y, gnorm = e0.gnorm;
  double ymin = y, gmin = gnorm, incmin = INFINITY;
  bool converged = false;
  int k = 0;
  const double eps = 2.220446049250313e-16;
  while (k < maxit && !converged) {
    ++k;
    assemble(A, S, J, t, A.z, A.x);
    const int pit = solve(A, S, J, A.g, A.dir);
    const double inc = h->hscal[4];
    const bool dir_finite = (h->hscal[6] == 0.0) && std::isfinite(h->hscal[5]) && std::isfinite(inc);
    out.inc = inc;
    if (h->cfg.verbose > 1)
      fprintf(stderr, "[mgbx] newton J=%d m=%lld k=%d y=%.17g |g|=%.6g lam2=%.6g pcg=%d status=%d rel=%.3g erel=%.3g t=%g\n", J, (long long)m, k, y, gnorm, inc, pit,
              h->last_solve_status, h->last_solve_rel, h->last_solve_erel, t);
    // An iterative solve that broke down or stopped far from the requested residual is a FAILED solve, as a failed
    // factorisation is for the reference's direct `H \\ g` (src/utils.jl:142-145): for a CG iterate g.x_k <= g.H^-1 g, so an
    // under-converged direction under-estimates the Newton decrement and could end the iteration early with a wrong z.
    // The Newton run is reported as not converged; mgb_core then shrinks kappa (or phase I grows the box).
    bool solve_inexact = false;
    if (h->last_solve_status < 0) {   // breakdown (indefinite or non-finite): no direction at all
      if (h->cfg.verbose > 0)
        fprintf(stderr, "[mgbx] newton J=%d m=%lld k=%d: linear solve broke down after %d PCG iterations\n", J, (long long)m, k, pit < 0 ? -pit : pit);
      if (h->res) h->res->solve_failures++;
      break;
    }
    if (h->last_solve_rel > 0.5 && h->last_solve_erel > h->cfg.pcg_fail_etol) {   // no better than the zero vector: a failed solve
      if (h->cfg.verbose > 0)
        fprintf(stderr, "[mgbx] newton J=%d m=%lld k=%d: linear solve failed (status %d, |r|/|b| = %.3g after %d PCG iterations)\n", J, (long long)m, k,
                h->last_solve_status, h->last_solve_rel, pit < 0 ? -pit : pit);
      if (h->res) h->res->solve_failures++;
      break;
    }
    if (h->last_solve_rel > h->cfg.pcg_fail_rtol && h->last_solve_erel > h->cfg.pcg_fail_etol) {
      // under-converged: the direction is still a descent direction and is used (inexact Newton, guarded by the line search),
      // but its decrement is not trusted to end the iteration
      solve_inexact = true;
      if (h->res) h->res->solve_failures++;
      if (h->cfg.verbose > 0)
        fprintf(stderr, "[mgbx] newton J=%d m=%lld k=%d: inexact linear solve (status %d, |r|/|b| = %.3g, energy gained in the last 4 iterations %.3g, after %d PCG iterations)\n",
                J, (long long)m, k, h->last_solve_status, h->last_solve_rel, h->last_solve_erel, pit < 0 ? -pit : pit);
    }
    if (!dir_finite) {
      if (h->cfg.verbose > 0)
        fprintf(stderr, "[mgbx] newton J=%d m=%lld k=%d: non-finite direction (g.d=%g |d|^2=%g non-finite entries=%g, pcg=%d, |r|^2=%g |b|^2=%g)\n", J,
                (long long)m, k, inc, h->hscal[5], h->hscal[6], pit, h->hscal[9], h->hscal[11]);
      out.status = MGBX_NON_FINITE;
      break;
    }
    if (inc <= 0.0) {
      converged = std::fabs(inc) <= eps * std::max(std::fabs(y), 1.0);
      break;
    }
    double sstep = 1.0;
    double yn = y, gnn = gnorm;
    bool have_trial = false;   // xbest/gbest hold the last finite trial
    // exact line search by Illinois root finding on phi(sigma) = F1(x - sigma n).n  (newton.jl:4-27,84-103)
    while (o.line_search == 1 && sstep > 0.0) {
      bool ok = true;
      auto launch_trial = [&](double sigma) {
        if (!dist()) LAUNCH(KC_VEC, k_trial<<<red_grid(m), kRedThreads, 0, s>>>(m, A.x, A.dir, sigma, A.xn, h->partials, h->ticket, h->dscal + 7));
        else LAUNCH(KC_VEC, k_trial_seg<<<red_grid(m), kRedThreads, 0, s>>>(seglist(A, J), m, A.x, A.dir, sigma, A.xn, h->partials, h->ticket, h->dscal + 38));
      };
      auto phi = [&](double sigma) -> double {
        launch_trial(sigma);
        EvalOut e = eval_f01(A, J, t, A.z, A.xn, A.gn);
        if (!std::isfinite(e.y)) {   // "line search: non-finite barrier value"
          ok = false;
          return NAN;
        }
        dot2_fetch(A, J, A.gn, A.dir);
        if (!std::isfinite(h->hscal[4])) ok = false;   // @assert isfinite(fc)
        return h->hscal[4];
      };
      double a = 0.0, b = sstep, fa = inc, fb = phi(b), sstar = b;
      if (ok) {
        if (fa == 0.0) sstar = a;
        else if (fa * fb >= 0.0) sstar = b;
        else {
          bool found = false;
          for (int kk = 0; kk < 10000 && ok; ++kk) {
            const double c = (a * fb - b * fa) / (fb - fa);
            const double fc = phi(c);
            if (!ok) break;
            if (c <= std::min(a, b) || c >= std::max(a, b) || fc * fa == 0.0 || fc * fb == 0.0) {
              sstar = c;
              found = true;
              break;
            }
            if (fb * fc < 0.0) {
              a = b;
              fa = fb;
            } else {
              fa /= 2.0;
            }
            b = c;
            fb = fc;
          }
          if (!found) ok = false;   // trial rejected (or "Illinois solver failed to converge")
        }
      }
      if (ok) {
        launch_trial(sstar);
        EvalOut et = eval_f01(A, J, t, A.z, A.xn, A.gn);
        if (et.finite) {
          std::swap(A.xn, A.xbest);
          std::swap(A.gn, A.gbest);
          have_trial = true;
          yn = et.y;
          gnn = et.gnorm;
          break;
        }
      }
      sstep *= o.ls_beta;
    }
    // backtracking line search (newton.jl:139-154 with the trial loop of :35-50)
    while (o.line_search == 0 && sstep > 0.0) {
      if (!dist()) LAUNCH(KC_VEC, k_trial<<<red_grid(m), kRedThreads, 0, s>>>(m, A.x, A.dir, sstep, A.xn, h->partials, h->ticket, h->dscal + 7));
      else LAUNCH(KC_VEC, k_trial_seg<<<red_grid(m), kRedThreads, 0, s>>>(seglist(A, J), m, A.x, A.dir, sstep, A.xn, h->partials, h->ticket, h->dscal + 38));
      EvalOut et = eval_f01(A, J, t, A.z, A.xn, A.gn);
      const bool stalled = (h->hscal[7] == 0.0);
      if (et.finite) {
        std::swap(A.xn, A.xbest);
        std::swap(A.gn, A.gbest);
        have_trial = true;
        yn = et.y;
        gnn = et.gnorm;
        if (stalled || yn <= y - o.ls_c1 * inc * sstep) break;
      }
      sstep *= o.ls_beta;
    }
    // an under-converged solve under-estimates the decrement (g.x_k <= g.H^-1 g): only the stagnation rule may stop then
    if (stop_test(solve_inexact ? 0 : stop_kind, lambda_tol, theta, ymin, yn, gmin, gnn, std::sqrt(inc))) converged = true;
    if (have_trial) {
      std::swap(A.x, A.xbest);
      std::swap(A.g, A.gbest);
    }
    y = yn;
    gnorm = gnn;
    gmin = std::min(gmin, gnorm);
    ymin = std::min(ymin, y);
    incmin = std::min(inc, incmin);
  }
  out.converged = converged;
  out.k = k;
  out.y = y;
  out.gnorm = gnorm;
  return out;
}

int Engine::step(int which, double t, const mgbx_step_opts &o, mgbx_step_result *r) {
  Amg &A = h->amg[which];
  memset(r, 0, sizeof(*r));
  h->res = r;
  const int L = A.L;
  copy(A.zsave, A.z, (int64_t)A.nu * A.n);
  int status = MGBX_OK;
  // eta(j, J): Newton in range(R_fine[J]) around the current z (levels 1-based as in the reference)
  auto eta = [&](int j, int J, int stop_kind, double ltol, double theta, int mxit) -> bool {
    (void)j;
    if (status != MGBX_OK) return false;
    NewtonOut n = newton(A, J - 1, t, mxit, stop_kind, ltol, theta, o);
    r->its[J - 1] += n.k;
    r->y = n.y;
    r->gnorm = n.gnorm;
    r->inc = n.inc;
    if (n.status != MGBX_OK) {
      status = n.status;
      return false;
    }
    if (n.converged) {
      prolong_to_fine(A, J - 1, A.x, A.z, A.zf);
      std::swap(A.z, A.zf);
    }
    return n.converged;
  };
  std::function<bool(int, int)> dac = [&](int j, int J) -> bool {
    const int mn = (o.initial_step && J - j == 1) ? o.maxit : o.max_newton;
    if (eta(j, J, o.stop_kind, o.stop_lambda_tol, o.stop_theta, mn)) return true;
    const int jmid = (j + J) / 2;
    if (jmid == j || jmid == J) return false;
    return dac(j, jmid) && dac(jmid, J);
  };
  bool converged = dac(0, L);
  copy(A.zunfin, A.z, (int64_t)A.nu * A.n);   // SOL.z_unfinalized (mgb.jl:76-80)
  if (o.finalize && status == MGBX_OK) {
    const int before = r->its[L - 1];
    const bool foo = eta(L - 1, L, 0, 0.0, o.finalize_theta, o.maxit);
    r->its_finalize = r->its[L - 1] - before;   // bookkeeping: the reference adds the finalize pass into its[L]
    converged = converged && foo;
  }
  r->converged = converged ? 1 : 0;
  if (status != MGBX_OK || !converged) copy(A.z, A.zsave, (int64_t)A.nu * A.n);   // the caller discards a failed step (mgb.jl:147-163)
  sync();
  h->res = nullptr;
  if (status != MGBX_OK || !converged) return status != MGBX_OK ? status : MGBX_NOT_CONVERGED;
  return MGBX_OK;
}

int Engine::matched_t(double t_default, double *t_out, double *tstar_out) {
  Amg &A = h->amg[MGBX_MAIN];
  const int J = A.L - 1;
  const int64_t m = A.m[J];
  System &S = system_for(A, J);
  zero(A.x, m);
  EvalOut e0 = eval_f01(A, J, 0.0, A.z, A.x, A.g);        // g = grad of the barrier term
  EvalOut e1 = eval_f01(A, J, 1.0, A.z, A.x, A.gn);       // gn = gphi + gc
  (void)e0;
  (void)e1;
  LAUNCH(KC_VEC, k_axpby<<<nblk(m), 256, 0, s>>>(m, 1.0, A.gn, -1.0, A.g, A.gn));   // gn = gc
  assemble(A, S, J, 1.0, A.z, A.x);
  solve(A, S, J, A.g, A.dir);      // nphi
  solve(A, S, J, A.gn, A.xn);      // nc
  const double d = h->hscal[4];    // gc . nc
  (void)m;
  dot2_fetch(A, J, A.xn, A.g);
  const double b1 = h->hscal[4];
  dot2_fetch(A, J, A.dir, A.gn);
  const double b = b1 + h->hscal[4];
  *tstar_out = NAN;
  *t_out = t_default;
  if (!(d > 0.0)) return MGBX_OK;
  const double tstar = -b / (2.0 * d);
  *tstar_out = tstar;
  if (!(std::isfinite(tstar) && tstar > 0.0)) return MGBX_OK;
  *t_out = std::min(std::max(tstar, std::sqrt(2.220446049250313e-16)), t_default);
  return MGBX_OK;
}

// -------------------------------------------------------------------------------------------------
// create
// -------------------------------------------------------------------------------------------------
void upload_convex(mgbx_handle *h, const mgbx_convex &Q, int64_t n, int nD_user, ConvexDev &cd) {
  Pool &pool = h->pool;
  cudaStream_t s = h->stream;
  memset(&cd, 0, sizeof(cd));
  if (Q.npieces < 0 || Q.npieces > MGBX_MAX_PIECES) throw ArgError("convex set: unsupported number of pieces");
  cd.npieces = Q.npieces;
  for (int k = 0; k < Q.npieces; ++k) {
    const mgbx_piece &q = Q.pieces[k];
    PieceDev &d = cd.pc[k];
    if (q.kind != MGBX_PIECE_EP && q.kind != MGBX_PIECE_LINEAR) throw ArgError("convex piece: unknown kind");
    if (q.ni < 1 || q.ni > MGBX_MAX_NI || q.nc < 1 || q.nc > MGBX_MAX_NC) throw ArgError("convex piece: ni / nc out of range");
    if (q.kind == MGBX_PIECE_EP && q.nc != q.ni) throw ArgError("EP piece needs a square A (nc == ni == nz)");
    if (q.kind == MGBX_PIECE_EP && q.nc < 1) throw ArgError("EP piece needs nz >= 1");
    d.kind = q.kind;
    d.ni = q.ni;
    d.nc = q.nc;
    for (int c = 0; c < q.ni; ++c) {
      d.idx[c] = q.idx ? q.idx[c] : c;
      if (d.idx[c] < 0 || d.idx[c] >= nD_user) throw ArgError("convex piece indexes a D row that does not exist");
    }
    // grid compression: identity A / zero b / uniform p, mu are passed as constants (no HBM traffic)
    bool Aid = (q.nc == q.ni);
    if (Aid && q.A)
      for (int c = 0; c < q.ni && Aid; ++c)
        for (int r = 0; r < q.nc && Aid; ++r) {
          const double want = (r == c) ? 1.0 : 0.0;
          const double *col = q.A + (int64_t)(c * q.nc + r) * n;
          for (int64_t i = 0; i < n; ++i)
            if (col[i] != want) {
              Aid = false;
              break;
            }
        }
    if (!q.A && !(q.nc == q.ni)) throw ArgError("convex piece: A missing");
    d.A = (Aid || !q.A) ? nullptr : pool.upload<double>(q.A, (size_t)n * q.nc * q.ni, s);
    bool bz = true;
    if (q.b)
      for (int64_t i = 0; i < n * q.nc; ++i)
        if (q.b[i] != 0.0) {
          bz = false;
          break;
        }
    d.b = (bz || !q.b) ? nullptr : pool.upload<double>(q.b, (size_t)n * q.nc, s);
    d.p_uniform = 2.0;
    d.mu_uniform = 0.0;
    d.p = d.mu = nullptr;
    if (q.kind == MGBX_PIECE_EP) {
      if (!q.p || !q.mu) throw ArgError("EP piece: p / mu grids missing");
      bool pu = true, mu_u = true;
      for (int64_t i = 1; i < n; ++i) {
        if (q.p[i] != q.p[0]) pu = false;
        if (q.mu[i] != q.mu[0]) mu_u = false;
      }
      if (pu) d.p_uniform = q.p[0];
      else d.p = pool.upload<double>(q.p, n, s);
      if (mu_u) d.mu_uniform = q.mu[0];
      else d.mu = pool.upload<double>(q.mu, n, s);
    }
  }
  cd.select = nullptr;
  if (Q.select) {
    bool all = true;
    for (int64_t i = 0; i < n * Q.npieces; ++i)
      if (Q.select[i] == 0.0) {
        all = false;
        break;
      }
    if (!all) cd.select = pool.upload<double>(Q.select, (size_t)n * Q.npieces, s);
  }
  cd.feas = 0;
  cd.NC = nD_user + 1;
  cd.NF = nD_user;
}

void create_amg(mgbx_handle *h, const mgbx_amg &in, Amg &A) {
  Pool &pool = h->pool;
  cudaStream_t s = h->stream;
  if (in.n <= 0 || in.N <= 0 || in.p <= 0 || in.n != in.N * (int64_t)in.p) throw ArgError("amg: n must equal p*N");
  if (in.nu < 1 || in.nu > MGBX_MAX_ND) throw ArgError("amg: nu out of range");
  if (in.nD < 1 || in.nD > MGBX_MAX_ND) throw ArgError("amg: nD out of range (MGBX_MAX_ND)");
  if (in.L < 1 || in.L > MGBX_MAX_LEVELS) throw ArgError("amg: L out of range");
  if (in.nops < 0 || in.nops > MGBX_MAX_OPS) throw ArgError("amg: too many distinct operators");
  A.n = in.n;
  A.N = in.N;
  A.p = in.p;
  A.nu = in.nu;
  A.nD = in.nD;
  A.L = in.L;
  A.nops = in.nops;
  A.n_global = in.n_global > 0 ? in.n_global : in.n;
  A.var_local.assign(in.nu, 0);
  for (int v = 0; v < in.nu; ++v) A.var_local[v] = (in.var_local && in.var_local[v]) ? 1 : 0;
  A.any_local = false;
  for (char c : A.var_local) A.any_local = A.any_local || c;
  for (int j = 0; j < in.nD; ++j) {
    A.D_var[j] = in.D_var[j];
    A.D_op[j] = in.D_op[j];
    if (A.D_var[j] < 0 || A.D_var[j] >= in.nu) throw ArgError("amg: D row references a state variable that does not exist");
    if (A.D_op[j] >= in.nops) throw ArgError("amg: D row references an operator that does not exist");
  }
  const size_t ppN = (size_t)in.p * in.p * in.N;
  for (int o = 0; o < in.nops; ++o) A.ops[o] = pool.upload<double>(in.op_data[o], ppN, s);
  // dense (spectral) discretisation on a tensor grid: are all operators Kronecker products kron(A1, B1) of n1 x n1 factors
  // (src/spectral2d.jl:28-35)?  Then the Hessian assembly is sum-factorised (build_system, dense_kernels.cuh).
  A.kron_n1 = 0;
  if (in.N == 1 && in.p > 64 && in.nops > 0) {
    const int n1 = isqrt_exact(in.n);
    bool ok = n1 > 1;
    A.kronA.assign(in.nops, {});
    A.kronB.assign(in.nops, {});
    for (int o = 0; o < in.nops && ok; ++o) {
      const double *D = in.op_data[o];   // column-major n x n
      const int64_t nn = in.n;
      ok = kron_factor([&](int64_t r, int64_t c) { return D[r + c * nn]; }, n1, n1, n1, n1, A.kronA[o], A.kronB[o]);
    }
    if (ok) A.kron_n1 = n1;
  }
  A.w = pool.upload<double>(in.w, in.n, s);
  A.voff.resize(in.L);
  A.m.resize(in.L);
  if (!in.R_fine) throw ArgError("amg: R_fine missing");
  for (int l = 0; l < in.L; ++l) {
    // var_offsets == NULL: read the per-variable column blocks off R_fine[l] (what a shim that only sees the reference's
    // `AMG` struct can provide, src/multigrid.jl:278-288)
    if (in.var_offsets) A.voff[l].assign(in.var_offsets + (size_t)l * (in.nu + 1), in.var_offsets + (size_t)(l + 1) * (in.nu + 1));
    else A.voff[l] = derive_var_offsets(in.R_fine[l], in.nu, in.n);
    A.m[l] = A.voff[l][in.nu];
    if (A.voff[l][0] != 0) throw ArgError("amg: var_offsets must start at 0");
    for (int v = 0; v < in.nu; ++v)
      if (A.voff[l][v + 1] < A.voff[l][v]) throw ArgError("amg: var_offsets must be non-decreasing");
    if (l == in.L - 1 && (in.R_fine[l].cols != A.m[l] || in.R_fine[l].rows != (int64_t)in.nu * in.n))
      throw ArgError("amg: R_fine dimension mismatch (rows must be nu*n, cols must match var_offsets)");
  }
  HostTimer tm;
  const bool vb = h->cfg.verbose > 0;
  if (vb) fprintf(stderr, "[mgbx] create_amg: operators + weights queued %.3fs\n", tm.lap());
  A.hRL = csr_from_abi(in.R_fine[in.L - 1]);
  if (vb) fprintf(stderr, "[mgbx]   R_fine[L-1] checked/converted (nnz=%lld) %.3fs\n", (long long)A.hRL.nnz(), tm.lap());
  A.RL = upload_csr(pool, A.hRL, s);
  A.RLt = upload_csr(pool, transpose(A.hRL), s);
  if (vb) fprintf(stderr, "[mgbx]   R, R' uploaded %.3fs\n", tm.lap());
  A.hT.resize(std::max(0, in.L - 1));
  A.T.resize(A.hT.size());
  A.Tt.resize(A.hT.size());
  for (int l = 0; l + 1 < in.L; ++l) {
    if (in.T) {
      if (in.T[l].rows != A.m[l + 1] || in.T[l].cols != A.m[l]) throw ArgError("amg: T dimension mismatch");
      A.hT[l] = csr_from_abi(in.T[l]);
    } else {
      // the reference discards the level transfers (src/multigrid.jl:166-170): recover them from R_fine[l] = R_fine[l+1] T[l]
      if (in.R_fine[l].cols != A.m[l] || in.R_fine[l + 1].cols != A.m[l + 1]) throw ArgError("amg: R_fine[l] columns do not match var_offsets");
      A.hT[l] = recover_transfer(in.R_fine[l + 1], in.R_fine[l]);
    }
    A.T[l] = upload_csr(pool, A.hT[l], s);
    A.Tt[l] = upload_csr(pool, transpose(A.hT[l]), s);
  }
  if (vb) fprintf(stderr, "[mgbx]   level transfers %.3fs\n", tm.lap());
  const int64_t nun = (int64_t)in.nu * in.n;
  A.z = pool.zeros<double>(nun, s);
  A.zsave = pool.zeros<double>(nun, s);
  A.zinit = pool.zeros<double>(nun, s);
  A.zunfin = pool.zeros<double>(nun, s);
  A.zf = pool.zeros<double>(nun, s);
  A.gb = pool.zeros<double>(nun, s);
  A.G = pool.zeros<double>((size_t)in.n * in.nD, s);
  A.f = pool.zeros<double>((size_t)in.n * in.nD, s);
  A.Hn = pool.alloc<double>((size_t)in.n * (in.nD * (in.nD + 1) / 2));
  A.hEEinv = pool.alloc<double>((size_t)in.n * 10);
  A.hKE = pool.alloc<double>((size_t)in.n * in.nD * 4);
  A.slack = pool.alloc<double>(in.n);
  A.chain.resize(in.L);
  A.chain2.resize(in.L);
  for (int l = 0; l < in.L; ++l) {
    A.chain[l] = pool.alloc<double>(A.m[l]);
    A.chain2[l] = pool.alloc<double>(A.m[l]);
  }
  int64_t mmax = 0;
  for (int l = 0; l < in.L; ++l) mmax = std::max(mmax, A.m[l]);
  A.x = pool.zeros<double>(mmax, s);
  A.xn = pool.zeros<double>(mmax, s);
  A.g = pool.zeros<double>(mmax, s);
  A.gn = pool.zeros<double>(mmax, s);
  A.dir = pool.zeros<double>(mmax, s);
  A.rhs = pool.zeros<double>(mmax, s);
  A.tmp = pool.zeros<double>(mmax, s);
  A.xbest = pool.zeros<double>(mmax, s);
  A.gbest = pool.zeros<double>(mmax, s);
  CK(cudaStreamSynchronize(s));
  if (vb) fprintf(stderr, "[mgbx]   work vectors + sync %.3fs\n", tm.lap());
}


// feasibility AMG (src/multigrid.jl:522-536): state [user..., slack], rows [user D...; slack:id; each component:id]
void attach_feasibility(mgbx_handle *h, const mgbx_amg &a1) {
  Amg &A = h->amg[0];
  if (h->has_feas) throw ArgError("feasibility AMG already attached");
  if (a1.n != A.n || a1.nu != A.nu + 1 || a1.nD != A.nD + 1 + A.nu)
    throw ArgError("feasibility AMG must have nu+1 state variables and nD+1+nu rows (src/multigrid.jl:522-536)");
  create_amg(h, a1, h->amg[1]);
  Amg &F = h->amg[1];
  F.cd = A.cd;          // same grids, wrapped
  F.cd.feas = 1;
  F.cd.NC = A.nD + 1;
  F.cd.NF = F.nD;
  F.cd.fb = 1.0;
  F.cd.fR = 10.0;
  // phase-I cost: integral of the slack = row nD of D (0-based) (src/mgb.jl:446-448)
  std::vector<double> c1((size_t)F.n * F.nD, 0.0);
  for (int64_t i = 0; i < F.n; ++i) c1[(size_t)A.nD * F.n + i] = 1.0;
  CK(cudaMemcpyAsync(F.f, c1.data(), sizeof(double) * c1.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->has_feas = true;
}

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
  h->cur_rtol2 = h->cfg.pcg_rtol * h->cfg.pcg_rtol;
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
      CK(cudaFuncSetAttribute(k_coarse_inverse, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)coarse_inverse_smem(kCoarseMaxDense)));
      CK(cudaFuncSetAttribute(k_dense_solve_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dense_solve_small_smem(kCoarseMaxDense)));
      CK(cudaFuncSetAttribute(k_chol_diag_inv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCholDiagSmem));
      CK(cudaFuncSetAttribute(k_chol_solve_blocked, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * kDenseMaxUnknowns)));
    }
    CK(cudaEventCreate(&h->ev0));
    CK(cudaEventCreate(&h->ev1));
    h->partials = h->pool.zeros<double>((size_t)kRedBlocks * 8, h->stream);
    h->ticket = h->pool.zeros<unsigned int>(4, h->stream);
    h->dscal = h->pool.zeros<double>(64, h->stream);
    CK(cudaMallocHost((void **)&h->hscal, sizeof(double) * 64));
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
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
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
    if (which < 0 || which > 1 || (which == 1 && !h->has_feas)) throw ArgError("mgbx_step: no such AMG");
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
    if (which < 0 || which > 1 || (which == 1 && !h->has_feas)) throw ArgError("mgbx_scalars: no such AMG");
    Engine E(h);
    Amg &A = h->amg[which];
    memset(out, 0, sizeof(*out));
    // c_dot_Dz = sum_j dot(w .* f[:, j], D_j z): the linear part of f0 at t = 1, s = 0
    CK(cudaMemsetAsync(A.x, 0, sizeof(double) * A.m[A.L - 1], h->stream));
    EvalOut e = E.eval_f01(A, A.L - 1, 1.0, A.z, A.x, A.gn);
    out->c_dot_Dz = e.lin;
    out->all_finite = 1;
    for (int v = 0; v < A.nu; ++v) {
      E_LAUNCH(KC_VEC, k_maxabs<<<E.red_grid(A.n), kRedThreads, 0, h->stream>>>(A.n, A.z + (int64_t)v * A.n, h->partials, h->ticket, h->dscal));
      if (E.dist()) E.allreduce(h->dscal, 3, kNcclMax);
      E.fetch(3);
      out->var_max[v] = h->hscal[0];
      out->var_absmax[v] = h->hscal[1];
      if (h->hscal[2] != 0.0) out->all_finite = 0;
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
    for (int v = 0; v < A.nu; ++v) {
      E_LAUNCH(KC_VEC, k_maxabs<<<E.red_grid(A.n), kRedThreads, 0, h->stream>>>(A.n, A.z + (int64_t)v * A.n, h->partials, h->ticket, h->dscal));
      if (E.dist()) E.allreduce(h->dscal, 3, kNcclMax);
      E.fetch(3);
      zmax = std::max(zmax, h->hscal[1]);
    }
    *zabsmax = zmax;
    *b = 0.0;
    if (*needs_phase1) {
      if (!h->has_feas) return MGBX_OK;   // the host attaches the feasibility AMG (mgbx_attach_feasibility) and calls again
      Amg &F = h->amg[1];
      // slack_i = 2*max(slack_fn(D z0), 1);  b = 2*max(1, max slack)   (src/mgb.jl:437-445)
      NodeParams P = E.node_params(A, 0.0);   // A.zf holds z0 from the probe
      E_LAUNCH(KC_NODE_F01, launch_node<NODE_SLACK>(P, E.red_grid(A.n), h->stream));
      E_LAUNCH(KC_VEC, k_phase1_slack<<<nblk(A.n), 256, 0, h->stream>>>(A.n, A.slack, F.zinit + (int64_t)A.nu * A.n));
      E.copy(F.zinit, A.z, (int64_t)A.nu * A.n);
      E.copy(F.z, F.zinit, (int64_t)F.nu * F.n);
      E_LAUNCH(KC_VEC, k_maxabs<<<E.red_grid(A.n), kRedThreads, 0, h->stream>>>(A.n, F.zinit + (int64_t)A.nu * A.n, h->partials, h->ticket, h->dscal));
      if (E.dist()) E.allreduce(h->dscal, 3, kNcclMax);
      E.fetch(3);
      *b = 2.0 * std::max(1.0, h->hscal[0]);
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
    if (which < 0 || which > 1 || (which == 1 && !h->has_feas)) throw ArgError("no such AMG");
    Amg &A = h->amg[which];
    if (level < 0 || level >= A.L) throw ArgError("no such level");
    if (order != 0 && order != 1) throw ArgError("order must be 0 or 1 (use mgbx_hessian_values for f2)");
    Engine E(h);
    CK(cudaMemcpyAsync(A.xn, s, sizeof(double) * A.m[level], cudaMemcpyHostToDevice, h->stream));
    EvalOut e = E.eval_f01(A, level, t, A.z, A.xn, A.gn);
    if (order == 0) out[0] = e.y;
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
    if (which < 0 || which > 1 || (which == 1 && !h->has_feas)) throw ArgError("no such AMG");
    Amg &A = h->amg[which];
    if (level < 0 || level >= A.L) throw ArgError("no such level");
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
    if (which < 0 || which > 1 || (which == 1 && !h->has_feas)) throw ArgError("no such AMG");
    Amg &A = h->amg[which];
    if (level < 0 || level >= A.L) throw ArgError("no such level");
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
    {
      E.prolong_to_fine(A, level, A.xn, A.z, A.zf);
      NodeParams P = E.node_params(A, t);
      P.nK = S.nK;
      P.nE = 0;
      for (int j = 0; j < MGBX_MAX_ND; ++j) {
        P.Krow[j] = S.Krow[j];
        P.Erow[j] = -1;
      }
      P.Hn = A.Hn;
      E_LAUNCH(KC_NODE_F2, launch_node<NODE_F2>(P, E.red_grid(A.n), h->stream));
      ElemParams EP = E.elem_params(A);
      E_LAUNCH(KC_BLOCKHESS, k_blockhess<<<nblk(S.hblk_size), 256, 0, h->stream>>>(EP, S.pl, A.Hn, S.Hblk));
      E_LAUNCH(KC_GATHER, k_sell_gather<<<nblk(S.lev[0].A.nnz), 256, 0, h->stream>>>(S.top, S.Hblk, S.lev[0].A.val));
      if (E.dist()) E.allreduce(S.lev[0].A.val, S.lev[0].A.nnz);
      const int ktop = A.L - 1 - level;
      for (int k = 0; k < ktop; ++k) {
        SysLevel &Lv = S.lev[k];
        SysLevel &Lc = S.lev[k + 1];
        if (Lv.T_identity) continue;   // aliased
        E_LAUNCH(KC_SPGEMM, k_sell_gather<<<nblk(Lv.AT.nnz), 256, 0, h->stream>>>(Lv.s1, Lv.A.val, Lv.AT.val));
        E_LAUNCH(KC_SPGEMM, k_sell_gather<<<nblk(Lc.A.nnz), 256, 0, h->stream>>>(Lv.s2, Lv.AT.val, Lc.A.val));
      }
      SysLevel &Lv = S.lev[ktop];
      CK(cudaMemcpyAsync(val, Lv.A.val, sizeof(double) * Lv.A.nnz, cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
    }
    return MGBX_OK;
  });
}

int mgbx_solve_newton_system(mgbx_handle *h, int which, int level, double t, const double *s, const double *rhs, double *x,
                             int32_t *pcg_iters) {
  if (!h || !s || !rhs || !x) return MGBX_ERR_ARG;
  return guarded(h, [&]() -> int {
    if (which < 0 || which > 1 || (which == 1 && !h->has_feas)) throw ArgError("no such AMG");
    Amg &A = h->amg[which];
    if (level < 0 || level >= A.L) throw ArgError("no such level");
    Engine E(h);
    System &S = E.system_for(A, level);
    const int64_t m = A.m[level];
    CK(cudaMemcpyAsync(A.xn, s, sizeof(double) * m, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(A.gn, rhs, sizeof(double) * m, cudaMemcpyHostToDevice, h->stream));
    E.assemble(A, S, level, t, A.z, A.xn);
    const int it = E.solve(A, S, level, A.gn, A.dir);
    if (pcg_iters) *pcg_iters = it;
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
