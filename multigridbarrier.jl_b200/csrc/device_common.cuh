// device_common.cuh -- parameter structs, size helpers and __device__ helpers shared by the kernel headers and the host
// units.  It defines no kernel: each __global__ lives in exactly one of kernels.cuh (evaluation, assembly), dense_kernels.cuh
// (DMMA GEMM and sum-factorised assembly), solver_kernels.cuh (preconditioner setup, condensation, direct solves) or
// setup_kernels.cuh (plan construction), and each of those is compiled by one translation unit only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "elem_schur.cuh"
#include "node_barrier.cuh"

namespace mgbx {

#define MGBX_MAX_OPS 8
constexpr int kRedBlocks = 592;   // 148 SMs x 4
constexpr int kRedThreads = 256;

struct DevCsr {
  int64_t rows = 0, cols = 0, nnz = 0;
  int64_t *ptr = nullptr;
  int32_t *idx = nullptr;
  double *val = nullptr;
};

// ------------------------------------------------------------------------------------------------
// reductions
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xffffffffu, v, o));
  return v;
}

// Block-reduce NV values (op[k] == 0: sum, 1: max); result valid in thread 0.
template <int NV>
__device__ __forceinline__ void block_reduce(double (&v)[NV], const int (&op)[NV]) {
  __shared__ double sm[NV][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    v[k] = op[k] ? warp_max(v[k]) : warp_sum(v[k]);
    if (lane == 0) sm[k][wid] = v[k];
  }
  __syncthreads();
  if (wid == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      double x = lane < nw ? sm[k][lane] : (op[k] ? -INFINITY : 0.0);
      v[k] = op[k] ? warp_max(x) : warp_sum(x);
    }
  }
  __syncthreads();
}

// Grid-wide fixed-order reduction: every block deposits its partials, the last block to arrive
// (atomic ticket) combines them in block order and writes out[0..NV).
template <int NV>
__device__ __forceinline__ void grid_reduce(double (&v)[NV], const int (&op)[NV], double *partials,
                                            unsigned int *ticket, double *out) {
  block_reduce<NV>(v, op);
  __shared__ bool last;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) partials[(size_t)k * gridDim.x + blockIdx.x] = v[k];
    __threadfence();
    const unsigned int t = atomicAdd(ticket, 1u);
    last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (last) {
    __threadfence();
    double a[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      double acc = op[k] ? -INFINITY : 0.0;
      for (unsigned int b = threadIdx.x; b < gridDim.x; b += blockDim.x) {
        const double x = ((volatile double *)partials)[(size_t)k * gridDim.x + b];
        acc = op[k] ? fmax(acc, x) : acc + x;
      }
      a[k] = acc;
    }
    block_reduce<NV>(a, op);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int k = 0; k < NV; ++k) out[k] = a[k];
      *ticket = 0;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// per-node barrier evaluation
// ------------------------------------------------------------------------------------------------
enum { NODE_F01 = 0, NODE_F2 = 1, NODE_SLACK = 2 };

struct NodeParams {
  int64_t n;
  int p, nu, nD;
  int D_var[MGBX_MAX_ND], D_op[MGBX_MAX_ND];
  const double *ops[MGBX_MAX_OPS];   // each N x (p x p), offset e*p*p + col*p + row
  const double *zf;                  // nu*n broken state  z0 + R s
  const double *w, *f, *bw;          // weights, cost grid n x nD, barrier weights or nullptr
  double t, inv_n;
  ConvexDev cd;
  // F01 outputs
  double *G;                         // n x nD: bw*F1 + w*t*f
  double *partials;                  // 4 x gridDim
  unsigned int *ticket;
  double *red_out;                   // [0] sum bw*F0 (or sum F0), [1] sum w*(c.Dz), [2] #non-finite F0, [3] max slack
  // F2 outputs (condensed when nE > 0)
  int nK, nE;
  int Krow[MGBX_MAX_ND];             // D rows of the kept variables
  int Erow[MGBX_MAX_ND];             // per D row: index of its eliminated variable, or -1
  double *Hn;                        // n x nK(nK+1)/2, packed (a<=b): a*nK - a(a-1)/2 + (b-a)
  double *hEEinv;                    // n x nE(nE+1)/2
  double *hKE;                       // n x (nK*nE): entry (a, ev) at column a*nE + ev
  unsigned schur_pieces, schur_elim; // pieces condensed analytically by node_eval / the eliminated variables they cover (bit masks)
  // SLACK output
  double *slack;                     // n
};

// the analytic condensation only applies when something is eliminated
__device__ __forceinline__ unsigned nE_mask_guard(const NodeParams &P) { return P.nE > 0 ? P.schur_pieces : 0u; }

__device__ __forceinline__ void node_Dz(const NodeParams &P, int64_t i, double *y) {
  const int64_t e = i / P.p;
  const int r = (int)(i - e * P.p);
  for (int j = 0; j < P.nD; ++j) {
    const int v = P.D_var[j], o = P.D_op[j];
    const double *zv = P.zf + (int64_t)v * P.n;
    if (o < 0) {
      y[j] = zv[i];
    } else {
      const double *blk = P.ops[o] + e * (int64_t)(P.p * P.p) + r;
      const double *ze = zv + e * P.p;
      double acc = 0.0;
      for (int c = 0; c < P.p; ++c) acc += blk[(int64_t)c * P.p] * ze[c];
      y[j] = acc;
    }
  }
}

// small symmetric positive definite inverse (nE <= 4) by Cholesky; packed lower-by-rows in/out is
// avoided: we work on a full nE x nE array.
__device__ __forceinline__ void spd_inverse(double *M, int m) {
  // in-place Cholesky M = L L'
  double L[16];
  for (int i = 0; i < m; ++i)
    for (int j = 0; j <= i; ++j) {
      double s = M[i * m + j];
      for (int k = 0; k < j; ++k) s -= L[i * m + k] * L[j * m + k];
      L[i * m + j] = (i == j) ? sqrt(s) : s / L[j * m + j];
    }
  // Linv
  double Li[16];
  for (int i = 0; i < m; ++i)
    for (int j = 0; j < m; ++j) Li[i * m + j] = 0.0;
  for (int j = 0; j < m; ++j) {
    Li[j * m + j] = 1.0 / L[j * m + j];
    for (int i = j + 1; i < m; ++i) {
      double s = 0.0;
      for (int k = j; k < i; ++k) s -= L[i * m + k] * Li[k * m + j];
      Li[i * m + j] = s / L[i * m + i];
    }
  }
  for (int i = 0; i < m; ++i)
    for (int j = 0; j < m; ++j) {
      double s = 0.0;
      for (int k = (i > j ? i : j); k < m; ++k) s += Li[k * m + i] * Li[k * m + j];
      M[i * m + j] = s;
    }
}

// ------------------------------------------------------------------------------------------------
// element blocks
// ------------------------------------------------------------------------------------------------
struct ElemParams {
  int64_t n, N;
  int p, nD;
  int D_var[MGBX_MAX_ND], D_op[MGBX_MAX_ND];
  const double *ops[MGBX_MAX_OPS];
  int nK;                    // rows used (Hessian: kept rows; gradient: all rows)
  int Krow[MGBX_MAX_ND];
};

// pairs (va, vb) of state variables whose Hessian blocks are assembled
struct PairList {
  int npairs;
  int va[16], vb[16];
};

// ------------------------------------------------------------------------------------------------
// condensation helpers (node-local elimination of the :full variables)
// ------------------------------------------------------------------------------------------------
struct CondParams {
  int64_t n;
  int nD, nK, nE;
  int Krow[MGBX_MAX_ND];
  int64_t Eoff[4];            // first index of eliminated variable ev in the level-L vector
  const double *hEEinv, *hKE;
};

// an element-local eliminated variable (elem_schur.cuh): nc coefficients per element, the only eliminated variable
struct ElemLocal {
  int nc;
  const int64_t *c0;          // per element: index of its first coefficient within the variable's block
  const double *P;            // per element: the p x nc block of R_fine (row-major)
  double *R;                  // per element: packed factor R of W = A^{1/2} P (elem_rsize(nc)), written by each assembly
};

// ------------------------------------------------------------------------------------------------
// multi-GPU (element partition): a level vector is a list of segments, one per state variable; `shared`
// segments are replicated on every rank, `local` segments hold the rank's own node-local unknowns.  Reductions
// over such vectors are split: the shared part is summed redundantly (identically) on every rank, the local
// part is a partial sum completed by an all-reduce.
// ------------------------------------------------------------------------------------------------
struct SegList {
  int n;
  int64_t off[MGBX_MAX_ND + 1];   // segment q = [off[q], off[q+1])
  int local[MGBX_MAX_ND];
};
__device__ __forceinline__ int seg_is_local(const SegList &S, int64_t i) {
  int q = 0;
  while (q + 1 < S.n && i >= S.off[q + 1]) ++q;
  return S.local[q];
}

// ------------------------------------------------------------------------------------------------
// Fused element kernels (north-star items 1 + 2): one pass per barrier evaluation.
//   k_elem<NODE_F01>  apply_D -> F0/F1 -> (1/n) F1 + w.*c -> sum_k D_k' y_k      (k_node<F01> + k_blockgrad in one kernel)
//   k_elem<NODE_F2>   apply_D -> F2 -> node-local Schur condensation -> sum_jk D_j' diag(h_jk) D_k   (k_node<F2> + k_blockhess)
// A block owns `epb` whole elements per tile (one thread per broken node) and walks tiles grid-stride.  The
// operator blocks of the tile are staged ONCE in shared memory (padded against bank conflicts) and serve both
// the forward application D z and the adjoint / triple product; the per-node samples (G or the packed Hessian)
// are exchanged through shared memory and never touch HBM.  Replaces, per evaluation, nD block matvecs +
// map_rows + nD adjoint matvecs (src/convex.jl:155-179) resp. nD^2 block_fused_triple! calls each allocating
// p x p x N (src/convex.jl:185-200, src/BlockMatrices.jl:170-212).
// ------------------------------------------------------------------------------------------------
struct ElemFused {
  NodeParams np;
  PairList pl;
  double *Hblk;     // F2: pairs x N x p x p
  double *gb;       // F01: nu x n
  int64_t N;
  int epb;          // elements per tile
  int p1, ES;       // padded column stride and element stride of the staged operator blocks (doubles)
  int nex;          // exchange rows
  int nops;
};

inline size_t elem_fused_smem(int nops, int epb, int ES, int nu, int nex, int p) {
  return sizeof(double) * ((size_t)nops * epb * ES + (size_t)(nu + nex) * epb * p);
}

// ------------------------------------------------------------------------------------------------
// k_elem_plap<MODE, DIM>: the fused element kernel specialised for the reference's default problem family
// (src/mgb.jl:587-613,711-727): state (u, s), D = [u:id; u:d_1..d_DIM; s:id], one Euclidean-power cone on rows
// 1..DIM+1 with identity A, zero b and uniform p, mu; s condensed node-locally.  Same shared-memory staging and
// the same outputs (gb; hEEinv, hKE, Hblk) as the generic k_elem, but every loop over D rows / pieces / index maps
// is resolved at compile time: the generic kernel is instruction-bound (~1700 warp instructions per warp of nodes,
// 90% of them index bookkeeping), this one is bound by the operator-block stream.
// ------------------------------------------------------------------------------------------------
struct FastDiv {
  unsigned int mul, d;   // q = umulhi(t, mul) for 0 <= t < 2^16, 1 <= d < 2^16
};
inline FastDiv make_fastdiv(unsigned int d) {
  FastDiv f;
  f.d = d;
  f.mul = (unsigned int)((0x100000000ull + d - 1) / d);
  return f;
}
__device__ __forceinline__ unsigned int fdiv(unsigned int t, const FastDiv &f) { return f.d == 1 ? t : __umulhi(t, f.mul); }

struct PlapParams {
  int64_t n, N;
  int p, epb, p1, ES;
  int bulk;                    // 0: per-double cp.async staging; 1: one bulk copy per operator slab (p1 == p, ES == p*p);
                               // 2: one bulk copy per block column (p even, p1 and ES even).  Ragged tiles use the per-double path.
  FastDiv dp, dpp;
  const double *ops[3];
  const double *zu, *zs;       // broken state of u and s (n each)
  const double *w, *f, *bw;    // f: n x (DIM+2)
  double t, inv_n, pexp, mu;
  // F01
  double *gbu, *gbs;
  double *partials;
  unsigned int *ticket;
  double *red_out;
  // F2
  double *hEEinv, *hKE, *Hblk;
};

// shared memory: two input buffers (operator blocks + the tile's node inputs, filled by cp.async one tile ahead) + exchange rows
inline size_t elem_plap_smem(int dim, int epb, int ES, int p, bool condensed = true) {
  const size_t tm = (size_t)epb * p;
  const size_t buf = (size_t)dim * epb * ES + (size_t)(4 + dim + 2) * tm;
  const int nh = (dim * (dim + 1)) / 2;
  const int nex = condensed ? (nh > dim ? nh : dim) : nh + dim + 1;
  return sizeof(double) * (2 * buf + (size_t)nex * tm);
}

__device__ __forceinline__ void cp_async8(void *smem, const void *gmem) {
  const unsigned int sa = (unsigned int)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ---- bulk asynchronous copies (cp.async.bulk, the 1-D form of TMA: SASS UBLKCP) completing on an mbarrier -------------------
__device__ __forceinline__ void mbar_init(unsigned long long *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned int)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned int bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((unsigned int)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned int parity) {
  const unsigned int a = (unsigned int)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(a),
      "r"(parity)
      : "memory");
}
// bytes: multiple of 16; smem and gmem 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void *smem, const void *gmem, unsigned int bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"((unsigned int)__cvta_generic_to_shared(smem)),
               "l"(gmem), "r"(bytes), "r"((unsigned int)__cvta_generic_to_shared(bar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
// sliced-ELL gather:  out[nz] = sum_{k < cnt[nz]} w[off + 32k] * in[src[off + 32k]],  off = sptr[nz/32] + nz%32
// ------------------------------------------------------------------------------------------------
struct SellPlan {
  int64_t nout = 0, nslices = 0, nterms = 0;   // nterms: real (unpadded) terms
  int64_t *sptr = nullptr;                      // nslices + 1 entry offsets
  int32_t *cnt = nullptr;                       // nout
  int32_t *src = nullptr;                       // padded entries
  double *w = nullptr;                          // padded entries, or nullptr (all weights 1)
};

__device__ __forceinline__ int64_t csr_find(const DevCsr &A, int64_t row, int32_t col) {
  int64_t lo = A.ptr[row], hi = A.ptr[row + 1];
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int32_t c = A.idx[mid];
    if (c < col) lo = mid + 1;
    else if (c > col) hi = mid;
    else return mid;
  }
  return -1;
}

// coarse dense inverse (k_coarse_inverse) and small direct solve (k_dense_solve_small): one CTA, m <= kCoarseMaxDense
//   coarse inverse shared layout: S[m][m+1] (scaled matrix -> Cholesky factor L), Li[m(m+1)/2] (packed inverse of L), d[m]
constexpr int kCoarseMaxDense = 128;
inline size_t coarse_inverse_smem(int m) { return sizeof(double) * ((size_t)m * (m + 1) + (size_t)m * (m + 1) / 2 + m); }
inline size_t dense_solve_small_smem(int m) { return sizeof(double) * ((size_t)m * (m + 1) + 2 * (size_t)m); }

constexpr int kGemmBM = 64, kGemmBN = 64, kGemmBK = 16, kGemmLd = kGemmBK + 4;

__device__ __forceinline__ void dmma_m8n8k4(double &d0, double &d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// blocked dense Cholesky (solver_kernels.cuh): panel width and the diagonal-block kernel's shared memory
constexpr int kCholNB = 64;
constexpr size_t kCholDiagSmem = sizeof(double) * 2 * kCholNB * (kCholNB + 1);
constexpr int kDenseMaxUnknowns = 8192;   // blocked Cholesky: the triangular solve keeps the right-hand side in shared memory (64 KB)

// ------------------------------------------------------------------------------------------------
// Sum-factorised (Kronecker) assembly for tensor-product spectral discretisations (spectral2d).
// There :dx = kron(DX, I), :dy = kron(I, DX), :id = kron(I, I) (src/spectral2d.jl:28-35) and every prolongation is
// R = kron(R1, R1) (src/spectral2d.jl:22-25), so each D_j R_v = kron(P_j, Q_j) with n1 x c factors, and the block (a, b) of
// R'HR = sum_{j in a, k in b} (P_j (x) Q_j)' diag(h_jk) (P_k (x) Q_k)   has the entries
//     [(i, i'), (l, l')] = sum_e P_j[e, i] P_k[e, l] * ( sum_f Q_j[f, i'] h_jk[e, f] Q_k[f, l'] ).
// Inner sum: k_kron_w (n1 small products per node row e);  outer sum over (pair, e): ONE DMMA GEMM per block with the
// constant operand AA[(i, l)][c n1 + e] = P_j[e, i] P_k[e, l] (built once) -- 2 c1a c1b c2a c2b (pairs n1) flops instead of
// the 2 n^3 per pair of the unstructured product (n = n1^2): 31 GFLOP instead of 1.6 TFLOP per assembly at n1 = 64.
// ------------------------------------------------------------------------------------------------
struct KronCombo {
  const double *Qj, *Qk;   // n1 x c2a / n1 x c2b, row-major
  const double *h;         // node samples h_jk (n = n1 * n1), node q = e * n1 + f
};
constexpr int kKronMaxCombos = 16;
struct KronWArgs {
  int n1, c2a, c2b, ncombo, K;   // K = ncombo * n1
  KronCombo c[kKronMaxCombos];
};

// Element-block -> CSR gather plan.  One thread per non-zero (i, j) of the top pattern: the pair of state
// variables is fixed by the variable blocks i and j live in; the elements incident to i come from the
// transposed element incidence; inside an element the rows r (resp. c) whose R row carries column i (resp. j)
// are found by binary search.  Terms are emitted in the order (element, r, c): fixed, so the gather is
// deterministic.  FILL == 0 counts (cnt, slice widths), FILL == 1 writes src / w.
struct TopPlanParams {
  DevCsr R;                    // level->broken prolongation of the system's top level (rows nu*n)
  DevCsr EincT;                // system unknown -> incident elements (sorted)
  DevCsr pat;                  // top pattern
  const int32_t *rowof;        // row of every non-zero of pat
  int64_t n, N;
  int p, nkept, unit;
  int kept[MGBX_MAX_ND];       // state variable of kept slot q
  int64_t off[MGBX_MAX_ND + 1];    // system offsets of the kept slots
  int64_t rcol0[MGBX_MAX_ND];      // first R column of the kept slot's variable
  int pair_of[MGBX_MAX_ND * MGBX_MAX_ND];   // [qa * nkept + qb] -> pair index or -1
};

}  // namespace mgbx
