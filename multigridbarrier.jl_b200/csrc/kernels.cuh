// kernels.cuh -- sm_100a device kernels of the barrier-Newton hot path.
//
// What each kernel replaces in the reference (paths under /root/reference):
//   k_node            apply_D + map_rows_gpu(F0/F1/F2) + the (1/n)·y + w.*c combination
//                     src/convex.jl:125,155-202,213-257; ext/MultiGridBarrierCUDAExt/map_rows_gpu.jl:20-63,
//                     block_ops.jl:118-133 (_block_matvec_kernel!)
//   k_blockgrad       sum_k D_k' y_k                    src/convex.jl:173-178; block_ops.jl:135-148
//   k_blockhess       sum_{j,k} D_j' diag(y_jk) D_k     src/convex.jl:185-200; block_ops.jl:58-75 (called nD^2 times there)
//   (solver_kernels.cuh: k_sell_gather = R'HR into the fixed pattern and the Galerkin products)
//   k_spmv*           R*s, R'*g                          CUSPARSE in the reference (src/convex.jl:156,178)
//   k_l1diag          smoother diagonals and the Gershgorin bound of every level of the solve kernel
//   (pcg2.cu: k_pcg2 = the multigrid-preconditioned CG solve, replacing cuDSS LDL' (ext/.../cudss_solver.jl:264-381))
//   (dense_kernels.cuh: DMMA GEMM and blocked Cholesky of the spectral path)
// All reductions are fixed-order (block tree + last-block pass): results are run-to-run deterministic.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

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
// sparse matrix-vector products.  G threads cooperate on one row (G = 1, 4, 32).
//   y = alpha * A x + (y0 ? y0 : 0)
// ------------------------------------------------------------------------------------------------
template <int G>
__global__ void __launch_bounds__(256) k_spmv(DevCsr A, const double *__restrict__ x, const double *y0, double alpha,
                                               double *y) {
  const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t row = gtid / G;
  const int sub = (int)(gtid % G);
  if (row >= A.rows) return;   // G divides 32 and the block size, so whole groups exit together
  const int64_t b = A.ptr[row], e = A.ptr[row + 1];
  double acc = 0.0;
  for (int64_t k = b + sub; k < e; k += G) acc += A.val[k] * x[A.idx[k]];
  if (G > 1) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o, G);
  }
  if (sub == 0) y[row] = alpha * acc + (y0 ? y0[row] : 0.0);
}

// dinv = 1 / sum_k |a_ik|  (l1-Jacobi), diag = 1 / a_ii, and the Gershgorin bound of lambda_max(D^-1 A),
// max_i sum_k |a_ik| / a_ii, folded with atomicMax on the bit pattern (non-negative doubles order like integers;
// max is order-independent, so the result is deterministic).  *lam_bits must be zeroed before the launch.
__global__ void __launch_bounds__(256) k_l1diag(DevCsr A, double *dinv, double *diag, unsigned long long *lam_bits) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double ratio = 0.0;
  if (row < A.rows) {
    double s = 0.0, d = 0.0;
    for (int64_t k = A.ptr[row]; k < A.ptr[row + 1]; ++k) {
      s += fabs(A.val[k]);
      if (A.idx[k] == row) d = A.val[k];
    }
    dinv[row] = s > 0.0 ? 1.0 / s : 0.0;
    if (diag) diag[row] = d > 0.0 ? 1.0 / d : 0.0;   // inverse diagonal (Chebyshev scaling)
    if (d > 0.0 && isfinite(s)) ratio = s / d;
  }
  if (lam_bits) {
    ratio = warp_max(ratio);
    if ((threadIdx.x & 31) == 0 && ratio > 0.0) atomicMax(lam_bits, (unsigned long long)__double_as_longlong(ratio));
  }
}

// ------------------------------------------------------------------------------------------------
// per-node barrier kernel
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

// NDT >= nD bounds the per-thread arrays (y, F1, F2 = NDT^2 doubles) so that they stay in registers / L1
template <int MODE, int NDT>
__global__ void __launch_bounds__(kRedThreads) k_node(NodeParams P) {
  double red[4] = {0.0, 0.0, 0.0, -INFINITY};
  const int op[4] = {0, 0, 0, 1};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P.n; i += (int64_t)gridDim.x * blockDim.x) {
    double y[NDT];
    node_Dz(P, i, y);
    if (MODE == NODE_SLACK) {
      const double s = node_slack(P.cd, P.n, i, y);
      P.slack[i] = s;
      red[3] = fmax(red[3], s);
      continue;
    }
    const int nD = P.nD;
    const double bwi = P.bw ? P.bw[i] : 1.0;
    const bool active = !(P.bw && bwi == 0.0);
    double F1[NDT];
    if (MODE == NODE_F01) {
      double F0 = 0.0;
      if (active) F0 = node_eval(P.cd, P.n, i, y, 1, F1, nullptr);
      else
        for (int j = 0; j < nD; ++j) F1[j] = 0.0;
      const double wi = P.w[i];
      double lin = 0.0;
      const double sc = P.bw ? bwi : P.inv_n;
      for (int j = 0; j < nD; ++j) {
        const double c = P.t * P.f[i + (int64_t)j * P.n];
        lin += c * y[j];
        P.G[i + (int64_t)j * P.n] = (active ? sc * F1[j] : 0.0) + wi * c;
      }
      red[0] += active ? (P.bw ? bwi * F0 : F0) : 0.0;
      red[1] += wi * lin;
      if (!isfinite(F0)) red[2] += 1.0;
    } else {   // NODE_F2
      double F2[NDT * NDT];
      const double sc = P.bw ? bwi : P.inv_n;
      if (active) {
        node_eval(P.cd, P.n, i, y, 2, F1, F2, nE_mask_guard(P));
        for (int k = 0; k < nD * nD; ++k) F2[k] *= sc;
      } else {
        for (int k = 0; k < nD * nD; ++k) F2[k] = 0.0;
      }
      const int nK = P.nK, nE = P.nE;
      if (nE == 0) {
        int q = 0;
        for (int a = 0; a < nK; ++a)
          for (int b = a; b < nK; ++b, ++q) P.Hn[i + (int64_t)q * P.n] = F2[P.Krow[a] * nD + P.Krow[b]];
      } else {
        double hEE[16], hKE[NDT * 4];
        for (int k = 0; k < nE * nE; ++k) hEE[k] = 0.0;
        for (int k = 0; k < nK * nE; ++k) hKE[k] = 0.0;
        for (int j = 0; j < nD; ++j) {
          const int ej = P.Erow[j];
          if (ej < 0) continue;
          for (int k = 0; k < nD; ++k) {
            const int ek = P.Erow[k];
            if (ek >= 0) hEE[ej * nE + ek] += F2[j * nD + k];
          }
          for (int a = 0; a < nK; ++a) hKE[a * nE + ej] += F2[P.Krow[a] * nD + j];
        }
        spd_inverse(hEE, nE);
        {
          int q = 0;
          for (int a = 0; a < nE; ++a)
            for (int b = a; b < nE; ++b, ++q) P.hEEinv[i + (int64_t)q * P.n] = hEE[a * nE + b];
        }
        for (int k = 0; k < nK * nE; ++k) P.hKE[i + (int64_t)k * P.n] = hKE[k];
        // W = hEEinv * hEK  (nE x nK);  Hn = hKK - hKE W
        int q = 0;
        for (int a = 0; a < nK; ++a)
          for (int b = a; b < nK; ++b, ++q) {
            double s = F2[P.Krow[a] * nD + P.Krow[b]];
            for (int ev = 0; ev < nE; ++ev) {
              if ((P.schur_elim >> ev) & 1u) continue;   // already condensed analytically inside node_eval
              double wv = 0.0;
              for (int ew = 0; ew < nE; ++ew) wv += hEE[ev * nE + ew] * hKE[b * nE + ew];
              s -= hKE[a * nE + ev] * wv;
            }
            P.Hn[i + (int64_t)q * P.n] = s;
          }
      }
    }
  }
  if (MODE != NODE_F2) grid_reduce<4>(red, op, P.partials, P.ticket, P.red_out);
}

// ------------------------------------------------------------------------------------------------
// element-block kernels
// ------------------------------------------------------------------------------------------------
struct ElemParams {
  int64_t n, N;
  int p, nD;
  int D_var[MGBX_MAX_ND], D_op[MGBX_MAX_ND];
  const double *ops[MGBX_MAX_OPS];
  int nK;                    // rows used (Hessian: kept rows; gradient: all rows)
  int Krow[MGBX_MAX_ND];
};

// gb[v*n + e*p + c] = sum_{j in rows(v), j in Krow} sum_q D_j[q][c] * G[j*n + e*p + q]
// one thread per (variable slot, broken node)
__global__ void __launch_bounds__(256) k_blockgrad(ElemParams P, const double *__restrict__ G, double *gb, int nu) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= (int64_t)nu * P.n) return;
  const int v = (int)(tid / P.n);
  const int64_t i = tid - (int64_t)v * P.n;
  const int64_t e = i / P.p;
  const int c = (int)(i - e * P.p);
  double acc = 0.0;
  for (int jj = 0; jj < P.nK; ++jj) {
    const int j = P.Krow[jj];
    if (P.D_var[j] != v) continue;
    const int o = P.D_op[j];
    const double *g = G + (int64_t)j * P.n;
    if (o < 0) acc += g[i];
    else {
      const double *blk = P.ops[o] + e * (int64_t)(P.p * P.p) + (int64_t)c * P.p;
      const double *ge = g + e * P.p;
      for (int q = 0; q < P.p; ++q) acc += blk[q] * ge[q];
    }
  }
  gb[tid] = acc;
}

// Hblk[((pair*N + e)*p + r)*p + c] = sum_{j in rows(a), k in rows(b)} sum_q D_j[q][r] h_jk[q] D_k[q][c]
// with h packed over the kept rows.  One thread per (pair, e, r, c).
struct PairList {
  int npairs;
  int va[16], vb[16];
};
__global__ void __launch_bounds__(256) k_blockhess(ElemParams P, PairList PL, const double *__restrict__ Hn, double *Hblk) {
  const int pp = P.p * P.p;
  const int64_t total = (int64_t)PL.npairs * P.N * pp;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= total) return;
  const int c = (int)(tid % P.p);
  const int r = (int)((tid / P.p) % P.p);
  const int64_t e = (tid / pp) % P.N;
  const int pr = (int)(tid / ((int64_t)pp * P.N));
  const int va = PL.va[pr], vb = PL.vb[pr];
  const int nK = P.nK;
  const int64_t base = e * P.p;
  double acc = 0.0;
  for (int ja = 0; ja < nK; ++ja) {
    const int j = P.Krow[ja];
    if (P.D_var[j] != va) continue;
    const int oj = P.D_op[j];
    for (int kb = 0; kb < nK; ++kb) {
      const int k = P.Krow[kb];
      if (P.D_var[k] != vb) continue;
      const int ok = P.D_op[k];
      const int a = ja < kb ? ja : kb, b = ja < kb ? kb : ja;
      const double *h = Hn + (int64_t)(a * nK - (a * (a - 1)) / 2 + (b - a)) * P.n + base;
      if (oj < 0 && ok < 0) {
        if (r == c) acc += h[r];
      } else if (oj < 0) {
        acc += h[r] * P.ops[ok][e * (int64_t)pp + (int64_t)c * P.p + r];
      } else if (ok < 0) {
        acc += P.ops[oj][e * (int64_t)pp + (int64_t)r * P.p + c] * h[c];
      } else {
        const double *dj = P.ops[oj] + e * (int64_t)pp + (int64_t)r * P.p;
        const double *dk = P.ops[ok] + e * (int64_t)pp + (int64_t)c * P.p;
        double s = 0.0;
        for (int q = 0; q < P.p; ++q) s += dj[q] * h[q] * dk[q];
        acc += s;
      }
    }
  }
  Hblk[tid] = acc;
}

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

// Gt[Krow[a]*n + i] = - sum_ev hKE[a][ev] * (hEEinv * gE)[ev],  gE[ev] = g[Eoff[ev] + i]; other rows of Gt are not touched
__global__ void __launch_bounds__(256) k_condense_rhs(CondParams P, const double *__restrict__ g, double *Gt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  double gE[4], tE[4], Hi[16];
  const int nE = P.nE;
  for (int ev = 0; ev < nE; ++ev) gE[ev] = g[P.Eoff[ev] + i];
  int q = 0;
  for (int a = 0; a < nE; ++a)
    for (int b = a; b < nE; ++b, ++q) {
      const double v = P.hEEinv[i + (int64_t)q * P.n];
      Hi[a * nE + b] = v;
      Hi[b * nE + a] = v;
    }
  for (int ev = 0; ev < nE; ++ev) {
    double s = 0.0;
    for (int ew = 0; ew < nE; ++ew) s += Hi[ev * nE + ew] * gE[ew];
    tE[ev] = s;
  }
  for (int a = 0; a < P.nK; ++a) {
    double s = 0.0;
    for (int ev = 0; ev < nE; ++ev) s += P.hKE[i + (int64_t)(a * nE + ev) * P.n] * tE[ev];
    Gt[i + (int64_t)P.Krow[a] * P.n] = -s;
  }
}

// xE = hEEinv (gE - hEK * DnK):  x[Eoff[ev] + i]; DnK = rows Krow of D applied to the broken vector nb
__global__ void __launch_bounds__(256) k_backsubst(CondParams P, NodeParams NP, const double *__restrict__ g, double *x) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  double y[MGBX_MAX_ND];
  node_Dz(NP, i, y);   // NP.zf = broken image of the kept part of the direction
  const int nE = P.nE;
  double rE[4], Hi[16];
  for (int ev = 0; ev < nE; ++ev) {
    double s = g[P.Eoff[ev] + i];
    for (int a = 0; a < P.nK; ++a) s -= P.hKE[i + (int64_t)(a * nE + ev) * P.n] * y[P.Krow[a]];
    rE[ev] = s;
  }
  int q = 0;
  for (int a = 0; a < nE; ++a)
    for (int b = a; b < nE; ++b, ++q) {
      const double v = P.hEEinv[i + (int64_t)q * P.n];
      Hi[a * nE + b] = v;
      Hi[b * nE + a] = v;
    }
  for (int ev = 0; ev < nE; ++ev) {
    double s = 0.0;
    for (int ew = 0; ew < nE; ++ew) s += Hi[ev * nE + ew] * rE[ew];
    x[P.Eoff[ev] + i] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// vector kernels (all scalars stay on the device)
// ------------------------------------------------------------------------------------------------
// out[0] = a.b, out[1] = a.a, out[2] = #non-finite entries of a
__global__ void __launch_bounds__(kRedThreads) k_dot2(int64_t m, const double *__restrict__ a, const double *__restrict__ b,
                                                       double *partials, unsigned int *ticket, double *out) {
  double red[3] = {0.0, 0.0, 0.0};
  const int op[3] = {0, 0, 0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double x = a[i];
    red[0] += x * (b ? b[i] : 0.0);
    red[1] += x * x;
    if (!isfinite(x)) red[2] += 1.0;
  }
  grid_reduce<3>(red, op, partials, ticket, out);
}

// xn = x - s*d;  out[0] = |xn - x|^2 (exactly as evaluated in floating point: stall detection, src/newton.jl:141)
__global__ void __launch_bounds__(kRedThreads) k_trial(int64_t m, const double *__restrict__ x, const double *__restrict__ d, double s,
                                                        double *xn, double *partials, unsigned int *ticket, double *out) {
  double red[1] = {0.0};
  const int op[1] = {0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double xi = x[i];
    const double v = xi - s * d[i];
    xn[i] = v;
    const double df = v - xi;
    red[0] += df * df;
  }
  grid_reduce<1>(red, op, partials, ticket, out);
}

__global__ void k_axpby(int64_t m, double a, const double *__restrict__ x, double b, const double *__restrict__ y, double *out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) out[i] = a * x[i] + (y ? b * y[i] : 0.0);
}

// start vector of the power iteration on D^-1 A (pcg2_lambda_power: a sharper lambda_max for the Chebyshev interval than the
// Gershgorin bound): smooth + oscillatory parts, never orthogonal to the top eigenvector in practice
__global__ void k_pw_init(int64_t m, double *v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) v[i] = 1.0 + 0.5 * cos(0.7 * (double)i) + ((i & 1) ? 0.25 : -0.25);
}

// per-variable max and max|.| of the state: out[2k] = max, out[2k+1] = absmax  (one launch per variable)
__global__ void __launch_bounds__(kRedThreads) k_maxabs(int64_t m, const double *__restrict__ a, double *partials, unsigned int *ticket,
                                                         double *out) {
  double red[3] = {-INFINITY, -INFINITY, 0.0};
  const int op[3] = {1, 1, 0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = a[i];
    red[0] = fmax(red[0], v);
    red[1] = fmax(red[1], fabs(v));
    if (!isfinite(v)) red[2] += 1.0;
  }
  grid_reduce<3>(red, op, partials, ticket, out);
}

// sl[i] = 2*max(slack[i], 1)   (src/mgb.jl:437-440)
__global__ void k_phase1_slack(int64_t n, const double *slack, double *out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = 2.0 * fmax(slack[i], 1.0);
}

// ------------------------------------------------------------------------------------------------
// dense helpers (the blocked DMMA Cholesky lives in dense_kernels.cuh)
// ------------------------------------------------------------------------------------------------
// Ad = 0 then Ad[i][j] = a_ij * d_i * d_j  with d = 1/sqrt(a_ii)
__global__ void k_dense_scale_diag(DevCsr A, double *d) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= A.rows) return;
  double dg = 0.0;
  for (int64_t k = A.ptr[row]; k < A.ptr[row + 1]; ++k)
    if (A.idx[k] == row) dg = A.val[k];
  d[row] = dg > 0.0 ? 1.0 / sqrt(dg) : 1.0;
}
__global__ void k_csr_to_dense(DevCsr A, const double *d, double *Ad) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= A.rows) return;
  const double di = d[row];
  for (int64_t k = A.ptr[row]; k < A.ptr[row + 1]; ++k) Ad[row * A.rows + A.idx[k]] = A.val[k] * di * d[A.idx[k]];
}

// y = M x for a dense symmetric m x m matrix stored as m columns (coarse inverse); one warp per row
__global__ void __launch_bounds__(256) k_dense_symv(const double *__restrict__ M, int m, const double *__restrict__ x, double *y) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= m) return;
  const double *r = M + (size_t)row * m;
  double s = 0.0;
  for (int j = lane; j < m; j += 32) s += r[j] * x[j];
  s = warp_sum(s);
  if (lane == 0) y[row] = s;
}


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

// out[0..2] = {a.b, a.a, #non-finite entries of a} over the LOCAL segments, out[3..5] the same over the SHARED ones
__global__ void __launch_bounds__(kRedThreads) k_dot2_seg(SegList S, int64_t m, const double *__restrict__ a, const double *__restrict__ b,
                                                           double *partials, unsigned int *ticket, double *out) {
  double red[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  const int op[6] = {0, 0, 0, 0, 0, 0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double x = a[i];
    const int o = seg_is_local(S, i) ? 0 : 3;
    red[o] += x * (b ? b[i] : 0.0);
    red[o + 1] += x * x;
    if (!isfinite(x)) red[o + 2] += 1.0;
  }
  grid_reduce<6>(red, op, partials, ticket, out);
}

// xn = x - s*d;  out[0] = |xn - x|^2 over the SHARED segments, out[1] over the LOCAL ones
__global__ void __launch_bounds__(kRedThreads) k_trial_seg(SegList S, int64_t m, const double *__restrict__ x, const double *__restrict__ d,
                                                            double s, double *xn, double *partials, unsigned int *ticket, double *out) {
  double red[2] = {0.0, 0.0};
  const int op[2] = {0, 0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double xi = x[i];
    const double v = xi - s * d[i];
    xn[i] = v;
    const double df = v - xi;
    red[seg_is_local(S, i) ? 1 : 0] += df * df;
  }
  grid_reduce<2>(red, op, partials, ticket, out);
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

template <int MODE, int NDT>
__global__ void __launch_bounds__(256) k_elem(ElemFused Q) {
  extern __shared__ double esm[];
  const NodeParams &P = Q.np;
  const int p = P.p, pp = p * p, p1 = Q.p1, ES = Q.ES, epb = Q.epb;
  const int TM = epb * p;                       // node slots per tile
  double *ops_s = esm;                          // [op][el][c][r] padded
  double *zs = ops_s + (size_t)Q.nops * epb * ES;   // [var][slot]
  double *ex = zs + (size_t)P.nu * TM;          // [row][slot]
  const int tid = threadIdx.x;
  double red[4] = {0.0, 0.0, 0.0, -INFINITY};
  const int op4[4] = {0, 0, 0, 1};
  const int64_t ntiles = (Q.N + epb - 1) / epb;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t e0 = tile * epb;
    const int ne = (int)min((int64_t)epb, Q.N - e0);
    const int T = ne * p;
    const int64_t node0 = e0 * p;
    __syncthreads();   // previous tile fully consumed
    for (int o = 0; o < Q.nops; ++o) {
      const double *src = P.ops[o] + e0 * (int64_t)pp;
      double *dst = ops_s + (size_t)o * epb * ES;
      for (int t = tid; t < ne * pp; t += blockDim.x) {
        const int el = t / pp, rem = t - el * pp;
        const int c = rem / p, r = rem - c * p;
        dst[el * ES + c * p1 + r] = src[t];
      }
    }
    for (int v = 0; v < P.nu; ++v)
      for (int t = tid; t < T; t += blockDim.x) zs[v * TM + t] = P.zf[(int64_t)v * P.n + node0 + t];
    __syncthreads();
    const int el = tid / p, q = tid - el * p;
    const bool on = tid < T;
    const int64_t i = node0 + tid;
    if (on) {
      double y[NDT];
      for (int j = 0; j < P.nD; ++j) {
        const int v = P.D_var[j], o = P.D_op[j];
        if (o < 0) y[j] = zs[v * TM + tid];
        else {
          const double *blk = ops_s + (size_t)o * epb * ES + el * ES + q;
          const double *ze = zs + v * TM + el * p;
          double acc = 0.0;
          for (int c = 0; c < p; ++c) acc += blk[c * p1] * ze[c];
          y[j] = acc;
        }
      }
      const int nD = P.nD;
      const double bwi = P.bw ? P.bw[i] : 1.0;
      const bool active = !(P.bw && bwi == 0.0);
      const double sc = P.bw ? bwi : P.inv_n;
      double F1[NDT];
      if (MODE == NODE_F01) {
        double F0 = 0.0;
        if (active) F0 = node_eval(P.cd, P.n, i, y, 1, F1, nullptr);
        else
          for (int j = 0; j < nD; ++j) F1[j] = 0.0;
        const double wi = P.w[i];
        double lin = 0.0;
        for (int j = 0; j < nD; ++j) {
          const double c = P.t * P.f[i + (int64_t)j * P.n];
          lin += c * y[j];
          ex[j * TM + tid] = (active ? sc * F1[j] : 0.0) + wi * c;
        }
        red[0] += active ? (P.bw ? bwi * F0 : F0) : 0.0;
        red[1] += wi * lin;
        if (!isfinite(F0)) red[2] += 1.0;
      } else {
        double F2[NDT * NDT];
        if (active) {
          node_eval(P.cd, P.n, i, y, 2, F1, F2, nE_mask_guard(P));
          for (int k = 0; k < nD * nD; ++k) F2[k] *= sc;
        } else {
          for (int k = 0; k < nD * nD; ++k) F2[k] = 0.0;
        }
        const int nK = P.nK, nE = P.nE;
        if (nE == 0) {
          int qq = 0;
          for (int a = 0; a < nK; ++a)
            for (int b = a; b < nK; ++b, ++qq) ex[qq * TM + tid] = F2[P.Krow[a] * nD + P.Krow[b]];
        } else {
          double hEE[16], hKE[NDT * 4];
          for (int k = 0; k < nE * nE; ++k) hEE[k] = 0.0;
          for (int k = 0; k < nK * nE; ++k) hKE[k] = 0.0;
          for (int j = 0; j < nD; ++j) {
            const int ej = P.Erow[j];
            if (ej < 0) continue;
            for (int k = 0; k < nD; ++k) {
              const int ek = P.Erow[k];
              if (ek >= 0) hEE[ej * nE + ek] += F2[j * nD + k];
            }
            for (int a = 0; a < nK; ++a) hKE[a * nE + ej] += F2[P.Krow[a] * nD + j];
          }
          spd_inverse(hEE, nE);
          {
            int qq = 0;
            for (int a = 0; a < nE; ++a)
              for (int b = a; b < nE; ++b, ++qq) P.hEEinv[i + (int64_t)qq * P.n] = hEE[a * nE + b];
          }
          for (int k = 0; k < nK * nE; ++k) P.hKE[i + (int64_t)k * P.n] = hKE[k];
          int qq = 0;
          for (int a = 0; a < nK; ++a)
            for (int b = a; b < nK; ++b, ++qq) {
              double s = F2[P.Krow[a] * nD + P.Krow[b]];
              for (int ev = 0; ev < nE; ++ev) {
                if ((P.schur_elim >> ev) & 1u) continue;   // already condensed analytically inside node_eval
                double wv = 0.0;
                for (int ew = 0; ew < nE; ++ew) wv += hEE[ev * nE + ew] * hKE[b * nE + ew];
                s -= hKE[a * nE + ev] * wv;
              }
              ex[qq * TM + tid] = s;
            }
        }
      }
    }
    __syncthreads();
    if (MODE == NODE_F01) {
      // gb[v][node0 + (el, c)] = sum_{j in rows(v)} sum_q D_j[q][c] G_j[q]
      if (on) {
        const int c = q;
        for (int v = 0; v < P.nu; ++v) {
          double acc = 0.0;
          for (int j = 0; j < P.nD; ++j) {
            if (P.D_var[j] != v) continue;
            const int o = P.D_op[j];
            const double *g = ex + j * TM + el * p;
            if (o < 0) acc += g[c];
            else {
              const double *blk = ops_s + (size_t)o * epb * ES + el * ES + c * p1;
              for (int k = 0; k < p; ++k) acc += blk[k] * g[k];
            }
          }
          Q.gb[(int64_t)v * P.n + i] = acc;
        }
      }
    } else {
      // Hblk[((pair*N + e)*p + r)*p + c] = sum_{ja in rows(va), kb in rows(vb)} sum_q D_ja[q][r] h[q] D_kb[q][c]
      const int nK = P.nK;
      const int per = ne * pp;
      for (int pr = 0; pr < Q.pl.npairs; ++pr) {
        const int va = Q.pl.va[pr], vb = Q.pl.vb[pr];
        double *out = Q.Hblk + ((int64_t)pr * Q.N + e0) * pp;
        for (int t = tid; t < per; t += blockDim.x) {
          const int e2 = t / pp, rem = t - e2 * pp;
          const int r = rem / p, c = rem - r * p;
          double acc = 0.0;
          for (int ja = 0; ja < nK; ++ja) {
            const int j = P.Krow[ja];
            if (P.D_var[j] != va) continue;
            const int oj = P.D_op[j];
            for (int kb = 0; kb < nK; ++kb) {
              const int k = P.Krow[kb];
              if (P.D_var[k] != vb) continue;
              const int ok = P.D_op[k];
              const int a = ja < kb ? ja : kb, b = ja < kb ? kb : ja;
              const double *h = ex + (a * nK - (a * (a - 1)) / 2 + (b - a)) * TM + e2 * p;
              if (oj < 0 && ok < 0) {
                if (r == c) acc += h[r];
              } else if (oj < 0) {
                acc += h[r] * ops_s[(size_t)ok * epb * ES + e2 * ES + c * p1 + r];
              } else if (ok < 0) {
                acc += ops_s[(size_t)oj * epb * ES + e2 * ES + r * p1 + c] * h[c];
              } else {
                const double *dj = ops_s + (size_t)oj * epb * ES + e2 * ES + r * p1;
                const double *dk = ops_s + (size_t)ok * epb * ES + e2 * ES + c * p1;
                double s = 0.0;
                for (int k2 = 0; k2 < p; ++k2) s += dj[k2] * h[k2] * dk[k2];
                acc += s;
              }
            }
          }
          out[t] = acc;
        }
      }
    }
  }
  if (MODE == NODE_F01) grid_reduce<4>(red, op4, P.partials, P.ticket, P.red_out);
}

}  // namespace mgbx

namespace mgbx {

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

// Tiles are software-pipelined: while tile k is evaluated, the operator blocks and node inputs of tile k+1 stream into the
// other shared-memory buffer with cp.async (LDGSTS), so the evaluation never waits on HBM latency after the first tile.
// COND: the slack is condensed node-locally (fine-level systems); !COND: nothing is eliminated and the four block pairs
// (u,u), (u,s), (s,u), (s,s) are written (the coarse-level systems of the mgb_step recovery path).
template <int MODE, int DIM, bool COND>
__global__ void __launch_bounds__(256, 3) k_elem_plap(PlapParams P) {
  extern __shared__ __align__(16) double esm[];
  constexpr int NH = (DIM * (DIM + 1)) / 2;
  constexpr int NEX = NH > DIM ? NH : DIM;
  constexpr int NF = DIM + 2;
  const int p = P.p, pp = p * p, p1 = P.p1, ES = P.ES, epb = P.epb;
  const int TM = epb * p;
  const size_t bufsz = (size_t)DIM * epb * ES + (size_t)(4 + NF) * TM;
  double *ex = esm + 2 * bufsz;                    // [row][slot]: F01 DIM rows, F2 NH rows
  (void)NEX;
  const int tid = threadIdx.x;
  double red[4] = {0.0, 0.0, 0.0, -INFINITY};
  const int op4[4] = {0, 0, 0, 1};
  const int64_t ntiles = (P.N + epb - 1) / epb;
  const double al = 2.0 / P.pexp;
  // completion barriers of the two input buffers (bulk staging); a tile arms its buffer's barrier with the bytes it will receive
  __shared__ __align__(8) unsigned long long mbar[2];
  unsigned int mphase = 0u;   // bit b: parity of buffer b's next completion
  if (P.bulk) {
    if (tid == 0) {
      mbar_init(&mbar[0], 1);
      mbar_init(&mbar[1], 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
  }
  // buffer layout: ops [a][el][c][r] padded | us | ss | ws | bws | fs[NF]
  auto issue = [&](int64_t tile, int b) {
    double *buf = esm + (size_t)b * bufsz;
    const int64_t e0 = tile * epb;
    const int ne = (int)min((int64_t)epb, P.N - e0);
    const int T = ne * p;
    const int64_t node0 = e0 * p;
    if (P.bulk) {
      // whole slabs move with one instruction each (UBLKCP); a ragged last tile (odd sizes break the 16-byte rule) falls through
      // to the per-double path below and arms the barrier with zero bytes
      const bool regular = ((ne & 1) == 0 || (p & 1) == 0) && ((T & 1) == 0);
      if (regular) {
        double *nd = buf + (size_t)DIM * epb * ES;
        const int narr = 3 + (P.bw ? 1 : 0) + NF;
        const unsigned int opbytes = (unsigned int)(ne * pp * 8), ndbytes = (unsigned int)(T * 8);
        if (tid == 0) {
          fence_proxy_async_smem();
          mbar_expect_tx(&mbar[b], DIM * opbytes + narr * ndbytes);
        }
        __syncwarp();
        if (P.bulk == 1) {
          if (tid < DIM) bulk_g2s(buf + (size_t)tid * epb * ES, P.ops[tid] + e0 * (int64_t)pp, opbytes, &mbar[b]);
        } else {
          for (int t = tid; t < DIM * ne * p; t += 256) {   // one block column (p doubles) per copy into the padded layout
            const int a = t / (ne * p), rem = t - a * ne * p;
            const int el = (int)fdiv((unsigned int)rem, P.dp), c = rem - el * p;
            bulk_g2s(buf + (size_t)a * epb * ES + el * ES + c * p1, P.ops[a] + (e0 + el) * (int64_t)pp + c * p, (unsigned int)(p * 8), &mbar[b]);
          }
        }
        if (tid >= 32 && tid < 32 + narr) {
          const int k = tid - 32;
          const double *src;
          double *dst;
          if (k == 0) { src = P.zu; dst = nd; }
          else if (k == 1) { src = P.zs; dst = nd + TM; }
          else if (k == 2) { src = P.w; dst = nd + 2 * TM; }
          else if (P.bw && k == 3) { src = P.bw; dst = nd + 3 * TM; }
          else {
            const int j = k - 3 - (P.bw ? 1 : 0);
            src = P.f + (int64_t)j * P.n;
            dst = nd + (4 + j) * TM;
          }
          bulk_g2s(dst, src + node0, ndbytes, &mbar[b]);
        }
        cp_async_commit();   // (empty group: keeps the wait_group bookkeeping of the ragged path uniform)
        return;
      }
      if (tid == 0) mbar_expect_tx(&mbar[b], 0);
    }
#pragma unroll
    for (int a = 0; a < DIM; ++a) {
      const double *src = P.ops[a] + e0 * (int64_t)pp;
      double *dst = buf + (size_t)a * epb * ES;
      for (int t = tid; t < ne * pp; t += 256) {
        const int el = (int)fdiv((unsigned int)t, P.dpp), rem = t - el * pp;
        const int c = (int)fdiv((unsigned int)rem, P.dp), r = rem - c * p;
        cp_async8(dst + el * ES + c * p1 + r, src + t);
      }
    }
    double *nd = buf + (size_t)DIM * epb * ES;
    if (tid < T) {
      const int64_t i = node0 + tid;
      cp_async8(nd + tid, P.zu + i);
      cp_async8(nd + TM + tid, P.zs + i);
      cp_async8(nd + 2 * TM + tid, P.w + i);
      if (P.bw) cp_async8(nd + 3 * TM + tid, P.bw + i);
#pragma unroll
      for (int j = 0; j < NF; ++j) cp_async8(nd + (4 + j) * TM + tid, P.f + i + (int64_t)j * P.n);
    }
    cp_async_commit();
  };
  int b = 0;
  if ((int64_t)blockIdx.x < ntiles) issue(blockIdx.x, 0);
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t next = tile + gridDim.x;
    if (next < ntiles) {
      issue(next, b ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    if (P.bulk) {
      mbar_wait(&mbar[b], (mphase >> b) & 1u);
      mphase ^= 1u << b;
    }
    __syncthreads();
    const double *ops_s = esm + (size_t)b * bufsz;
    const double *us = ops_s + (size_t)DIM * epb * ES;
    const double *ss = us + TM, *ws = us + 2 * TM, *bws = us + 3 * TM, *fs = us + 4 * TM;
    const int64_t e0 = tile * epb;
    const int ne = (int)min((int64_t)epb, P.N - e0);
    const int T = ne * p;
    const int64_t node0 = e0 * p;
    const int el = (int)fdiv((unsigned int)tid, P.dp), qn = tid - el * p;
    const bool on = tid < T;
    const int64_t i = node0 + tid;
    double G0 = 0.0, Gs = 0.0;
    if (on) {
      double q[DIM];
      const double *ue = us + el * p;
#pragma unroll
      for (int a = 0; a < DIM; ++a) {
        const double *blk = ops_s + (size_t)a * epb * ES + el * ES + qn;
        double acc = 0.0;
        for (int c = 0; c < p; ++c) acc += blk[c * p1] * ue[c];
        q[a] = acc;
      }
      const double uu = ue[qn];
      const double s = ss[tid];
      const double bwi = P.bw ? bws[tid] : 1.0;
      const bool active = !(P.bw && bwi == 0.0);
      const double sc = P.bw ? bwi : P.inv_n;
      const double wi = ws[tid];
      double qsq = 0.0;
#pragma unroll
      for (int a = 0; a < DIM; ++a) qsq += q[a] * q[a];
      const double ls = Log(s);
      const double sa = exp(al * ls);
      const double r = sa - qsq;
      const bool in = s > 0.0;
      const double inv_r = 1.0 / r;
      const double sam1 = in ? sa / s : safe_pow(s, al - 1.0);
      if (MODE == NODE_F01) {
        const double F0 = active ? (-Log(r) - P.mu * ls) : 0.0;
        const double c0 = P.t * fs[tid];
        const double cs = P.t * fs[(DIM + 1) * TM + tid];
        double lin = c0 * uu + cs * s;
        G0 = wi * c0;
        const double gs = -al * sam1 * inv_r - P.mu / s;
        Gs = (active ? sc * gs : 0.0) + wi * cs;
#pragma unroll
        for (int a = 0; a < DIM; ++a) {
          const double ca = P.t * fs[(a + 1) * TM + tid];
          lin += ca * q[a];
          ex[a * TM + tid] = (active ? sc * 2.0 * inv_r * q[a] : 0.0) + wi * ca;
        }
        red[0] += active ? (P.bw ? bwi * F0 : F0) : 0.0;
        red[1] += wi * lin;
        if (!isfinite(F0)) red[2] += 1.0;
      } else {
        if (active) {
          const double inv_r2 = inv_r * inv_r;
          const double coef = -2.0 * al * sam1 * inv_r2;
          const double sam2 = in ? sam1 / s : safe_pow(s, al - 2.0);
          const double s2am2 = in ? sam1 * sam1 : safe_pow(s, 2.0 * al - 2.0);
          // H_ss = A + B with A = (al s^(al-1) / r)^2 (the square of the coupling) and B the rest.  The node-local Schur
          // complement of the slack is  H_qq - H_qs H_sq / H_ss = (2/r) I + (4/r^2) (B / (A + B)) q q':  formed this way, not by
          // subtracting two terms of size 4 q q'/r^2 ~ t^2 whose difference is O(t) across q and O(1) along q -- at t ~ 1e8 the
          // subtraction leaves NO correct digit along q (absolute error eps t^2 ~ 1) and the reduced matrix turns indefinite.
          const double hA = al * al * s2am2 * inv_r2, hB = -al * (al - 1.0) * sam2 * inv_r + P.mu / (s * s);
          const double hss = sc * (hA + hB);
          const double ihs = COND ? 1.0 / hss : 0.0;
          const double schur = hB / (hA + hB);
          double hqs[DIM];
#pragma unroll
          for (int a = 0; a < DIM; ++a) hqs[a] = sc * coef * q[a];
          if (COND) {
            P.hEEinv[i] = ihs;
            P.hKE[i] = 0.0;
#pragma unroll
            for (int a = 0; a < DIM; ++a) P.hKE[i + (int64_t)(a + 1) * P.n] = hqs[a];
          } else {
#pragma unroll
            for (int a = 0; a < DIM; ++a) ex[(NH + a) * TM + tid] = hqs[a];
            ex[(NH + DIM) * TM + tid] = hss;
          }
          int k = 0;
#pragma unroll
          for (int a = 0; a < DIM; ++a)
#pragma unroll
            for (int bb = a; bb < DIM; ++bb, ++k) {
              const double qq4 = 4.0 * q[a] * q[bb] * inv_r2, dg = (a == bb ? 2.0 * inv_r : 0.0);
              ex[k * TM + tid] = COND ? sc * (qq4 * schur + dg) : sc * (qq4 + dg);
            }
        } else {
          if (COND) {
            P.hEEinv[i] = 0.0;
#pragma unroll
            for (int a = 0; a <= DIM; ++a) P.hKE[i + (int64_t)a * P.n] = 0.0;
          }
#pragma unroll
          for (int k = 0; k < (COND ? NH : NH + DIM + 1); ++k) ex[k * TM + tid] = 0.0;
        }
      }
    }
    __syncthreads();
    if (MODE == NODE_F01) {
      if (on) {
        double acc = G0;
#pragma unroll
        for (int a = 0; a < DIM; ++a) {
          const double *blk = ops_s + (size_t)a * epb * ES + el * ES + qn * p1;
          const double *g = ex + a * TM + el * p;
          for (int k = 0; k < p; ++k) acc += blk[k] * g[k];
        }
        P.gbu[i] = acc;
        P.gbs[i] = Gs;
      }
    } else {
      double *out = P.Hblk + e0 * (int64_t)pp;
      for (int t = tid; t < ne * pp; t += 256) {
        const int e2 = (int)fdiv((unsigned int)t, P.dpp), rem = t - e2 * pp;
        const int r = (int)fdiv((unsigned int)rem, P.dp), c = rem - r * p;
        const double *h = ex + e2 * p;
        const double *base = ops_s + e2 * ES;
        double acc = 0.0;
        for (int k = 0; k < p; ++k) {
          double dr[DIM], dc[DIM];
#pragma unroll
          for (int a = 0; a < DIM; ++a) {
            dr[a] = base[(size_t)a * epb * ES + r * p1 + k];
            dc[a] = base[(size_t)a * epb * ES + c * p1 + k];
          }
          int kk = 0;
#pragma unroll
          for (int a = 0; a < DIM; ++a)
#pragma unroll
            for (int bb = a; bb < DIM; ++bb, ++kk) {
              const double hv = h[kk * TM + k];
              acc += (a == bb) ? dr[a] * hv * dc[a] : hv * (dr[a] * dc[bb] + dr[bb] * dc[a]);
            }
        }
        out[t] = acc;
        if (!COND) {
          // (u,s): sum_a D_a[c][r] h_as[c];  (s,u): its transpose;  (s,s): diag(h_ss)
          double us_ = 0.0, su_ = 0.0;
#pragma unroll
          for (int a = 0; a < DIM; ++a) {
            us_ += base[(size_t)a * epb * ES + r * p1 + c] * h[(NH + a) * TM + c];
            su_ += h[(NH + a) * TM + r] * base[(size_t)a * epb * ES + c * p1 + r];
          }
          const int64_t pstride = P.N * (int64_t)pp;
          out[pstride + t] = us_;
          out[2 * pstride + t] = su_;
          out[3 * pstride + t] = (r == c) ? h[(NH + DIM) * TM + r] : 0.0;
        }
      }
    }
    __syncthreads();   // the exchange rows and (two tiles later) this input buffer are reused
    b ^= 1;
  }
  if (MODE == NODE_F01) grid_reduce<4>(red, op4, P.partials, P.ticket, P.red_out);
}

}  // namespace mgbx
