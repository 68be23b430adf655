// solver_kernels.cuh -- the Galerkin gather plans (sliced-ELL), the coarse dense inverse and the small direct solve.
// The Newton-system solve itself is k_pcg2 (pcg2.hpp / pcg2.cu).
//
// What this replaces in the reference (paths under /root/reference):
//   k_sell_gather        the numeric Galerkin products A_c = T'(A T) (north-star item 3) and the R'HR scatter
//                        of src/BlockMatrices.jl:506-555, as fixed-order gathers over a sliced-ELL term list
//                        (coalesced index/weight streams, deterministic; the reference CUDA ext uses FP64 atomics,
//                        block_ops.jl:229-249).
//   k_prod_plan<0|1>     build those term lists on the device (setup, once per system).
//   k_coarse_inverse     dense Cholesky + explicit inverse of the coarsest level in shared memory (one CTA).
//   k_dense_solve_small  solve(Symmetric(H), g) (src/utils.jl:142-145) of a small system in one CTA.
#pragma once
#include "kernels.cuh"

namespace mgbx {

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

__global__ void __launch_bounds__(256) k_sell_gather(SellPlan P, const double *__restrict__ in, double *__restrict__ out) {
  const int64_t nz = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (nz >= P.nout) return;
  const int64_t off = P.sptr[nz >> 5] + (nz & 31);
  const int c = P.cnt[nz];
  double acc = 0.0;
  if (P.w) {
    for (int k = 0; k < c; ++k) acc += P.w[off + 32 * (int64_t)k] * in[P.src[off + 32 * (int64_t)k]];
  } else {
    for (int k = 0; k < c; ++k) acc += in[P.src[off + 32 * (int64_t)k]];
  }
  out[nz] = acc;
}

__global__ void k_f64_to_f32(int64_t n, const double *__restrict__ a, float *__restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (float)a[i];
}

// row index of every non-zero of a CSR pattern
__global__ void k_csr_rows(DevCsr A, int32_t *rowof) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= A.rows) return;
  for (int64_t k = A.ptr[row]; k < A.ptr[row + 1]; ++k) rowof[k] = (int32_t)row;
}

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

// Term list of C = Lm * Rm into the fixed pattern C.  variable_left: the values of Lm change between
// uses (source = nz of Lm, weight = value of Rm), otherwise the values of Rm change.  One thread per
// non-zero of C walks row i of Lm and looks column c up in the rows of Rm: no atomics, fixed order.
// FILL == 0: cnt[nz] and per-slice width;  FILL == 1: write src / w.
template <int FILL>
__global__ void __launch_bounds__(256) k_prod_plan(DevCsr Lm, DevCsr Rm, DevCsr C, const int32_t *__restrict__ rowof, int variable_left,
                                                    SellPlan P, int32_t *width) {
  const int64_t nz = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int count = 0;
  if (nz < C.nnz) {
    const int64_t i = rowof[nz];
    const int32_t c = C.idx[nz];
    const int64_t off = FILL ? P.sptr[nz >> 5] + (nz & 31) : 0;
    for (int64_t a = Lm.ptr[i]; a < Lm.ptr[i + 1]; ++a) {
      const int64_t b = csr_find(Rm, Lm.idx[a], c);
      if (b < 0) continue;
      if (FILL) {
        P.src[off + 32 * (int64_t)count] = (int32_t)(variable_left ? a : b);
        P.w[off + 32 * (int64_t)count] = variable_left ? Rm.val[b] : Lm.val[a];
      }
      ++count;
    }
    if (!FILL) P.cnt[nz] = count;
  }
  if (!FILL) {
    int wmax = count;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wmax = max(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
    if ((threadIdx.x & 31) == 0 && nz < C.nnz) width[nz >> 5] = wmax;
  }
}

// ------------------------------------------------------------------------------------------------
// coarse dense inverse: Minv = (D A D)^{-1} with D = diag(a_ii)^{-1/2} folded back in, so that
// x = Minv_out * b solves A x = b.  One CTA, everything in shared memory, m <= kCoarseMaxDense.
//   shared layout: S[m][m+1] (scaled matrix -> Cholesky factor L), Li[m(m+1)/2] (packed inverse of L), d[m]
// ------------------------------------------------------------------------------------------------
constexpr int kCoarseMaxDense = 128;
inline size_t coarse_inverse_smem(int m) { return sizeof(double) * ((size_t)m * (m + 1) + (size_t)m * (m + 1) / 2 + m); }

__global__ void __launch_bounds__(1024) k_coarse_inverse(DevCsr A, double *Minv) {
  extern __shared__ double sm[];
  const int m = (int)A.rows;
  const int ld = m + 1;
  double *S = sm;
  double *Li = S + (size_t)m * ld;
  double *d = Li + (size_t)m * (m + 1) / 2;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int t = tid; t < m * ld; t += nt) S[t] = 0.0;
  __syncthreads();
  for (int row = tid; row < m; row += nt) {
    double dg = 0.0;
    for (int64_t k = A.ptr[row]; k < A.ptr[row + 1]; ++k)
      if (A.idx[k] == row) dg = A.val[k];
    d[row] = dg > 0.0 ? 1.0 / sqrt(dg) : 1.0;
  }
  __syncthreads();
  for (int row = tid; row < m; row += nt)
    for (int64_t k = A.ptr[row]; k < A.ptr[row + 1]; ++k) S[row * ld + A.idx[k]] = A.val[k] * d[row] * d[A.idx[k]];
  __syncthreads();
  // right-looking Cholesky on the lower triangle
  for (int j = 0; j < m; ++j) {
    if (tid == 0) {   // a non-positive pivot means numerical indefiniteness: keep the preconditioner finite (any SPD
      const double v = S[j * ld + j];   // approximation is a valid preconditioner); positive pivots are used as they are
      S[j * ld + j] = sqrt((v > 0.0 && isfinite(v)) ? v : 1e-16);
    }
    __syncthreads();
    const double piv = S[j * ld + j];
    for (int i = j + 1 + tid; i < m; i += nt) S[i * ld + j] /= piv;
    __syncthreads();
    const int rem = m - j - 1;
    for (int t = tid; t < rem * rem; t += nt) {
      const int i = j + 1 + t / rem, k = j + 1 + t % rem;
      if (k <= i) S[i * ld + k] -= S[i * ld + j] * S[k * ld + j];
    }
    __syncthreads();
  }
  // Li = L^{-1}, one warp per column c: x_c = 1/L_cc, x_i = -(sum_{k=c}^{i-1} L_ik x_k)/L_ii
  const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  for (int c = wid; c < m; c += nw) {
    if (lane == 0) Li[(size_t)c * (c + 1) / 2 + c] = 1.0 / S[c * ld + c];
    __syncwarp();
    for (int i = c + 1; i < m; ++i) {
      double s = 0.0;
      for (int k = c + lane; k < i; k += 32) s += S[i * ld + k] * Li[(size_t)k * (k + 1) / 2 + c];
      s = warp_sum(s);
      if (lane == 0) Li[(size_t)i * (i + 1) / 2 + c] = -s / S[i * ld + i];
      __syncwarp();
    }
  }
  __syncthreads();
  // Minv[i][j] = d_i d_j sum_{k >= max(i,j)} Li[k][i] Li[k][j]
  for (int t = tid; t < m * m; t += nt) {
    const int i = t / m, j = t % m;
    double s = 0.0;
    for (int k = (i > j ? i : j); k < m; ++k) s += Li[(size_t)k * (k + 1) / 2 + i] * Li[(size_t)k * (k + 1) / 2 + j];
    Minv[t] = s * d[i] * d[j];
  }
}


// ------------------------------------------------------------------------------------------------
// Robust direct solve of a small system (m <= kCoarseMaxDense) in one CTA:  x = A^{-1} b.
// Mirrors the reference's `Symmetric(H) \ g` (src/utils.jl:142-145: Cholesky, falling back to a pivoted
// factorisation when H is numerically indefinite): diagonally scaled Cholesky first; if a pivot is not
// positive, Gaussian elimination with partial pivoting on the same matrix.  info[0] = 0 / 1 says which ran.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_dense_solve_small(DevCsr A, const double *__restrict__ b, double *x, int *info) {
  extern __shared__ double sm[];
  const int m = (int)A.rows;
  const int ld = m + 1;
  double *S = sm;                       // m x (m+1)
  double *rhs = S + (size_t)m * ld;     // m
  double *d = rhs + m;                  // m
  __shared__ int fail, piv;
  const int tid = threadIdx.x, nt = blockDim.x;
  auto load = [&](bool scaled) {
    for (int t = tid; t < m * ld; t += nt) S[t] = 0.0;
    __syncthreads();
    for (int row = tid; row < m; row += nt)
      for (int64_t k = A.ptr[row]; k < A.ptr[row + 1]; ++k)
        S[row * ld + A.idx[k]] = scaled ? A.val[k] * d[row] * d[A.idx[k]] : A.val[k];
    __syncthreads();
  };
  for (int row = tid; row < m; row += nt) {
    double dg = 0.0;
    for (int64_t k = A.ptr[row]; k < A.ptr[row + 1]; ++k)
      if (A.idx[k] == row) dg = A.val[k];
    d[row] = (dg > 0.0 && isfinite(dg)) ? 1.0 / sqrt(dg) : 1.0;
  }
  if (tid == 0) fail = 0;
  __syncthreads();
  load(true);
  for (int j = 0; j < m && !fail; ++j) {
    if (tid == 0) {
      const double v = S[j * ld + j];
      if (!(v > 0.0) || !isfinite(v)) fail = 1;
      else S[j * ld + j] = sqrt(v);
    }
    __syncthreads();
    if (fail) break;
    const double pv = S[j * ld + j];
    for (int i = j + 1 + tid; i < m; i += nt) S[i * ld + j] /= pv;
    __syncthreads();
    const int rem = m - j - 1;
    for (int t = tid; t < rem * rem; t += nt) {
      const int i = j + 1 + t / rem, k = j + 1 + t % rem;
      if (k <= i) S[i * ld + k] -= S[i * ld + j] * S[k * ld + j];
    }
    __syncthreads();
  }
  __syncthreads();
  if (!fail) {
    // L L' y = D b, x = D y  (one warp: the triangular solves are sequential in the row index)
    for (int i = tid; i < m; i += nt) rhs[i] = b[i] * d[i];
    __syncthreads();
    if (tid < 32) {
      for (int k = 0; k < m; ++k) {
        double sacc = 0.0;
        for (int j = tid; j < k; j += 32) sacc += S[k * ld + j] * rhs[j];
        sacc = warp_sum(sacc);
        if (tid == 0) rhs[k] = (rhs[k] - sacc) / S[k * ld + k];
        __syncwarp();
      }
      for (int k = m - 1; k >= 0; --k) {
        if (tid == 0) rhs[k] = rhs[k] / S[k * ld + k];
        __syncwarp();
        const double xk = rhs[k];
        for (int j = tid; j < k; j += 32) rhs[j] -= S[k * ld + j] * xk;
        __syncwarp();
      }
    }
    __syncthreads();
    for (int i = tid; i < m; i += nt) x[i] = rhs[i] * d[i];
    if (tid == 0 && info) info[0] = 0;
    return;
  }
  // pivoted elimination on the unscaled matrix
  load(false);
  for (int i = tid; i < m; i += nt) rhs[i] = b[i];
  __syncthreads();
  for (int k = 0; k < m; ++k) {
    if (tid == 0) {
      int best = k;
      double bv = fabs(S[k * ld + k]);
      for (int i = k + 1; i < m; ++i) {
        const double v = fabs(S[i * ld + k]);
        if (v > bv) {
          bv = v;
          best = i;
        }
      }
      piv = best;
    }
    __syncthreads();
    const int pr = piv;
    if (pr != k) {
      for (int j = tid; j < m; j += nt) {
        const double t = S[k * ld + j];
        S[k * ld + j] = S[pr * ld + j];
        S[pr * ld + j] = t;
      }
      if (tid == 0) {
        const double t = rhs[k];
        rhs[k] = rhs[pr];
        rhs[pr] = t;
      }
    }
    __syncthreads();
    const double pv = S[k * ld + k];
    // multipliers in column k (kept in place), then the trailing update
    for (int i = k + 1 + tid; i < m; i += nt) S[i * ld + k] /= pv;
    __syncthreads();
    const int rem = m - k - 1;
    for (int t = tid; t < rem * rem; t += nt) {
      const int i = k + 1 + t / rem, j = k + 1 + t % rem;
      S[i * ld + j] -= S[i * ld + k] * S[k * ld + j];
    }
    for (int i = k + 1 + tid; i < m; i += nt) rhs[i] -= S[i * ld + k] * rhs[k];
    __syncthreads();
  }
  if (tid < 32) {
    for (int k = m - 1; k >= 0; --k) {
      double sacc = 0.0;
      for (int j = k + 1 + tid; j < m; j += 32) sacc += S[k * ld + j] * rhs[j];
      sacc = warp_sum(sacc);
      if (tid == 0) rhs[k] = (rhs[k] - sacc) / S[k * ld + k];
      __syncwarp();
    }
  }
  __syncthreads();
  for (int i = tid; i < m; i += nt) x[i] = rhs[i];
  if (tid == 0 && info) info[0] = 1;
}
inline size_t dense_solve_small_smem(int m) { return sizeof(double) * ((size_t)m * (m + 1) + 2 * (size_t)m); }

}  // namespace mgbx
