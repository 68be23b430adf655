// solver_kernels.cuh -- kernels of the linear solve around k_pcg2 (compiled by linear_solve.cu only): smoother
// diagonals, FP32 copies and the power-iteration start of the preconditioner levels, the node-local condensation of the
// right-hand side and its back-substitution, the coarse dense inverse, and the direct solves.
// The Newton-system solve itself is k_pcg2 (pcg2.hpp / pcg2.cu).
//
// What this replaces in the reference (paths under /root/reference):
//   k_coarse_inverse     dense Cholesky + explicit inverse of the coarsest level in shared memory (one CTA).
//   k_dense_solve_small  solve(Symmetric(H), g) (src/utils.jl:142-145) of a small system in one CTA.
//   k_chol_*             the same for up to 8192 unknowns: blocked Cholesky (panel width 64, the panel solve and the
//                        trailing update are k_dgemm_nt DMMA GEMMs) and the triangular solves.
#pragma once

#include "device_common.cuh"

namespace mgbx {

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

// Element-local eliminated variable (elem_schur.cuh), one thread per element:
// Gt[Krow[a]*n + i] = - q_{a,i} (P_e y)_i,  y = H_ss,e^-1 g_c,e  (so that rhs_u = g_u - R_u' H_us H_ss^-1 g_c after k_blockgrad)
__global__ void __launch_bounds__(256) k_condense_rhs_elem(CondParams P, ElemLocal EL, int64_t N, int p, const double *__restrict__ g, double *Gt) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  const int nc = EL.nc;
  double y[kElemMaxNc];
  const double *gc = g + P.Eoff[0] + EL.c0[e];
  for (int k = 0; k < nc; ++k) y[k] = gc[k];
  elem_hss_solve(nc, EL.R + e * elem_rsize(nc), y);
  for (int r = 0; r < p; ++r) {
    const int64_t i = e * p + r;
    double v = 0.0;
    for (int k = 0; k < nc; ++k) v += EL.P[i * nc + k] * y[k];
    for (int a = 0; a < P.nK; ++a) Gt[i + (int64_t)P.Krow[a] * P.n] = -P.hKE[i + (int64_t)a * P.n] * v;
  }
}

// dc_e = H_ss,e^-1 (g_c,e - P_e' sum_a q_a (D_a du)):  x[Eoff[0] + c0[e] + k]
__global__ void __launch_bounds__(256) k_backsubst_elem(CondParams P, ElemLocal EL, NodeParams NP, int64_t N, const double *__restrict__ g, double *x) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  const int nc = EL.nc, p = NP.p;
  double rc[kElemMaxNc];
  const int64_t col = P.Eoff[0] + EL.c0[e];
  for (int k = 0; k < nc; ++k) rc[k] = g[col + k];
  for (int r = 0; r < p; ++r) {
    const int64_t i = e * p + r;
    double y[MGBX_MAX_ND];
    node_Dz(NP, i, y);   // NP.zf = broken image of the kept part of the direction
    double s = 0.0;
    for (int a = 0; a < P.nK; ++a) s += P.hKE[i + (int64_t)a * P.n] * y[P.Krow[a]];
    for (int k = 0; k < nc; ++k) rc[k] -= EL.P[i * nc + k] * s;
  }
  elem_hss_solve(nc, EL.R + e * elem_rsize(nc), rc);
  for (int k = 0; k < nc; ++k) x[col + k] = rc[k];
}

// start vector of the power iteration on D^-1 A (pcg2_lambda_power: a sharper lambda_max for the Chebyshev interval than the
// Gershgorin bound): smooth + oscillatory parts, never orthogonal to the top eigenvector in practice
__global__ void k_pw_init(int64_t m, double *v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) v[i] = 1.0 + 0.5 * cos(0.7 * (double)i) + ((i & 1) ? 0.25 : -0.25);
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

__global__ void k_f64_to_f32(int64_t n, const double *__restrict__ a, float *__restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (float)a[i];
}

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
  // right-looking Cholesky on the lower triangle.  A non-positive pivot means numerical indefiniteness: keep the
  // preconditioner finite and SPD (any SPD approximation is a valid preconditioner) by decoupling unknown j -- unit pivot,
  // zero column below it, so no trailing update.  (A tiny pivot instead divides the column by it, grows the trailing
  // matrix by its inverse square, and overflows after a few such pivots.)  Positive pivots are used as they are.
  __shared__ int drop;
  for (int j = 0; j < m; ++j) {
    if (tid == 0) {
      const double v = S[j * ld + j];
      drop = !(v > 0.0 && isfinite(v));
      S[j * ld + j] = drop ? 1.0 : sqrt(v);
    }
    __syncthreads();
    const double piv = S[j * ld + j];
    for (int i = j + 1 + tid; i < m; i += nt) S[i * ld + j] = drop ? 0.0 : S[i * ld + j] / piv;
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

// factor the nb x nb diagonal block at (k0, k0) in shared memory, write L11 back and inv(L11) (row-major, ld 64) to Linv
__global__ void __launch_bounds__(1024) k_chol_diag_inv(double *A, int m, int k0, double *Linv) {
  extern __shared__ double chol_sm[];   // 2 x 64 x 65 doubles (dynamic: above the 48 KB static limit)
  double (*L)[kCholNB + 1] = reinterpret_cast<double (*)[kCholNB + 1]>(chol_sm);
  double (*Li)[kCholNB + 1] = reinterpret_cast<double (*)[kCholNB + 1]>(chol_sm + kCholNB * (kCholNB + 1));
  const int nb = min(kCholNB, m - k0);
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int t = tid; t < kCholNB * kCholNB; t += nt) {
    const int i = t / kCholNB, j = t % kCholNB;
    L[i][j] = (i < nb && j <= i) ? A[(size_t)(k0 + i) * m + k0 + j] : 0.0;
    Li[i][j] = 0.0;
  }
  __syncthreads();
  for (int j = 0; j < nb; ++j) {
    if (tid == 0) L[j][j] = sqrt(L[j][j]);
    __syncthreads();
    const double pv = L[j][j];
    for (int i = j + 1 + tid; i < nb; i += nt) L[i][j] /= pv;
    __syncthreads();
    const int rem = nb - j - 1;
    for (int t = tid; t < rem * rem; t += nt) {
      const int i = j + 1 + t / rem, k = j + 1 + t % rem;
      if (k <= i) L[i][k] -= L[i][j] * L[k][j];
    }
    __syncthreads();
  }
  // inverse of the triangular block, one warp per column
  const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
  for (int c = wid; c < nb; c += nw) {
    if (lane == 0) Li[c][c] = 1.0 / L[c][c];
    __syncwarp();
    for (int i = c + 1; i < nb; ++i) {
      double sacc = 0.0;
      for (int k = c + lane; k < i; k += 32) sacc += L[i][k] * Li[k][c];
      sacc = warp_sum(sacc);
      if (lane == 0) Li[i][c] = -sacc / L[i][i];
      __syncwarp();
    }
  }
  __syncthreads();
  for (int t = tid; t < kCholNB * kCholNB; t += nt) {
    const int i = t / kCholNB, j = t % kCholNB;
    if (i < nb && j <= i) A[(size_t)(k0 + i) * m + k0 + j] = L[i][j];
    Linv[t] = (i < nb && j < nb) ? Li[i][j] : 0.0;
  }
}

// x = (L L')^{-1} (d .* b) .* d for ONE right-hand side with the blocked factor and the panel inverses (Linv: panels x 64 x 64).
// One CTA walks the panels (the dependency is sequential anyway): y_blk = inv(L11) b_blk, then b_rest -= L21 y_blk; and back.
__global__ void __launch_bounds__(1024) k_chol_solve_blocked(const double *__restrict__ A, int m, const double *__restrict__ Linv,
                                                              const double *__restrict__ d, const double *__restrict__ b, double *x) {
  extern __shared__ double v[];   // m
  __shared__ double blk[kCholNB];
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < m; i += nt) v[i] = b[i] * d[i];
  __syncthreads();
  const int npan = (m + kCholNB - 1) / kCholNB;
  for (int pnl = 0; pnl < npan; ++pnl) {
    const int k0 = pnl * kCholNB, nb = min(kCholNB, m - k0);
    const double *Li = Linv + (size_t)pnl * kCholNB * kCholNB;
    if (tid < nb) {
      double sacc = 0.0;
      for (int j = 0; j <= tid; ++j) sacc += Li[tid * kCholNB + j] * v[k0 + j];
      blk[tid] = sacc;
    }
    __syncthreads();
    if (tid < nb) v[k0 + tid] = blk[tid];
    for (int i = k0 + nb + tid; i < m; i += nt) {
      const double *row = A + (size_t)i * m + k0;
      double sacc = 0.0;
      for (int j = 0; j < nb; ++j) sacc += row[j] * blk[j];
      v[i] -= sacc;
    }
    __syncthreads();
  }
  for (int pnl = npan - 1; pnl >= 0; --pnl) {
    const int k0 = pnl * kCholNB, nb = min(kCholNB, m - k0);
    const double *Li = Linv + (size_t)pnl * kCholNB * kCholNB;
    // y_blk[j] -= sum_{i >= k0+nb} L[i][k0+j] x[i]   (column sums: warp per j, lanes over rows)
    const int lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
    for (int j = wid; j < nb; j += nw) {
      double sacc = 0.0;
      for (int i = k0 + nb + lane; i < m; i += 32) sacc += A[(size_t)i * m + k0 + j] * v[i];
      sacc = warp_sum(sacc);
      if (lane == 0) blk[j] = v[k0 + j] - sacc;
    }
    __syncthreads();
    // x_blk = inv(L11)' y_blk
    if (tid < nb) {
      double sacc = 0.0;
      for (int i = tid; i < nb; ++i) sacc += Li[i * kCholNB + tid] * blk[i];
      v[k0 + tid] = sacc;
    }
    __syncthreads();
  }
  for (int i = tid; i < m; i += nt) x[i] = v[i] * d[i];
}

}  // namespace mgbx
