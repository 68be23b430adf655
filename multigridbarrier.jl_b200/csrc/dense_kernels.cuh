// dense_kernels.cuh -- the spectral (dense) assembly path on the FP64 tensor cores (compiled by evaluate.cu only).
//
// For spectral1d / spectral2d the "element" is the whole domain: the derivative operators are dense n x n Chebyshev
// differentiation matrices (src/spectral1d.jl:63-109, src/spectral2d.jl:15-42) and R is a dense basis-evaluation
// matrix, so  H = sum_jk D_j' diag(h_jk) D_k  and  R'HR  (src/convex.jl:181-202, src/BlockMatrices.jl:506-555 with one
// p x p block) are true dense contractions.  They run here as FP64 DMMA GEMMs (mma.sync m8n8k4 f64, the only FP64
// tensor-core path on sm_100a; tcgen05 has no FP64 kind).  One kernel form covers all three products:
//     C[i*ldc + j] (+)= alpha * sum_k A[i*lda + k] * s[k] * B[j*ldb + k]  ("NT": both operands contiguous along k)
//   (1) Hd[r][c]  += sum_q  D_j[q][r] h[q] D_k[q][c]     A = ops_j, B = ops_k (column-major n x n), s = h
//   (2) Wt[j][r]   = sum_c  Rt_b[j][c] Hd[r][c]          A = Rt_b (m_b x n),  B = Hd
//   (3) A_top[i][j] = sum_r Rt_a[i][r] Wt[j][r]          A = Rt_a (m_a x n),  B = Wt, C = a block of the m x m system
#pragma once

#include "device_common.cuh"

namespace mgbx {

// 128 threads = 4 warps in a 2 x 2 arrangement; each warp owns a 32 x 32 sub-tile = 4 x 4 DMMA tiles.
__global__ void __launch_bounds__(128) k_dgemm_nt(int M, int N, int K, const double *__restrict__ A, int64_t lda, const double *__restrict__ B,
                                                   int64_t ldb, const double *__restrict__ s, double *C, int64_t ldc, int accumulate, double alpha) {
  __shared__ double As[kGemmBM][kGemmLd], Bs[kGemmBN][kGemmLd];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp >> 1, wn = warp & 1;
  const int i0 = blockIdx.y * kGemmBM, j0 = blockIdx.x * kGemmBN;
  double acc[4][4][2];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
  const int lr = lane >> 2, lk = lane & 3;
  for (int k0 = 0; k0 < K; k0 += kGemmBK) {
    // stage 64 x 16 of A (scaled by s) and of B: thread t loads rows t/2 (+ 0), k-half t%2 (8 consecutive doubles)
    {
      const int row = tid >> 1, kh = (tid & 1) * 8;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int k = k0 + kh + q;
        const bool kin = k < K;
        const double sv = (kin && s) ? s[k] : 1.0;
        As[row][kh + q] = (kin && i0 + row < M) ? A[(int64_t)(i0 + row) * lda + k] * sv : 0.0;
        Bs[row][kh + q] = (kin && j0 + row < N) ? B[(int64_t)(j0 + row) * ldb + k] : 0.0;
      }
    }
    __syncthreads();
#pragma unroll
    for (int k4 = 0; k4 < kGemmBK; k4 += 4) {
      double af[4], bf[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) af[a] = As[wm * 32 + a * 8 + lr][k4 + lk];
#pragma unroll
      for (int b = 0; b < 4; ++b) bf[b] = Bs[wn * 32 + b * 8 + lr][k4 + lk];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) dmma_m8n8k4(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
    }
    __syncthreads();
  }
  // C fragment: row = lane / 4, cols = 2 * (lane % 4) + {0, 1}
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int i = i0 + wm * 32 + a * 8 + lr;
      const int j = j0 + wn * 32 + b * 8 + 2 * lk;
      if (i < M) {
        double *c = C + (int64_t)i * ldc + j;
        if (j < N) c[0] = (accumulate ? c[0] : 0.0) + alpha * acc[a][b][0];
        if (j + 1 < N) c[1] = (accumulate ? c[1] : 0.0) + alpha * acc[a][b][1];
      }
    }
}

// Hd[r][c] += (ident_j ? delta : D_j[.][r]) ... the three cheap cases of D_j' diag(h) D_k with an identity operand:
//   mode 0: both identities          Hd[r][r] += h[r]
//   mode 1: D_j = I, D_k = Dk        Hd[r][c] += h[r] * Dk[r][c]        (Dk column-major: Dk[c*n + r])
//   mode 2: D_j = Dj, D_k = I        Hd[r][c] += Dj[c][r] * h[c]        (Dj[r*n + c])
__global__ void __launch_bounds__(256) k_dense_hess_ident(int n, int mode, const double *__restrict__ h, const double *__restrict__ D, double *Hd) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (mode == 0) {
    if (t < n) Hd[t * n + t] += h[t];
    return;
  }
  if (t >= (int64_t)n * n) return;
  const int r = (int)(t / n), c = (int)(t % n);
  if (mode == 1) Hd[t] += h[r] * D[(int64_t)c * n + r];
  else Hd[t] += D[(int64_t)r * n + c] * h[c];
}

// W[(i' c2b + l') K + c n1 + e] = sum_f Qj[f, i'] h[e n1 + f] Qk[f, l']     grid: (ncombo * n1) blocks
__global__ void __launch_bounds__(256) k_kron_w(KronWArgs P, double *__restrict__ W) {
  extern __shared__ double kw_sm[];   // h row (n1), Qj scaled by h (n1 x c2a), Qk (n1 x c2b)
  const int c = blockIdx.x / P.n1, e = blockIdx.x % P.n1;
  const KronCombo cb = P.c[c];
  double *hs = kw_sm, *qj = hs + P.n1, *qk = qj + (size_t)P.n1 * P.c2a;
  for (int f = threadIdx.x; f < P.n1; f += blockDim.x) hs[f] = cb.h[(size_t)e * P.n1 + f];
  __syncthreads();
  for (int t = threadIdx.x; t < P.n1 * P.c2a; t += blockDim.x) qj[t] = cb.Qj[t] * hs[t / P.c2a];
  for (int t = threadIdx.x; t < P.n1 * P.c2b; t += blockDim.x) qk[t] = cb.Qk[t];
  __syncthreads();
  const int nout = P.c2a * P.c2b;
  for (int o = threadIdx.x; o < nout; o += blockDim.x) {
    const int ia = o / P.c2b, lb = o % P.c2b;
    double acc = 0.0;
    for (int f = 0; f < P.n1; ++f) acc += qj[f * P.c2a + ia] * qk[f * P.c2b + lb];
    W[(size_t)o * P.K + (size_t)c * P.n1 + e] = acc;
  }
}

// Atop[(offa + i c2a + i') m + offb + l c2b + l'] = C[(i c1b + l) N + i' c2b + l'],  N = c2a c2b
__global__ void __launch_bounds__(256) k_kron_scatter(int c1a, int c2a, int c1b, int c2b, const double *__restrict__ C, double *Atop, int64_t m,
                                                      int64_t offa, int64_t offb) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t ma = (int64_t)c1a * c2a, mb = (int64_t)c1b * c2b;
  if (t >= ma * mb) return;
  const int64_t ra = t / mb, rb = t % mb;          // unknown indices within the two variables
  const int i = (int)(ra / c2a), ip = (int)(ra % c2a), l = (int)(rb / c2b), lp = (int)(rb % c2b);
  Atop[(offa + ra) * m + offb + rb] = C[((int64_t)i * c1b + l) * ((int64_t)c2a * c2b) + (int64_t)ip * c2b + lp];
}

}  // namespace mgbx
