// setup_kernels.cuh -- plan construction on the device (runs once per linear-system family, at the first
// Newton iteration that needs it).  Not on the per-iteration hot path, but on the end-to-end path of every
// mgb_solve call, so it is done on the GPU instead of in host loops:
//   device_symbolic      sparsity pattern of a sparse product (candidate keys -> radix sort -> unique), the
//                        symbolic half of the Galerkin products A T and T'(A T)
//   k_top_plan           term list of the element-block -> CSR gather (the scatter_idx of
//                        src/BlockMatrices.jl:448-491, inverted into a fixed-order gather)
//   k_prod_plan<0|1>     term lists of the Galerkin gathers (k_sell_gather)
//   k_csr_block_to_dense_t  dense prolongation blocks of the spectral path
// CUB (radix sort / scan / unique) is used for the sort; everything else is hand-written.  Compiled by setup.cu only.
#pragma once
#include <cub/cub.cuh>

#include "device_common.cuh"

namespace mgbx {

// number of candidate (row, col) pairs of row i of A*B
__global__ void k_sym_count(DevCsr A, DevCsr B, int64_t *cand) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > A.rows) return;
  if (i == A.rows) {
    cand[i] = 0;
    return;
  }
  int64_t c = 0;
  for (int64_t k = A.ptr[i]; k < A.ptr[i + 1]; ++k) {
    const int64_t r = A.idx[k];
    c += B.ptr[r + 1] - B.ptr[r];
  }
  cand[i] = c;
}

__global__ void k_sym_fill(DevCsr A, DevCsr B, const int64_t *__restrict__ offs, unsigned long long *keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.rows) return;
  int64_t pos = offs[i];
  for (int64_t k = A.ptr[i]; k < A.ptr[i + 1]; ++k) {
    const int64_t r = A.idx[k];
    for (int64_t q = B.ptr[r]; q < B.ptr[r + 1]; ++q) keys[pos++] = ((unsigned long long)i << 32) | (unsigned int)B.idx[q];
  }
}

// ptr[i] = first position with key >= (i << 32); idx = low words
__global__ void k_sym_finish(const unsigned long long *__restrict__ uniq, int64_t nnz, int64_t rows, int64_t *ptr, int32_t *idx) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nnz) idx[t] = (int32_t)(uniq[t] & 0xffffffffull);
  if (t <= rows) {
    const unsigned long long key = (unsigned long long)t << 32;
    int64_t lo = 0, hi = nnz;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (uniq[mid] < key) lo = mid + 1;
      else hi = mid;
    }
    ptr[t] = lo;
  }
}

template <int FILL>
__global__ void __launch_bounds__(256) k_top_plan(TopPlanParams Q, SellPlan P, int32_t *width) {
  const int64_t nz = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int count = 0;
  if (nz < Q.pat.nnz) {
    const int64_t i = Q.rowof[nz], j = Q.pat.idx[nz];
    int qa = 0, qb = 0;
    while (qa + 1 < Q.nkept && i >= Q.off[qa + 1]) ++qa;
    while (qb + 1 < Q.nkept && j >= Q.off[qb + 1]) ++qb;
    const int pr = Q.pair_of[qa * Q.nkept + qb];
    if (pr >= 0) {
      const int va = Q.kept[qa], vb = Q.kept[qb];
      const int32_t ci = (int32_t)(Q.rcol0[qa] + (i - Q.off[qa])), cj = (int32_t)(Q.rcol0[qb] + (j - Q.off[qb]));
      const int p = Q.p;
      const int64_t off = FILL ? P.sptr[nz >> 5] + (nz & 31) : 0;
      for (int64_t t = Q.EincT.ptr[i]; t < Q.EincT.ptr[i + 1]; ++t) {
        const int64_t e = Q.EincT.idx[t];
        for (int r = 0; r < p; ++r) {
          const int64_t ka = csr_find(Q.R, (int64_t)va * Q.n + e * p + r, ci);
          if (ka < 0) continue;
          for (int c = 0; c < p; ++c) {
            const int64_t kb = csr_find(Q.R, (int64_t)vb * Q.n + e * p + c, cj);
            if (kb < 0) continue;
            if (FILL) {
              P.src[off + 32 * (int64_t)count] = (int32_t)((((int64_t)pr * Q.N + e) * p + r) * p + c);
              if (!Q.unit) P.w[off + 32 * (int64_t)count] = Q.R.val[ka] * Q.R.val[kb];
            }
            ++count;
          }
        }
      }
    }
    if (!FILL) P.cnt[nz] = count;
  }
  if (!FILL) {
    int wmax = count;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wmax = max(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
    if ((threadIdx.x & 31) == 0 && nz < Q.pat.nnz) width[nz >> 5] = wmax;
  }
}

// row index of every non-zero of a CSR pattern
__global__ void k_csr_rows(DevCsr A, int32_t *rowof) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= A.rows) return;
  for (int64_t k = A.ptr[row]; k < A.ptr[row + 1]; ++k) rowof[k] = (int32_t)row;
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

// Rt[j][i] = R[i][cols j] for the row block [r0, r0+n) and column block [c0, c0+mv) of a CSR matrix (dense transposed copy)
__global__ void k_csr_block_to_dense_t(DevCsr R, int64_t r0, int n, int64_t c0, int mv, double *Rt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (int64_t k = R.ptr[r0 + i]; k < R.ptr[r0 + i + 1]; ++k) {
    const int64_t c = R.idx[k] - c0;
    if (c >= 0 && c < mv) Rt[c * (int64_t)n + i] = R.val[k];
  }
}

}  // namespace mgbx
