// dense_check.cu -- test harness for the dense direct solvers and the FP64 DMMA GEMM (csrc/solver_kernels.cuh,
// csrc/dense_kernels.cuh), loaded with ctypes by tests/test_gpu_dense.py.  Every entry point takes host arrays, copies them
// to the device, launches the library's kernels exactly as the engine does (grid, block, dynamic shared memory and the
// raised shared-memory limits of solve_kernels_init), copies the result back and frees everything before it returns.
// The return value is 0 or a cudaError_t; dc_error_string names it.
//
// The launch sequence of chol_factor_solve is a copy of Engine::dense_factor / dense_apply / direct_solve
// (csrc/linear_solve.cu); the tests that go through the C ABI check the engine's own sequence.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "dense_kernels.cuh"
#include "solver_kernels.cuh"

using namespace mgbx;

namespace {

#define DC_CK(call)                          \
  do {                                       \
    const cudaError_t e_ = (call);           \
    if (e_ != cudaSuccess) return (int)e_;   \
  } while (0)

template <class T>
struct DevBuf {
  T *p = nullptr;
  ~DevBuf() {
    if (p) cudaFree(p);
  }
  cudaError_t alloc(size_t n) { return cudaMalloc((void **)&p, sizeof(T) * std::max<size_t>(n, 1)); }
  cudaError_t upload(const T *h, size_t n) {
    const cudaError_t e = alloc(n);
    return (e != cudaSuccess || n == 0) ? e : cudaMemcpy(p, h, sizeof(T) * n, cudaMemcpyHostToDevice);
  }
  cudaError_t download(T *h, size_t n) const { return n ? cudaMemcpy(h, p, sizeof(T) * n, cudaMemcpyDeviceToHost) : cudaSuccess; }
};

// the raised dynamic shared-memory limits, as solve_kernels_init sets them
cudaError_t init_once() {
  static bool done = false;
  if (done) return cudaSuccess;
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(k_coarse_inverse, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)coarse_inverse_smem(kCoarseMaxDense))) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_dense_solve_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dense_solve_small_smem(kCoarseMaxDense))) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_chol_diag_inv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCholDiagSmem)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_chol_solve_blocked, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * kDenseMaxUnknowns))) != cudaSuccess)
    return e;
  done = true;
  return cudaSuccess;
}

int nblk(int64_t n) { return (int)((n + 255) / 256); }

// r = b - A x, one thread per row in the CSR order (the refinement residual of Engine::direct_solve)
__global__ void k_residual(DevCsr A, const double *__restrict__ x, const double *__restrict__ b, double *r) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= A.rows) return;
  double s = b[row];
  for (int64_t k = A.ptr[row]; k < A.ptr[row + 1]; ++k) s -= A.val[k] * x[A.idx[k]];
  r[row] = s;
}

__global__ void k_add(int64_t m, double *x, const double *__restrict__ dx) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) x[i] += dx[i];
}

// the same grid as Engine::dgemm_nt (csrc/evaluate.cu)
cudaError_t launch_dgemm(int M, int N, int K, const double *A, int64_t lda, const double *B, int64_t ldb, const double *s, double *C, int64_t ldc,
                         int accumulate, double alpha) {
  if (M <= 0 || N <= 0) return cudaSuccess;
  dim3 grid((N + kGemmBN - 1) / kGemmBN, (M + kGemmBM - 1) / kGemmBM);
  k_dgemm_nt<<<grid, 128>>>(M, N, K, A, lda, B, ldb, s, C, ldc, accumulate, alpha);
  return cudaGetLastError();
}

struct Csr {
  DevBuf<int64_t> ptr;
  DevBuf<int32_t> idx;
  DevBuf<double> val;
  DevCsr d;
  cudaError_t upload(int64_t m, const int64_t *hp, const int32_t *hi, const double *hv) {
    cudaError_t e;
    const int64_t nnz = hp[m];
    if ((e = ptr.upload(hp, m + 1)) != cudaSuccess || (e = idx.upload(hi, nnz)) != cudaSuccess || (e = val.upload(hv, nnz)) != cudaSuccess) return e;
    d.rows = d.cols = m;
    d.nnz = nnz;
    d.ptr = ptr.p;
    d.idx = idx.p;
    d.val = val.p;
    return cudaSuccess;
  }
};

}  // namespace

extern "C" {

const char *dc_error_string(int e) { return cudaGetErrorString((cudaError_t)e); }

// C[i*ldc + j] (+)= alpha sum_k A[i*lda + k] s[k] B[j*ldb + k]; A is M x lda, B is N x ldb, C is M x ldc (row-major host
// arrays).  inplace: C aliases A on the device (ldc must equal lda) -- the L21 = A21 inv(L11)' form of the blocked Cholesky.
int dc_dgemm_nt(int M, int N, int K, const double *A, int64_t lda, const double *B, int64_t ldb, const double *s, double *C, int64_t ldc,
                int accumulate, double alpha, int inplace) {
  if (inplace && ldc != lda) return (int)cudaErrorInvalidValue;
  DevBuf<double> dA, dB, ds, dC;
  DC_CK(dA.upload(inplace ? C : A, (size_t)M * lda));
  DC_CK(dB.upload(B, (size_t)N * ldb));
  if (s) DC_CK(ds.upload(s, K));
  double *c = dA.p;
  if (!inplace) {
    DC_CK(dC.upload(C, (size_t)M * ldc));
    c = dC.p;
  }
  DC_CK(launch_dgemm(M, N, K, dA.p, lda, dB.p, ldb, s ? ds.p : nullptr, c, ldc, accumulate, alpha));
  DC_CK(cudaDeviceSynchronize());
  return (int)cudaMemcpy(C, c, sizeof(double) * (size_t)M * ldc, cudaMemcpyDeviceToHost);
}

// x = A^{-1} b by k_dense_solve_small (m <= 128); info: 0 = scaled Cholesky, 1 = pivoted elimination
int dc_dense_solve_small(int64_t m, const int64_t *ptr, const int32_t *idx, const double *val, const double *b, double *x, int *info) {
  if (m < 1 || m > kCoarseMaxDense) return (int)cudaErrorInvalidValue;
  DC_CK(init_once());
  Csr A;
  DevBuf<double> db, dx;
  DevBuf<int> di;
  DC_CK(A.upload(m, ptr, idx, val));
  DC_CK(db.upload(b, m));
  DC_CK(dx.alloc(m));
  DC_CK(di.alloc(1));
  DC_CK(cudaMemset(di.p, 0xff, sizeof(int)));
  k_dense_solve_small<<<1, 1024, dense_solve_small_smem((int)m)>>>(A.d, db.p, dx.p, di.p);
  DC_CK(cudaGetLastError());
  DC_CK(cudaDeviceSynchronize());
  DC_CK(dx.download(x, m));
  return (int)di.download(info, 1);
}

// x = A^{-1} b by the launch sequence of Engine::direct_solve: above 128 unknowns the scaled blocked Cholesky of
// Engine::dense_factor applied by k_chol_solve_blocked (Engine::dense_apply), k_dense_solve_small below; refine = 1 adds
// the one step of iterative refinement against the CSR matrix, refine = 0 returns the first solve.
int dc_chol_factor_solve(int64_t m, const int64_t *ptr, const int32_t *idx, const double *val, const double *b, double *x, int refine) {
  if (m < 1 || m > kDenseMaxUnknowns) return (int)cudaErrorInvalidValue;
  DC_CK(init_once());
  const int mi = (int)m;
  const bool small = m <= kCoarseMaxDense;
  const int npan = (mi + kCholNB - 1) / kCholNB;
  Csr A;
  DevBuf<double> db, dx, dr, dx2, dense, dscale, dinv;
  DC_CK(A.upload(m, ptr, idx, val));
  DC_CK(db.upload(b, m));
  DC_CK(dx.alloc(m));
  DC_CK(dr.alloc(m));
  DC_CK(dx2.alloc(m));
  if (!small) {
    DC_CK(dense.alloc((size_t)m * m));
    DC_CK(dscale.alloc(m));
    DC_CK(dinv.alloc((size_t)npan * kCholNB * kCholNB));
    DC_CK(cudaMemset(dense.p, 0, sizeof(double) * (size_t)m * m));
    k_dense_scale_diag<<<nblk(m), 256>>>(A.d, dscale.p);
    k_csr_to_dense<<<nblk(m), 256>>>(A.d, dscale.p, dense.p);
    DC_CK(cudaGetLastError());
    for (int p = 0; p < npan; ++p) {
      const int k0 = p * kCholNB, nb = std::min(kCholNB, mi - k0), rem = mi - k0 - nb;
      double *Li = dinv.p + (size_t)p * kCholNB * kCholNB;
      k_chol_diag_inv<<<1, 1024, kCholDiagSmem>>>(dense.p, mi, k0, Li);
      DC_CK(cudaGetLastError());
      if (rem > 0) {
        double *A21 = dense.p + (size_t)(k0 + nb) * m + k0;
        DC_CK(launch_dgemm(rem, nb, nb, A21, m, Li, kCholNB, nullptr, A21, m, 0, 1.0));
        DC_CK(launch_dgemm(rem, rem, nb, A21, m, A21, m, nullptr, dense.p + (size_t)(k0 + nb) * m + k0 + nb, m, 1, -1.0));
      }
    }
  }
  auto apply = [&](const double *rhs, double *out) {
    if (small) k_dense_solve_small<<<1, 1024, dense_solve_small_smem(mi)>>>(A.d, rhs, out, nullptr);
    else k_chol_solve_blocked<<<1, 1024, sizeof(double) * m>>>(dense.p, mi, dinv.p, dscale.p, rhs, out);
  };
  apply(db.p, dx.p);
  if (refine) {
    k_residual<<<nblk(m), 256>>>(A.d, dx.p, db.p, dr.p);
    apply(dr.p, dx2.p);
    k_add<<<nblk(m), 256>>>(m, dx.p, dx2.p);
  }
  DC_CK(cudaGetLastError());
  DC_CK(cudaDeviceSynchronize());
  return (int)dx.download(x, m);
}

// Minv (m x m, row-major) = the dense inverse of the V-cycle's coarsest level by k_coarse_inverse (m <= 128)
int dc_coarse_inverse(int64_t m, const int64_t *ptr, const int32_t *idx, const double *val, double *Minv) {
  if (m < 1 || m > kCoarseMaxDense) return (int)cudaErrorInvalidValue;
  DC_CK(init_once());
  Csr A;
  DevBuf<double> dM;
  DC_CK(A.upload(m, ptr, idx, val));
  DC_CK(dM.alloc((size_t)m * m));
  k_coarse_inverse<<<1, 1024, coarse_inverse_smem((int)m)>>>(A.d, dM.p);
  DC_CK(cudaGetLastError());
  DC_CK(cudaDeviceSynchronize());
  return (int)dM.download(Minv, (size_t)m * m);
}

}  // extern "C"
