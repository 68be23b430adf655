// Microbenchmark of ONE mat-vec phase of a persistent solve kernel (the CSR phase of the first solve kernel, since replaced by k_pcg2),
// run the way the kernel runs it: cooperative launch, one CTA of 1024 threads per SM, the matrix L2-resident, phases
// separated by the same flip grid barrier, every phase reading the vector the previous phase wrote.
//
// Variants (results checked against variant 0 with one lane per row, which sums each row in index order):
//   rows<G>      the shipped mapping: G lanes per row, grid-strided passes over the rows
//   rows_pf<G>   + row pointers of the NEXT pass loaded before the current row is processed
//   rows_pf2     one lane per row, row pointers two passes ahead and the first U index/value pairs one pass ahead
//   stream       CSR-stream: a CTA takes a block of whole rows holding <= chunk non-zeros, all threads form the products
//                val*x[idx] with coalesced loads into shared memory, then one thread per row adds its products in order
//   sell         sliced ELL (32 rows per slice, column-major, padded): one lane per row, coalesced, all loads of a row
//                independent
// and, for the single-CTA tail levels: a 508-row matrix applied by one CTA from global memory vs from shared memory.
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o bench_spmv_phase bench_spmv_phase.cu && ./bench_spmv_phase
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include <vector>

#define CK(x)                                                                                   \
  do {                                                                                          \
    cudaError_t e_ = (x);                                                                       \
    if (e_ != cudaSuccess) {                                                                    \
      fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_));        \
      exit(1);                                                                                  \
    }                                                                                           \
  } while (0)

constexpr int kThreads = 1024;

struct Csr {
  int rows, nnz;
  const int *ptr, *idx;
  const double *val;
};

struct Stream {          // CSR-stream row blocks
  int nblocks, chunk;    // chunk = max non-zeros per block (<= kThreads * kStreamK)
  const int *brow;       // nblocks + 1 row boundaries
};
constexpr int kStreamK = 6;

struct Sell {
  int rows, nslices;
  const int *soff;       // nslices + 1 offsets (in entries) into idx / val; width = (soff[s+1]-soff[s]) / 32
  const int *idx;        // padded entries point at column 0 with value 0
  const double *val;
};

__device__ __forceinline__ void grid_barrier(unsigned int *bar) {
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int nb = 1;
    if (blockIdx.x == 0) nb = 0x80000000u - (gridDim.x - 1);
    unsigned int old, cur;
    asm volatile("atom.add.release.gpu.u32 %0,[%1],%2;" : "=r"(old) : "l"(bar), "r"(nb) : "memory");
    int spins = 0;
    do {
      asm volatile("ld.acquire.gpu.u32 %0,[%1];" : "=r"(cur) : "l"(bar) : "memory");
      if (++spins > 64) __nanosleep(40);
    } while (((old ^ cur) & 0x80000000u) == 0);
  }
  __syncthreads();
}

// ---- variant: rows<G> (the shipped mapping) ---------------------------------------------------------------------
template <int G>
__device__ void ph_rows(const Csr &A, const double *x, double *y, int tid, int nthr) {
  const int step = nthr / G, sub = tid % G, r0 = tid / G;
  for (int base = 0; base < A.rows; base += step) {
    const int row = base + r0;
    const bool valid = row < A.rows;
    double acc = 0.0;
    if (valid) {
      const int b = __ldg(A.ptr + row), e = __ldg(A.ptr + row + 1);
      for (int k = b + sub; k < e; k += G) acc += __ldg(A.val + k) * __ldcg(x + __ldg(A.idx + k));
    }
    if (G > 1) {
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o, G);
    }
    if (valid && sub == 0) y[row] = acc;
  }
}

// ---- variant: rows_pf<G> (next pass's row pointers in flight) ---------------------------------------------------
template <int G>
__device__ void ph_rows_pf(const Csr &A, const double *x, double *y, int tid, int nthr) {
  const int step = nthr / G, sub = tid % G;
  int row = tid / G;
  int b = 0, e = 0;
  if (row < A.rows) {
    b = __ldg(A.ptr + row);
    e = __ldg(A.ptr + row + 1);
  }
  for (int base = 0; base < A.rows; base += step) {
    const int nrow = row + step;
    int nb = 0, ne = 0;
    if (nrow < A.rows) {
      nb = __ldg(A.ptr + nrow);
      ne = __ldg(A.ptr + nrow + 1);
    }
    double acc = 0.0;
    for (int k = b + sub; k < e; k += G) acc += __ldg(A.val + k) * __ldcg(x + __ldg(A.idx + k));
    if (G > 1) {
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o, G);
    }
    if (row < A.rows && sub == 0) y[row] = acc;
    row = nrow;
    b = nb;
    e = ne;
  }
}

// ---- variant: rows_pf2 (one lane per row; pointers two passes ahead, first U entries one pass ahead) --------------
template <int U>
__device__ void ph_rows_pf2(const Csr &A, const double *x, double *y, int tid, int nthr) {
  int row = tid;
  int b = 0, e = 0, nb = 0, ne = 0;
  if (row < A.rows) {
    b = __ldg(A.ptr + row);
    e = __ldg(A.ptr + row + 1);
  }
  if (row + nthr < A.rows) {
    nb = __ldg(A.ptr + row + nthr);
    ne = __ldg(A.ptr + row + nthr + 1);
  }
  int ci[U];
  double cv[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const bool in = b + u < e;
    ci[u] = in ? __ldg(A.idx + b + u) : 0;
    cv[u] = in ? __ldg(A.val + b + u) : 0.0;
  }
  for (int base = 0; base < A.rows; base += nthr) {
    // pointers of the pass after next
    const int r2 = row + 2 * nthr;
    int b2 = 0, e2 = 0;
    if (r2 < A.rows) {
      b2 = __ldg(A.ptr + r2);
      e2 = __ldg(A.ptr + r2 + 1);
    }
    // index / value pairs of the next pass
    int ni[U];
    double nv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const bool in = nb + u < ne;
      ni[u] = in ? __ldg(A.idx + nb + u) : 0;
      nv[u] = in ? __ldg(A.val + nb + u) : 0.0;
    }
    // current row: the gathers are the only dependent loads left
    double xs[U];
#pragma unroll
    for (int u = 0; u < U; ++u) xs[u] = (b + u < e) ? __ldcg(x + ci[u]) : 0.0;
    double acc = 0.0;
#pragma unroll
    for (int u = 0; u < U; ++u) acc += cv[u] * xs[u];
    for (int k = b + U; k < e; ++k) acc += __ldg(A.val + k) * __ldcg(x + __ldg(A.idx + k));
    if (row < A.rows) y[row] = acc;
    row += nthr;
    b = nb;
    e = ne;
    nb = b2;
    ne = e2;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      ci[u] = ni[u];
      cv[u] = nv[u];
    }
  }
}

// ---- variant: CSR-stream ----------------------------------------------------------------------------------------
__device__ void ph_stream(const Csr &A, const Stream &S, const double *x, double *y, double *prod /* smem, chunk */) {
  for (int blk = blockIdx.x; blk < S.nblocks; blk += gridDim.x) {
    const int r0 = __ldg(S.brow + blk), r1 = __ldg(S.brow + blk + 1);
    const int k0 = __ldg(A.ptr + r0), k1 = __ldg(A.ptr + r1);
    // the row pointers of this block's rows (needed after the products) are requested first
    const int myrow = r0 + (int)threadIdx.x;
    int rb = 0, re = 0;
    if (myrow < r1) {
      rb = __ldg(A.ptr + myrow);
      re = __ldg(A.ptr + myrow + 1);
    }
    int ji[kStreamK];
    double jv[kStreamK];
#pragma unroll
    for (int q = 0; q < kStreamK; ++q) {
      const int k = k0 + q * kThreads + (int)threadIdx.x;
      const bool in = k < k1;
      ji[q] = in ? __ldg(A.idx + k) : 0;
      jv[q] = in ? __ldg(A.val + k) : 0.0;
    }
#pragma unroll
    for (int q = 0; q < kStreamK; ++q) {
      const int k = k0 + q * kThreads + (int)threadIdx.x;
      if (k < k1) prod[k - k0] = jv[q] * __ldcg(x + ji[q]);
    }
    __syncthreads();
    // rows of the block: more rows than threads cannot happen when every row has >= 1 entry and chunk <= K * threads,
    // but guard with a loop anyway
    for (int row = myrow; row < r1; row += kThreads) {
      if (row != myrow) {
        rb = __ldg(A.ptr + row);
        re = __ldg(A.ptr + row + 1);
      }
      double acc = 0.0;
      for (int k = rb; k < re; ++k) acc += prod[k - k0];
      y[row] = acc;
    }
    __syncthreads();
  }
}

// ---- variant: sliced ELL ----------------------------------------------------------------------------------------
__device__ void ph_sell(const Sell &E, const double *x, double *y, int tid, int nthr) {
  const int lane = tid & 31;
  for (int base = 0; base < E.rows; base += nthr) {
    const int row = base + tid;
    const int slice = row >> 5;
    double acc = 0.0;
    if (slice < E.nslices) {
      const int o0 = __ldg(E.soff + slice), o1 = __ldg(E.soff + slice + 1);
      const int w = (o1 - o0) >> 5;
      const int *ip = E.idx + o0 + lane;
      const double *vp = E.val + o0 + lane;
      int k = 0;
      for (; k + 4 <= w; k += 4) {
        const int j0 = __ldg(ip + 32 * k), j1 = __ldg(ip + 32 * (k + 1)), j2 = __ldg(ip + 32 * (k + 2)), j3 = __ldg(ip + 32 * (k + 3));
        const double v0 = __ldg(vp + 32 * k), v1 = __ldg(vp + 32 * (k + 1)), v2 = __ldg(vp + 32 * (k + 2)), v3 = __ldg(vp + 32 * (k + 3));
        const double x0 = __ldcg(x + j0), x1 = __ldcg(x + j1), x2 = __ldcg(x + j2), x3 = __ldcg(x + j3);
        acc += v0 * x0;
        acc += v1 * x1;
        acc += v2 * x2;
        acc += v3 * x3;
      }
      for (; k < w; ++k) acc += __ldg(vp + 32 * k) * __ldcg(x + __ldg(ip + 32 * k));
    }
    if (row < E.rows) y[row] = acc;
  }
}

// variant ids
enum { V_ROWS1 = 0, V_ROWS4, V_ROWS_PF1, V_ROWS_PF4, V_ROWS_PF2_4, V_ROWS_PF2_8, V_STREAM, V_SELL, V_COUNT };
static const char *kNames[V_COUNT] = {"rows<1>", "rows<4>", "rows_pf<1>", "rows_pf<4>", "rows_pf2<U=4>", "rows_pf2<U=8>", "stream", "sell"};

template <int V>
__global__ void __launch_bounds__(kThreads, 1) k_phase(Csr A, Stream S, Sell E, double *xa, double *xb, int iters, unsigned int *bar) {
  extern __shared__ double prod[];
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nthr = gridDim.x * blockDim.x;
  double *x = xa, *y = xb;
  for (int it = 0; it < iters; ++it) {
    if (V == V_ROWS1) ph_rows<1>(A, x, y, tid, nthr);
    else if (V == V_ROWS4) ph_rows<4>(A, x, y, tid, nthr);
    else if (V == V_ROWS_PF1) ph_rows_pf<1>(A, x, y, tid, nthr);
    else if (V == V_ROWS_PF4) ph_rows_pf<4>(A, x, y, tid, nthr);
    else if (V == V_ROWS_PF2_4) ph_rows_pf2<4>(A, x, y, tid, nthr);
    else if (V == V_ROWS_PF2_8) ph_rows_pf2<8>(A, x, y, tid, nthr);
    else if (V == V_STREAM) ph_stream(A, S, x, y, prod);
    else ph_sell(E, x, y, tid, nthr);
    grid_barrier(bar);
    double *t = x;
    x = y;
    y = t;
  }
}

// ---- single-CTA tail: the same 4-lane row mapping from global memory vs from shared memory -------------------------
template <bool SMEM>
__global__ void __launch_bounds__(kThreads, 1) k_tail(Csr A, double *xa, double *xb, int iters) {
  extern __shared__ unsigned char raw[];
  Csr B = A;
  if (SMEM) {
    double *sval = reinterpret_cast<double *>(raw);
    int *sidx = reinterpret_cast<int *>(sval + A.nnz);
    int *sptr = sidx + A.nnz;
    for (int k = threadIdx.x; k < A.nnz; k += blockDim.x) {
      sval[k] = A.val[k];
      sidx[k] = A.idx[k];
    }
    for (int r = threadIdx.x; r <= A.rows; r += blockDim.x) sptr[r] = A.ptr[r];
    __syncthreads();
    B.val = sval;
    B.idx = sidx;
    B.ptr = sptr;
  }
  constexpr int G = 4;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const int step = nthr / G, sub = tid % G, r0 = tid / G;
  double *x = xa, *y = xb;
  for (int it = 0; it < iters; ++it) {
    for (int base = 0; base < B.rows; base += step) {
      const int row = base + r0;
      const bool valid = row < B.rows;
      double acc = 0.0;
      if (valid) {
        const int b = B.ptr[row], e = B.ptr[row + 1];   // generic loads: global or shared
        for (int k = b + sub; k < e; k += G) acc += B.val[k] * __ldcg(x + B.idx[k]);
      }
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o, G);
      if (valid && sub == 0) y[row] = acc;
    }
    __syncthreads();
    double *t = x;
    x = y;
    y = t;
  }
}

// ------------------------------------------------------------------------------------------------------- host side
struct HostCsr {
  int rows = 0;
  std::vector<int> ptr, idx;
  std::vector<double> val;
};

// stencil matrix on an n x n grid; rows scaled to sum 1 (an averaging operator keeps the iterated vector bounded)
static HostCsr stencil(int n, const std::vector<std::pair<int, int>> &offs) {
  HostCsr A;
  A.rows = n * n;
  A.ptr.push_back(0);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) {
      std::vector<int> cols;
      for (auto &o : offs) {
        const int a = i + o.first, b = j + o.second;
        if (a >= 0 && a < n && b >= 0 && b < n) cols.push_back(a * n + b);
      }
      std::sort(cols.begin(), cols.end());
      for (int c : cols) {
        A.idx.push_back(c);
        A.val.push_back(1.0 / (double)cols.size());
      }
      A.ptr.push_back((int)A.idx.size());
    }
  return A;
}

// CSR-stream blocks: as many rounds as a 4096-entry chunk needs, chunk sized so that the blocks fill whole rounds
static std::vector<int> build_stream(const HostCsr &H, int grid, int &rounds, int &chunk) {
  const int nnz = (int)H.idx.size();
  rounds = std::max(1, (int)std::ceil((double)nnz / ((double)grid * 4096.0)));
  chunk = (int)std::ceil((double)nnz / ((double)grid * rounds)) + 64;
  chunk = std::min(chunk, kThreads * kStreamK);
  std::vector<int> brow{0};
  for (int r = 0, start = 0; r < H.rows; ++r) {
    if (H.ptr[r + 1] - H.ptr[start] > chunk || r + 1 - start > kThreads) {
      brow.push_back(r);
      start = r;
    }
  }
  brow.push_back(H.rows);
  return brow;
}

// sliced ELL, 32 rows per slice, column-major inside a slice, padded with (column 0, value 0)
static void build_sell(const HostCsr &H, std::vector<int> &soff, std::vector<int> &eidx, std::vector<double> &eval) {
  const int nslices = (H.rows + 31) / 32;
  soff.assign(nslices + 1, 0);
  for (int s = 0; s < nslices; ++s) {
    int w = 0;
    for (int r = 32 * s; r < std::min(H.rows, 32 * s + 32); ++r) w = std::max(w, H.ptr[r + 1] - H.ptr[r]);
    soff[s + 1] = soff[s] + 32 * w;
  }
  eidx.assign(soff.back(), 0);
  eval.assign(soff.back(), 0.0);
  for (int r = 0; r < H.rows; ++r) {
    const int s = r >> 5, lane = r & 31;
    for (int k = H.ptr[r]; k < H.ptr[r + 1]; ++k) {
      const int q = soff[s] + 32 * (k - H.ptr[r]) + lane;
      eidx[q] = H.idx[k];
      eval[q] = H.val[k];
    }
  }
}

template <class T>
static T *upload(const std::vector<T> &v) {
  T *d = nullptr;
  CK(cudaMalloc(&d, std::max<size_t>(v.size(), 1) * sizeof(T)));
  CK(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return d;
}

template <int V>
static float launch(const Csr &A, const Stream &S, const Sell &E, double *xa, double *xb, int iters, unsigned int *bar, int grid, size_t smem) {
  CK(cudaFuncSetAttribute(k_phase<V>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  Csr a = A;
  Stream s = S;
  Sell e = E;
  void *args[] = {&a, &s, &e, &xa, &xb, &iters, &bar};
  cudaEvent_t t0, t1;
  CK(cudaEventCreate(&t0));
  CK(cudaEventCreate(&t1));
  CK(cudaMemset(bar, 0, 1024));
  CK(cudaEventRecord(t0));
  CK(cudaLaunchCooperativeKernel((const void *)k_phase<V>, dim3(grid), dim3(kThreads), args, smem, 0));
  CK(cudaEventRecord(t1));
  CK(cudaEventSynchronize(t1));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, t0, t1));
  CK(cudaEventDestroy(t0));
  CK(cudaEventDestroy(t1));
  return ms;
}

typedef float (*launch_fn)(const Csr &, const Stream &, const Sell &, double *, double *, int, unsigned int *, int, size_t);

static void bench_matrix(const char *name, const HostCsr &H, int grid) {
  const int nnz = (int)H.idx.size();
  Csr A{H.rows, nnz, upload(H.ptr), upload(H.idx), upload(H.val)};
  int rounds = 0, chunk = 0;
  const std::vector<int> brow = build_stream(H, grid, rounds, chunk);
  Stream S{(int)brow.size() - 1, chunk, upload(brow)};
  std::vector<int> soff, eidx;
  std::vector<double> eval;
  build_sell(H, soff, eidx, eval);
  const int nslices = (int)soff.size() - 1;
  Sell E{H.rows, nslices, upload(soff), upload(eidx), upload(eval)};

  std::vector<double> x0(H.rows);
  for (int i = 0; i < H.rows; ++i) x0[i] = std::sin(0.001 * i) + 1.5;
  double *xa = upload(x0), *xb = upload(x0);
  unsigned int *bar;
  CK(cudaMalloc(&bar, 1024));
  const size_t smem = (size_t)kThreads * kStreamK * sizeof(double);
  const int iters = 200;   // even: the result of the last phase lands in xa
  const double bytes = 12.0 * nnz + 4.0 * H.rows + 16.0 * H.rows;
  printf("%s: rows %d, nnz %d (%.1f per row), stream blocks %d (chunk %d, %d rounds), sell padding %.2fx\n", name, H.rows, nnz,
         (double)nnz / H.rows, S.nblocks, chunk, rounds, (double)soff.back() / nnz);
  launch_fn fns[V_COUNT] = {launch<V_ROWS1>, launch<V_ROWS4>, launch<V_ROWS_PF1>, launch<V_ROWS_PF4>,
                            launch<V_ROWS_PF2_4>, launch<V_ROWS_PF2_8>, launch<V_STREAM>, launch<V_SELL>};
  std::vector<double> ref, out(H.rows);
  for (int v = 0; v < V_COUNT; ++v) {
    float best = 1e30f;
    for (int rep = 0; rep < 3; ++rep) {
      CK(cudaMemcpy(xa, x0.data(), H.rows * sizeof(double), cudaMemcpyHostToDevice));
      best = std::min(best, fns[v](A, S, E, xa, xb, iters, bar, grid, smem));
    }
    CK(cudaMemcpy(out.data(), xa, H.rows * sizeof(double), cudaMemcpyDeviceToHost));
    if (v == 0) ref = out;
    double err = 0.0;
    for (int i = 0; i < H.rows; ++i) err = std::max(err, std::fabs(out[i] - ref[i]));
    const double us = 1e3 * best / iters;
    printf("  %-14s %7.2f us per phase (incl. barrier)  %7.1f GB/s  max|diff| %.2e\n", kNames[v], us, bytes / us * 1e-3, err);
  }
  cudaFree((void *)A.ptr); cudaFree((void *)A.idx); cudaFree((void *)A.val);
  cudaFree((void *)S.brow); cudaFree((void *)E.soff); cudaFree((void *)E.idx); cudaFree((void *)E.val);
  cudaFree(xa); cudaFree(xb); cudaFree(bar);
}

static void bench_tail(const HostCsr &H) {
  const int nnz = (int)H.idx.size();
  Csr A{H.rows, nnz, upload(H.ptr), upload(H.idx), upload(H.val)};
  std::vector<double> x0(H.rows, 1.0);
  double *xa = upload(x0), *xb = upload(x0);
  const size_t smem = (size_t)nnz * 12 + (size_t)(H.rows + 1) * 4 + 16;
  const bool fits = smem <= 220 * 1024;
  if (fits) CK(cudaFuncSetAttribute(k_tail<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int iters = 2000;
  for (int mode = 0; mode < (fits ? 2 : 1); ++mode) {
    float best = 1e30f;
    for (int rep = 0; rep < 3; ++rep) {
      cudaEvent_t t0, t1;
      CK(cudaEventCreate(&t0));
      CK(cudaEventCreate(&t1));
      CK(cudaEventRecord(t0));
      if (mode == 0) k_tail<false><<<1, kThreads>>>(A, xa, xb, iters);
      else k_tail<true><<<1, kThreads, smem>>>(A, xa, xb, iters);
      CK(cudaEventRecord(t1));
      CK(cudaEventSynchronize(t1));
      CK(cudaGetLastError());
      float ms = 0;
      CK(cudaEventElapsedTime(&ms, t0, t1));
      best = std::min(best, ms);
      CK(cudaEventDestroy(t0));
      CK(cudaEventDestroy(t1));
    }
    printf("  tail %d rows, %d nnz, one CTA, matrix in %-6s: %.3f us per phase\n", H.rows, nnz, mode ? "shared" : "global", 1e3 * best / iters);
  }
  cudaFree((void *)A.ptr); cudaFree((void *)A.idx); cudaFree((void *)A.val); cudaFree(xa); cudaFree(xb);
}

#ifdef HOST_CHECK
// CPU check of the two layouts (no GPU needed):  g++ -x c++ is not enough (CUDA syntax), so
//   nvcc -DHOST_CHECK -O2 -o host_check bench_spmv_phase.cu && ./host_check
static int host_check(const char *name, const HostCsr &H, int grid) {
  int rounds = 0, chunk = 0, bad = 0;
  const std::vector<int> brow = build_stream(H, grid, rounds, chunk);
  std::vector<double> x(H.rows), y0(H.rows, 0.0), y1(H.rows, 0.0), y2(H.rows, 0.0);
  for (int i = 0; i < H.rows; ++i) x[i] = std::sin(0.001 * i) + 1.5;
  for (int r = 0; r < H.rows; ++r)
    for (int k = H.ptr[r]; k < H.ptr[r + 1]; ++k) y0[r] += H.val[k] * x[H.idx[k]];
  int maxnnz = 0, maxrows = 0;
  for (size_t b = 0; b + 1 < brow.size(); ++b) {
    const int r0 = brow[b], r1 = brow[b + 1], k0 = H.ptr[r0], k1 = H.ptr[r1];
    if (r1 <= r0) ++bad;
    maxnnz = std::max(maxnnz, k1 - k0);
    maxrows = std::max(maxrows, r1 - r0);
    std::vector<double> prod(k1 - k0);
    for (int k = k0; k < k1; ++k) prod[k - k0] = H.val[k] * x[H.idx[k]];
    for (int r = r0; r < r1; ++r)
      for (int k = H.ptr[r]; k < H.ptr[r + 1]; ++k) y1[r] += prod[k - k0];
  }
  if (maxnnz > chunk || maxnnz > kThreads * kStreamK || maxrows > kThreads) ++bad;
  std::vector<int> soff, eidx;
  std::vector<double> eval;
  build_sell(H, soff, eidx, eval);
  for (int r = 0; r < H.rows; ++r) {
    const int s = r >> 5, lane = r & 31, w = (soff[s + 1] - soff[s]) >> 5;
    for (int k = 0; k < w; ++k) y2[r] += eval[soff[s] + 32 * k + lane] * x[eidx[soff[s] + 32 * k + lane]];
  }
  double e1 = 0, e2 = 0;
  for (int r = 0; r < H.rows; ++r) {
    e1 = std::max(e1, std::fabs(y1[r] - y0[r]));
    e2 = std::max(e2, std::fabs(y2[r] - y0[r]));
  }
  const int nblocks = (int)brow.size() - 1;
  printf("%s: rows %d nnz %zu | stream: %d blocks for %d x %d slots, chunk %d, max block nnz %d rows %d, err %.1e | sell: pad %.2fx err %.1e | %s\n",
         name, H.rows, H.idx.size(), nblocks, grid, rounds, chunk, maxnnz, maxrows, e1, (double)soff.back() / H.idx.size(), e2,
         (bad || e1 > 0 || e2 > 1e-15 || nblocks > grid * rounds) ? "CHECK" : "ok");
  return bad;
}
#endif

int main() {
  int nsm = 148;
#ifndef HOST_CHECK
  CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, 0));
  printf("grid %d x %d\n", nsm, kThreads);
#endif
  const std::vector<std::pair<int, int>> p1 = {{0, 0}, {1, 0}, {-1, 0}, {0, 1}, {0, -1}, {1, 1}, {-1, -1}};
  std::vector<std::pair<int, int>> gal = {{0, 0}, {1, 0}, {-1, 0}, {0, 1}, {0, -1}, {1, 1}, {-1, -1}, {1, -1}, {-1, 1},
                                          {2, 0}, {-2, 0}, {0, 2}, {0, -2}, {2, 2}, {-2, -2}};
  std::vector<std::pair<int, int>> q1;   // 27-point pattern flattened onto the plane (5 x 5 + 2): long rows
  for (int a = -2; a <= 2; ++a)
    for (int b = -2; b <= 2; ++b) q1.push_back({a, b});
  q1.push_back({3, 0});
  q1.push_back({-3, 0});
#ifdef HOST_CHECK
  host_check("P1 511^2", stencil(511, p1), nsm);
  host_check("Galerkin 361^2", stencil(361, gal), nsm);
  host_check("Galerkin 181^2", stencil(181, gal), nsm);
  host_check("27/row 1000^2", stencil(1000, q1), nsm);
  host_check("tiny 5^2", stencil(5, gal), nsm);
  return 0;
#endif
  bench_matrix("P1 top level (C2 level 0)", stencil(511, p1), nsm);
  bench_matrix("Galerkin level (C2 level 1)", stencil(361, gal), nsm);
  bench_matrix("Galerkin level (C2 level 2)", stencil(181, gal), nsm);
  bench_matrix("27 per row, 1 M rows (3-D like)", stencil(1000, q1), nsm);
  bench_tail(stencil(23, gal));    // 529 rows ~ the 508-row tail level
  bench_tail(stencil(45, gal));    // 2025 rows ~ the 2032-row level
  return 0;
}
