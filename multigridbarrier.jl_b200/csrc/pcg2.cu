// pcg2.cu -- the persistent V-cycle-PCG solve kernel k_pcg2 (see pcg2.hpp for what it replaces and how).
//
// One cooperative launch = one Newton system H d = g solved to the requested relative residual:
//   repeat { z = V-cycle(r);  beta = r.z / r.z_old;  p = z + beta p;  Ap = A p;  alpha = r.z / p.Ap;  x += alpha p;  r -= alpha Ap }
// One CTA of 1024 threads per SM.  Phases are separated by a grid barrier (release/acquire on one counter).  Every level
// matrix is sliced ELL (32 rows per slice); CTA c owns the slices [c spc, (c+1) spc) of a level in every phase and its warps
// take them round-robin, lane = row.  Levels [nbig, nlev) are run by CTA 0 alone out of shared memory (matrices and vectors).
#include "pcg2.hpp"

#include <math.h>

namespace mgbx {
namespace {

__device__ __forceinline__ double warp_sum2(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void grid_barrier2(unsigned int *bar) {
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

// Optional phase profile (Pcg2Plan::prof != nullptr; debugging aid, env MGBX_PCG_PROF): thread 0 of CTA 0 appends
// (tag, globaltimer) after the barrier that ends a grid-wide phase; tag = level * 16 + kind.
enum { PK_FIRST2 = 0, PK_PRE = 1, PK_RESID = 2, PK_RESTRICT = 3, PK_TAIL = 4, PK_PROLONG = 5, PK_POST = 6, PK_DENSE = 7, PK_RZSUM = 8, PK_MATVEC = 9,
       PK_UPDATE = 10, PK_INIT = 11 };
__device__ __forceinline__ void prof_mark(unsigned long long *prof, int tag) {
  if (prof && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    const unsigned long long n = prof[0];
    if (n + 1 < (unsigned long long)kPcg2ProfCap) {
      prof[1 + 2 * n] = (unsigned long long)tag;
      prof[2 + 2 * n] = t;
      prof[0] = n + 1;
    }
  }
}

// Loads.  GRID scope: matrix data is immutable while the kernel runs (read-only path), vectors were written by other CTAs in
// the previous phase (read at L2).  CTA scope (tail): everything lives in shared memory or is private to CTA 0: plain loads.
template <bool GRID>
struct Ld {
  static __device__ __forceinline__ int i(const int *p) { return GRID ? __ldg(p) : *p; }
  static __device__ __forceinline__ double m(const double *p) { return GRID ? __ldg(p) : *p; }
  static __device__ __forceinline__ float mf(const float *p) { return GRID ? __ldg(p) : *p; }
  static __device__ __forceinline__ double v(const double *p) { return GRID ? __ldcg(p) : *p; }
};

// ---- multi-GPU (row-sharded levels): peer stores and the cross-GPU barrier ------------------------------------------------
// Every rank runs the same kernel on the same (replicated) matrices.  The rows of a sharded level are owned by the CTAs of all
// ranks together; what a CTA computes for its rows is stored locally AND into every peer's copy of the vector (NVLink stores
// into the peers' exchange arenas, mapped by CUDA IPC; the arenas have identical layouts, so a peer address is the local one
// plus a per-rank byte offset).  A cross-GPU barrier ends such a phase: CTA barrier, one system-scope fence per CTA, the CTAs
// arrive on a local counter, CTA 0 publishes the epoch to every peer's flag word and waits for theirs, then releases its grid.
struct XRt {                          // per-launch runtime state of the cross barrier, in shared memory (thread 0 only)
  unsigned long long epoch;           // barriers passed so far (continues across launches: the counters are monotonic)
  int aborted;
};
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ void xbarrier(const Pcg2Dist &D, XRt *rt) {
  __syncthreads();
  if (threadIdx.x == 0 && !rt->aborted) {
    // one system-scope fence per CTA, after the CTA barrier: it is cumulative over the stores (local and peer) the other threads
    // issued before the barrier -- the cooperative-groups grid-sync pattern.  (A fence by all 1024 threads, measured on 2 GPUs,
    // made a cross-GPU barrier cost ~10 us.)
    __threadfence_system();
    const unsigned long long e = ++rt->epoch;
    const unsigned long long t0 = gtime();
    const unsigned long long limit = 4000000000ull;   // 4 s: a peer that never arrives must not hang the GPU
    if (blockIdx.x != 0) {
      asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(D.xarrive) : "memory");
      unsigned long long cur;
      do {
        asm volatile("ld.acquire.gpu.u64 %0, [%1];" : "=l"(cur) : "l"(D.xrelease) : "memory");
        if (cur == ~0ull || gtime() - t0 > limit) {
          rt->aborted = 1;
          break;
        }
      } while (cur < e);
    } else {
      const unsigned int want = (unsigned int)((gridDim.x - 1) * e);   // monotonic arrival counter (wraps with the epoch)
      unsigned int got;
      bool ok = true;
      do {
        asm volatile("ld.acquire.gpu.u32 %0, [%1];" : "=r"(got) : "l"(D.xarrive) : "memory");
        if (gtime() - t0 > limit) ok = false;
      } while (ok && (int)(got - want) < 0);
      for (int q = 0; ok && q < D.nranks; ++q) {
        if (q == D.rank) continue;
        unsigned long long *pf = reinterpret_cast<unsigned long long *>(reinterpret_cast<char *>(D.flags + D.rank) + D.peer_off[q]);
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(pf), "l"(e) : "memory");
      }
      for (int q = 0; ok && q < D.nranks; ++q) {
        if (q == D.rank) continue;
        unsigned long long cur;
        do {
          asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(cur) : "l"(D.flags + q) : "memory");
          if (gtime() - t0 > limit) ok = false;
        } while (ok && cur < e);
      }
      if (!ok) rt->aborted = 1;
      const unsigned long long rel = ok ? e : ~0ull;   // ~0: tells the other CTAs to give up
      asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(D.xrelease), "l"(rel) : "memory");
    }
  }
  __syncthreads();
}

// where a phase stores a vector entry: locally, or locally and into every peer's copy
template <bool DIST>
struct Out {
  int npeer;
  long long off[kPcg2MaxRanks - 1];
  __device__ __forceinline__ void st(double *p, int i, double v) const {
    p[i] = v;
    if (DIST) {
      for (int q = 0; q < npeer; ++q) *reinterpret_cast<double *>(reinterpret_cast<char *>(p + i) + off[q]) = v;
    }
  }
};

template <bool GRID>
struct Scope {
  int cta, ncta, warp, nwarps, lane;
  unsigned int *bar;
  const Pcg2Dist *dist;   // != nullptr: this scope spans the CTAs of all ranks (cta = rank * CTAs per rank + local CTA) and
  XRt *xrt;               // its phases end with the cross-GPU barrier
  __device__ __forceinline__ void sync() const {
    if (GRID) {
      if (dist) xbarrier(*dist, xrt);
      else grid_barrier2(bar);
    } else {
      __syncthreads();
    }
  }
  // slices of M this CTA owns
  __device__ __forceinline__ void range(const SellMat &M, int &s0, int &s1) const {
    if (GRID) {
      s0 = cta * M.spc;
      s1 = min(M.nslices, s0 + M.spc);
    } else {
      s0 = 0;
      s1 = M.nslices;
    }
  }
  __device__ __forceinline__ int tid() const { return GRID ? (cta * nwarps + warp) * 32 + lane : warp * 32 + lane; }
  __device__ __forceinline__ int nthr() const { return GRID ? ncta * nwarps * 32 : nwarps * 32; }
};

// gathers of the right-hand vector entry j
template <bool GRID>
struct GatherX {
  const double *x;
  __device__ __forceinline__ double operator()(int j) const { return Ld<GRID>::v(x + j); }
};
template <bool GRID>
struct GatherScaled {   // b_j * idiag_j
  const double *b, *idiag;
  __device__ __forceinline__ double operator()(int j) const { return Ld<GRID>::v(b + j) * Ld<GRID>::m(idiag + j); }
};
template <bool GRID>
struct GatherAxpy {     // z_j + beta p_j
  const double *z, *p;
  double beta;
  __device__ __forceinline__ double operator()(int j) const { return Ld<GRID>::v(z + j) + beta * Ld<GRID>::v(p + j); }
};

// sum_k val[k] * g(idx[k]) over the entries of row (32 s + lane), in column order; four entries in flight
template <bool GRID, bool F32, class G>
__device__ __forceinline__ double sell_row(const SellMat &A, int s, int lane, const G &g) {
  const int b = Ld<GRID>::i(A.soff + s), e = Ld<GRID>::i(A.soff + s + 1);
  double acc = 0.0;
  int k = b + lane;
  for (; k + 96 < e; k += 128) {
    const int j0 = Ld<GRID>::i(A.idx + k), j1 = Ld<GRID>::i(A.idx + k + 32), j2 = Ld<GRID>::i(A.idx + k + 64), j3 = Ld<GRID>::i(A.idx + k + 96);
    double v0, v1, v2, v3;
    if (F32) {
      v0 = (double)Ld<GRID>::mf(A.valf + k);
      v1 = (double)Ld<GRID>::mf(A.valf + k + 32);
      v2 = (double)Ld<GRID>::mf(A.valf + k + 64);
      v3 = (double)Ld<GRID>::mf(A.valf + k + 96);
    } else {
      v0 = Ld<GRID>::m(A.val + k);
      v1 = Ld<GRID>::m(A.val + k + 32);
      v2 = Ld<GRID>::m(A.val + k + 64);
      v3 = Ld<GRID>::m(A.val + k + 96);
    }
    const double x0 = g(j0), x1 = g(j1), x2 = g(j2), x3 = g(j3);
    acc += v0 * x0;
    acc += v1 * x1;
    acc += v2 * x2;
    acc += v3 * x3;
  }
  if (k < e) {   // up to three entries left: all loads issued before the first use (warp-uniform predicates)
    const bool h1 = k + 32 < e, h2 = k + 64 < e;
    const int j0 = Ld<GRID>::i(A.idx + k), j1 = h1 ? Ld<GRID>::i(A.idx + k + 32) : j0, j2 = h2 ? Ld<GRID>::i(A.idx + k + 64) : j0;
    double v0, v1 = 0.0, v2 = 0.0;
    if (F32) {
      v0 = (double)Ld<GRID>::mf(A.valf + k);
      if (h1) v1 = (double)Ld<GRID>::mf(A.valf + k + 32);
      if (h2) v2 = (double)Ld<GRID>::mf(A.valf + k + 64);
    } else {
      v0 = Ld<GRID>::m(A.val + k);
      if (h1) v1 = Ld<GRID>::m(A.val + k + 32);
      if (h2) v2 = Ld<GRID>::m(A.val + k + 64);
    }
    const double x0 = g(j0), x1 = h1 ? g(j1) : 0.0, x2 = h2 ? g(j2) : 0.0;
    acc += v0 * x0;
    if (h1) acc += v1 * x1;
    if (h2) acc += v2 * x2;
  }
  // lanes of a row group: fixed-order tree, result in the group's first lane (all lanes of the warp take part)
  for (int o = A.lpr >> 1; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  return acc;
}
// row served by `lane` of the warp working on slice s, and whether this lane writes the row's result
__device__ __forceinline__ int sell_rowof(const SellMat &A, int s, int lane, bool &lead) {
  const int row = s * (32 / A.lpr) + lane / A.lpr;
  lead = (lane % A.lpr == 0) && row < A.rows;
  return row;
}
template <bool GRID, class G>
__device__ __forceinline__ double sell_row_any(const SellMat &A, int s, int lane, const G &g) {
  return A.valf ? sell_row<GRID, true>(A, s, lane, g) : sell_row<GRID, false>(A, s, lane, g);
}

// y = alpha * M x + (y0 ? y0 : 0)      (y may alias y0; y must not alias x)
// ys != nullptr: also ys = y .* yscale (the pre-scaled right-hand side the next level's first smoothing pass gathers)
template <bool GRID, bool DIST>
__device__ void ph_spmv(const Scope<GRID> &sc, const Out<DIST> &o, const SellMat &M, const double *x, const double *y0, double alpha, double *y,
                        double *ys = nullptr, const double *yscale = nullptr) {
  int s0, s1;
  sc.range(M, s0, s1);
  const GatherX<GRID> g{x};
  for (int s = s0 + sc.warp; s < s1; s += sc.nwarps) {
    bool lead;
    const int row = sell_rowof(M, s, sc.lane, lead);
    const double acc = sell_row_any<GRID>(M, s, sc.lane, g);
    if (lead) {
      const double v = alpha * acc + (y0 ? Ld<GRID>::v(y0 + row) : 0.0);
      o.st(y, row, v);
      if (ys) o.st(ys, row, v * Ld<GRID>::m(yscale + row));
    }
  }
}

// Smoothing.  Chebyshev on [lam/ratio, lam] with diagonal scaling (3-term recurrence; theta = (a+b)/2, delta = (b-a)/2,
// sigma = theta/delta, rho_0 = 1/sigma, rho_k = 1/(2 sigma - rho_{k-1}); d_0 = D^-1 r_0 / theta,
// d_k = rho_k rho_{k-1} d_{k-1} + (2 rho_k / delta) D^-1 r_k, x_{k+1} = x_k + d_k) -- or l1-Jacobi, which is the same
// update with th_inv = 1, c_dd = 0, c_dr = 1 and the l1 row sums in place of the diagonal.
struct Cheb {
  double th_inv, sigma, delta;
  __device__ __forceinline__ Cheb(double lam, double ratio) {
    const double b = lam, a = lam / ratio;
    const double theta = 0.5 * (a + b);
    delta = 0.5 * (b - a);
    sigma = theta / delta;
    th_inv = 1.0 / theta;
  }
  __device__ __forceinline__ double step(double rho_prev, double &c_dd, double &c_dr) const {
    const double rho = 1.0 / (2.0 * sigma - rho_prev);
    c_dd = rho * rho_prev;
    c_dr = 2.0 * rho / delta;
    return rho;
  }
};

// steps 0 and 1 from x = 0 in one pass: d0 = th_inv D^-1 b; r1 = b - A d0; d1 = c_dd d0 + c_dr D^-1 r1; x = d0 + d1
// bs = b .* idiag is written by whoever produced b (restriction, PCG update), so that the row sums gather ONE vector
template <bool GRID, bool DIST>
__device__ void ph_first2(const Scope<GRID> &sc, const Out<DIST> &o, const SellMat &A, const double *idiag, const double *b, const double *bs, double *xnew, double *d,
                          double th_inv, double c_dd, double c_dr) {
  int s0, s1;
  sc.range(A, s0, s1);
  const GatherX<GRID> g{bs};
  for (int s = s0 + sc.warp; s < s1; s += sc.nwarps) {
    bool lead;
    const int row = sell_rowof(A, s, sc.lane, lead);
    const double acc = sell_row_any<GRID>(A, s, sc.lane, g);
    if (lead) {
      const double di = Ld<GRID>::m(idiag + row), bi = Ld<GRID>::v(b + row);
      const double d0 = th_inv * bi * di;
      const double d1 = c_dd * d0 + c_dr * (bi - th_inv * acc) * di;
      o.st(xnew, row, d0 + d1);
      d[row] = d1;   // the recurrence vector is only ever read by its owner
    }
  }
}

// one step on an existing iterate: r = b - A x; d = (first ? th_inv D^-1 r : c_dd d + c_dr D^-1 r); xnew = x + d;
// returns this thread's share of sum_i dotw[i] xnew[i] (0 if dotw == nullptr)
template <bool GRID, bool DIST>
__device__ double ph_step(const Scope<GRID> &sc, const Out<DIST> &o, const SellMat &A, const double *idiag, const double *b, const double *x, double *xnew, double *d,
                          bool first, double th_inv, double c_dd, double c_dr, const double *dotw) {
  int s0, s1;
  sc.range(A, s0, s1);
  const GatherX<GRID> g{x};
  double part = 0.0;
  for (int s = s0 + sc.warp; s < s1; s += sc.nwarps) {
    bool lead;
    const int row = sell_rowof(A, s, sc.lane, lead);
    const double acc = sell_row_any<GRID>(A, s, sc.lane, g);
    if (lead) {
      const double rr = (Ld<GRID>::v(b + row) - acc) * Ld<GRID>::m(idiag + row);
      const double dn = first ? th_inv * rr : c_dd * d[row] + c_dr * rr;
      const double v = Ld<GRID>::v(x + row) + dn;
      d[row] = dn;
      o.st(xnew, row, v);
      if (dotw) part += Ld<GRID>::v(dotw + row) * v;
    }
  }
  return part;
}

// x = Minv b (dense, row-major), one warp per row
template <bool GRID>
__device__ void ph_dense(const Scope<GRID> &sc, const double *Minv, int m, const double *b, double *x) {
  const int w0 = GRID ? sc.cta * sc.nwarps + sc.warp : sc.warp;
  const int nw = GRID ? sc.ncta * sc.nwarps : sc.nwarps;
  for (int row = w0; row < m; row += nw) {
    const double *r = Minv + (size_t)row * m;
    double s = 0.0;
    for (int j = sc.lane; j < m; j += 32) s += __ldg(r + j) * Ld<GRID>::v(b + j);
    s = warp_sum2(s);
    if (sc.lane == 0) x[row] = s;
  }
}

// block-wide sum, result broadcast to every thread (fixed order)
__device__ __forceinline__ double block_sum_bcast2(double v) {
  __shared__ double wsum[32];
  __shared__ double total;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum2(v);
  __syncthreads();   // protects wsum / total from the previous call
  if (lane == 0) wsum[wid] = v;
  __syncthreads();
  if (wid == 0) {
    double x = lane < nw ? wsum[lane] : 0.0;
    x = warp_sum2(x);
    if (lane == 0) total = x;
  }
  __syncthreads();
  return total;
}

// deposit this CTA's partial, grid barrier, then every CTA sums all partials in the same fixed order
__device__ __forceinline__ double grid_sum2(double part, double *slot, unsigned int *bar) {
  const double bs = block_sum_bcast2(part);
  if (threadIdx.x == 0) slot[blockIdx.x] = bs;
  grid_barrier2(bar);
  double v = 0.0;
  for (unsigned int b = threadIdx.x; b < gridDim.x; b += blockDim.x) v += __ldcg(slot + b);
  return block_sum_bcast2(v);
}

struct VcArgs {
  int nlev, nbig, bottom_dense, nu, nu_bottom, smoother;
  double cheb_ratio;
  const double *dense_inv;
  unsigned long long *prof;
};

// V-cycle over the active levels [k0, k1) in scope `sc`; btop: right-hand side of level k0; lev: the level table of this scope
// (the plan's for the grid, CTA 0's shared-memory copy for the tail).  After the down-sweep of level k1-1 the coarser levels
// are run by `tail` (GRID scope only).  The result is in lev[k0].x: the ping-pong between x and x2 starts on the buffer that
// makes the last sweep land in x, so no pointer is ever swapped and every CTA agrees on where results live.
// dot_top != nullptr: returns this thread's share of sum dot_top[i] x[i] on level k0, and the barrier after the last sweep is
// left to the caller's grid_sum.
// Where level k's down-sweep starts and which diagonal it scales with: `cur` receives the first smoothing pass, `oth` is free
// until the next sweep -- it holds bs = b .* idg for that pass.  The producer of b (restriction / PCG update) and the consumer
// (ph_first2) must agree, hence one function.
struct SmoothBufs {
  double *cur, *oth;
  const double *idg;
  bool two;   // the level starts with the fused two-step pass (ph_first2), i.e. it reads bs
};
__device__ __forceinline__ SmoothBufs smooth_bufs(const VcArgs &P, const Pcg2Level &Lv, int k) {
  const bool last = (k == P.nlev - 1);
  const bool cheb = (P.smoother == 1) && !last;
  const int want = last ? P.nu_bottom : P.nu;
  const int done = (want >= 2) ? 2 : 1;
  const int npre = want - done, npost = last ? 0 : P.nu;
  SmoothBufs B;
  B.cur = ((npre + npost) & 1) ? Lv.x2 : Lv.x;
  B.oth = ((npre + npost) & 1) ? Lv.x : Lv.x2;
  B.idg = cheb ? Lv.idiag : Lv.dinv;
  B.two = (done == 2) && !(last && P.bottom_dense);
  return B;
}

// DIST: levels [0, nshard) are row-sharded over the ranks: their phases run in scope `scx` (all ranks' CTAs), store through
// `ox` (local + peers) and end with the cross-GPU barrier; the other levels are replicated (scope `sc`, local stores `ol`).
// A phase is classified by the level whose rows it WRITES.
template <bool GRID, bool DIST, class Tail>
__device__ double vcycle(const VcArgs &P, const Pcg2Level *lev, const Scope<GRID> &sc, const Scope<GRID> &scx, const Out<DIST> &ol, const Out<DIST> &ox,
                         int nshard, int k0, int k1, const double *btop, const double *dot_top, const Tail &tail) {
  double part = 0.0;
  // ---- down
  for (int k = k0; k < k1; ++k) {
    const Pcg2Level &Lv = lev[k];
    const bool sh = DIST && k < nshard, shc = DIST && (k + 1) < nshard;   // this level / the next coarser one sharded
    const Scope<GRID> &S = sh ? scx : sc;
    const Out<DIST> &O = sh ? ox : ol;
    const double *bk = (k == k0) ? btop : Lv.b;
    const bool last = (k == P.nlev - 1);
    if (last && P.bottom_dense) {
      ph_dense<GRID>(sc, P.dense_inv, Lv.m, bk, Lv.x);
      sc.sync();
      if (GRID) prof_mark(P.prof, k * 16 + PK_DENSE);
      continue;
    }
    const bool cheb = (P.smoother == 1) && !last;   // an iterated bottom level keeps l1-Jacobi
    const double *idg = cheb ? Lv.idiag : Lv.dinv;
    const int want = last ? P.nu_bottom : P.nu;
    const int done = (want >= 2) ? 2 : 1;
    const int npre = want - done, npost = last ? 0 : P.nu;
    double *cur = ((npre + npost) & 1) ? Lv.x2 : Lv.x, *oth = ((npre + npost) & 1) ? Lv.x : Lv.x2;
    const Cheb C(cheb ? *Lv.lam : 1.0, P.cheb_ratio);
    double rho = 1.0 / C.sigma, c_dd = 0.0, c_dr = 1.0;
    const double th_inv = cheb ? C.th_inv : 1.0;
    if (done == 2) {
      if (cheb) rho = C.step(rho, c_dd, c_dr);
      ph_first2<GRID, DIST>(S, O, Lv.A, idg, bk, oth, cur, Lv.r, th_inv, c_dd, c_dr);   // oth holds b .* idg (smooth_bufs)
    } else {
      for (int i = S.tid(); i < Lv.m; i += S.nthr()) {
        const double d0 = th_inv * Ld<GRID>::v(bk + i) * Ld<GRID>::m(idg + i);
        O.st(cur, i, d0);
        O.st(Lv.r, i, d0);
      }
    }
    S.sync();
    if (GRID) prof_mark(P.prof, k * 16 + PK_FIRST2);
    for (int it = 0; it < npre; ++it) {
      if (cheb) rho = C.step(rho, c_dd, c_dr);
      // l1-Jacobi: every sweep is a "first" step (x += dinv (b - A x))
      ph_step<GRID, DIST>(S, O, Lv.A, idg, bk, cur, oth, Lv.r, !cheb, th_inv, c_dd, c_dr, nullptr);
      S.sync();
      if (GRID) prof_mark(P.prof, k * 16 + PK_PRE);
      double *t = cur;
      cur = oth;
      oth = t;
    }
    if (!last) {
      ph_spmv<GRID, DIST>(S, O, Lv.A, cur, bk, -1.0, Lv.r);
      S.sync();
      if (GRID) prof_mark(P.prof, k * 16 + PK_RESID);
      {
        const SmoothBufs nb = smooth_bufs(P, lev[k + 1], k + 1);
        const Scope<GRID> &Sc = shc ? scx : sc;   // the restriction writes rows of level k + 1
        ph_spmv<GRID, DIST>(Sc, shc ? ox : ol, Lv.Tt, Lv.r, nullptr, 1.0, lev[k + 1].b, nb.two ? nb.oth : nullptr, nb.idg);
        Sc.sync();
      }
      if (GRID) prof_mark(P.prof, k * 16 + PK_RESTRICT);
    }
  }
  // ---- coarser levels
  if (GRID && k1 < P.nlev) {
    tail();
    sc.sync();
    prof_mark(P.prof, k1 * 16 + PK_TAIL);
  }
  // ---- up
  for (int k = k1 - 1; k >= k0; --k) {
    if (k == P.nlev - 1) continue;   // bottom level: nothing coarser
    const Pcg2Level &Lv = lev[k];
    const bool sh = DIST && k < nshard;
    const Scope<GRID> &S = sh ? scx : sc;
    const Out<DIST> &O = sh ? ox : ol;
    const double *bk = (k == k0) ? btop : Lv.b;
    const int want = P.nu;
    const int done = (want >= 2) ? 2 : 1;
    const int npre = want - done, npost = P.nu;
    const bool start_x2 = ((npre + npost) & 1) != 0;
    const bool cur_x2 = start_x2 != ((npre & 1) != 0);
    double *cur = cur_x2 ? Lv.x2 : Lv.x, *oth = cur_x2 ? Lv.x : Lv.x2;
    ph_spmv<GRID, DIST>(S, O, Lv.T, lev[k + 1].x, cur, 1.0, cur);   // x += T xc (row-local)
    S.sync();
    if (GRID) prof_mark(P.prof, k * 16 + PK_PROLONG);
    const bool cheb = (P.smoother == 1);
    const double *idg = cheb ? Lv.idiag : Lv.dinv;
    const Cheb C(cheb ? *Lv.lam : 1.0, P.cheb_ratio);
    const double th_inv = cheb ? C.th_inv : 1.0;
    double rho = 1.0 / C.sigma, c_dd = 0.0, c_dr = 1.0;
    for (int it = 0; it < npost; ++it) {
      const bool fin = (it == npost - 1) && (k == k0) && (dot_top != nullptr);
      if (cheb && it > 0) rho = C.step(rho, c_dd, c_dr);
      part += ph_step<GRID, DIST>(S, O, Lv.A, idg, bk, cur, oth, Lv.r, !cheb || it == 0, th_inv, c_dd, c_dr, fin ? dot_top : nullptr);
      if (!fin) {
        S.sync();
        if (GRID) prof_mark(P.prof, k * 16 + PK_POST);
      }
      double *t = cur;
      cur = oth;
      oth = t;
    }
  }
  return part;
}

struct NoTail {
  __device__ __forceinline__ void operator()() const {}
};

constexpr int kTailMaxLevels = 12;

// copy n elements global -> shared (CTA-wide), return the shared pointer
template <class T>
__device__ __forceinline__ T *to_smem(unsigned char *&cur, const T *src, int n) {
  T *dst = reinterpret_cast<T *>(cur);
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
  cur += ((size_t)n * sizeof(T) + 15) & ~(size_t)15;
  return dst;
}
template <class T>
__device__ __forceinline__ T *smem_alloc(unsigned char *&cur, int n) {
  T *dst = reinterpret_cast<T *>(cur);
  cur += ((size_t)n * sizeof(T) + 15) & ~(size_t)15;
  return dst;
}
__device__ __forceinline__ void sell_to_smem(unsigned char *&cur, SellMat &M) {
  if (M.nslices == 0) return;
  M.soff = to_smem(cur, M.soff, M.nslices + 1);
  M.idx = to_smem(cur, M.idx, M.entries);
  M.valf = to_smem(cur, M.valf, M.entries);   // the tail is preconditioner-only: FP32 values (8 bytes per entry) so that more levels fit
  M.val = nullptr;
}

template <bool DIST>
__global__ void __launch_bounds__(kPcg2Threads, 1) k_pcg2(const Pcg2Plan *plan_g, double rtol2, int maxit, int stall_window) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  __shared__ Pcg2Plan P;
  __shared__ double s_e[5];
  __shared__ XRt s_xrt;
  __shared__ Pcg2Level TL[kTailMaxLevels];   // CTA 0: tail levels with shared-memory matrices and vectors, index k - nbig
  {
    const uint64_t *src = reinterpret_cast<const uint64_t *>(plan_g);
    uint64_t *dst = reinterpret_cast<uint64_t *>(&P);
    for (int i = threadIdx.x; i < (int)(sizeof(Pcg2Plan) / sizeof(uint64_t)); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const int ntail = P.nlev - P.nbig;
  const bool tail_smem = (P.tail_smem_bytes > 0) && ntail > 0 && ntail <= kTailMaxLevels;
  if (blockIdx.x == 0 && ntail > 0 && ntail <= kTailMaxLevels) {
    if (threadIdx.x < ntail) TL[threadIdx.x] = P.lev[P.nbig + threadIdx.x];
    __syncthreads();
    if (tail_smem) {
      unsigned char *cur = dyn_smem;
      for (int q = 0; q < ntail; ++q) {
        // every thread performs the same pointer arithmetic; the copies are CTA-wide
        SellMat A = TL[q].A, T = TL[q].T, Tt = TL[q].Tt;
        if (!(q == ntail - 1 && P.bottom_dense)) sell_to_smem(cur, A);   // a dense bottom level never touches its sparse matrix
        sell_to_smem(cur, T);
        sell_to_smem(cur, Tt);
        const int m = TL[q].m;
        const double *idg = to_smem(cur, TL[q].idiag, m);
        const double *dnv = to_smem(cur, TL[q].dinv, m);
        double *vb = smem_alloc<double>(cur, m), *vx = smem_alloc<double>(cur, m), *vx2 = smem_alloc<double>(cur, m), *vr = smem_alloc<double>(cur, m);
        __syncthreads();
        if (threadIdx.x == 0) {
          TL[q].A = A;
          TL[q].T = T;
          TL[q].Tt = Tt;
          TL[q].idiag = idg;
          TL[q].dinv = dnv;
          TL[q].b = vb;
          TL[q].x = vx;
          TL[q].x2 = vx2;
          TL[q].r = vr;
        }
        __syncthreads();
      }
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const Scope<true> sc{(int)blockIdx.x, (int)gridDim.x, warp, nwarps, lane, P.bar, nullptr, nullptr};
  // multi-GPU: the scope of the sharded levels spans the CTAs of all ranks
  const int nshard = DIST ? P.dist.nshard : 0;
  const Scope<true> scx{DIST ? P.dist.rank * (int)gridDim.x + (int)blockIdx.x : (int)blockIdx.x, DIST ? P.dist.nranks * (int)gridDim.x : (int)gridDim.x,
                        warp, nwarps, lane, P.bar, DIST ? &P.dist : nullptr, DIST ? &s_xrt : nullptr};
  Out<DIST> ol, ox;
  ol.npeer = 0;
  ox.npeer = 0;
  if (DIST) {
    for (int q = 0; q < P.dist.nranks; ++q)
      if (q != P.dist.rank) ox.off[ox.npeer++] = P.dist.peer_off[q];
    if (threadIdx.x == 0) {
      unsigned long long e0;
      asm volatile("ld.acquire.gpu.u64 %0, [%1];" : "=l"(e0) : "l"(P.dist.xrelease) : "memory");
      s_xrt.epoch = e0;   // stable: the previous launch has completed on every CTA
      s_xrt.aborted = 0;
    }
    __syncthreads();
  }
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthr = (int64_t)gridDim.x * blockDim.x;
  const int m = P.lev[0].m;
  double *slot0 = P.partials, *slot1 = P.partials + kPcg2MaxGrid, *slot2 = P.partials + 2 * kPcg2MaxGrid;
  // rows of the top level this CTA owns (DIST: the update of x and r is row-owned, like every phase of a sharded level)
  const bool top_sh = DIST && nshard > 0;
  int own0 = 0, own1 = 0;
  if (top_sh) {
    int s0, s1;
    scx.range(P.lev[0].A, s0, s1);
    const int rps = 32 / P.lev[0].A.lpr;
    own0 = min(m, s0 * rps);
    own1 = min(m, max(s0, s1) * rps);
  }
  // sum over the whole (multi-GPU) grid: every CTA deposits its partial in every rank's slot array, one cross barrier, then
  // every CTA of every rank adds all partials in the same order
  auto xsum = [&](double part, double *slot) -> double {
    if (!top_sh) return grid_sum2(part, slot, P.bar);
    const double bs = block_sum_bcast2(part);
    if (threadIdx.x == 0) ox.st(slot, scx.cta, bs);
    scx.sync();
    double v = 0.0;
    for (int b = threadIdx.x; b < scx.ncta; b += blockDim.x) v += __ldcg(slot + b);
    return block_sum_bcast2(v);
  };
  const VcArgs VA{P.nlev, P.nbig, P.bottom_dense, P.nu, P.nu_bottom, P.smoother, P.cheb_ratio, P.dense_inv, P.prof};
  if (P.prof && tid == 0) P.prof[0] = 0;

  // the tail: CTA 0 alone.  With shared-memory vectors the entry right-hand side is copied in (it was written by the whole
  // grid) and the result copied out to the global vector the grid prolongates from.
  auto tail = [&]() {
    if (blockIdx.x != 0) return;
    const Scope<false> cta{0, 1, warp, nwarps, lane, nullptr, nullptr, nullptr};
    const int nb = P.nbig;
    const Pcg2Level *tl = TL - nb;   // indexed by level
    {
      // the entry right-hand side was written by the whole grid: copy it into CTA 0's vector (shared memory) together with its
      // pre-scaled copy for the first smoothing pass
      const SmoothBufs sb = smooth_bufs(VA, TL[0], nb);
      const double *gb = P.lev[nb].b;
      for (int i = threadIdx.x; i < TL[0].m; i += blockDim.x) {
        const double v = __ldcg(gb + i);
        if (tail_smem) TL[0].b[i] = v;
        if (sb.two) sb.oth[i] = v * sb.idg[i];
      }
      __syncthreads();
    }
    const Out<false> lo{0, {}};
    vcycle<false, false>(VA, tl, cta, cta, lo, lo, 0, nb, P.nlev, TL[0].b, nullptr, NoTail());
    if (tail_smem) {
      double *gx = P.lev[nb].x;
      for (int i = threadIdx.x; i < TL[0].m; i += blockDim.x) gx[i] = TL[0].x[i];
    }
  };

  // the p / p2 ping-pong lives in registers
  double *pv = P.p, *pv2 = P.p2;
  const SmoothBufs top_sb = smooth_bufs(VA, P.lev[0], 0);   // r .* idiag for the top level's first smoothing pass goes to top_sb.oth
  double part = 0.0;
  for (int64_t i = tid; i < m; i += nthr) {
    const double bi = P.b[i];
    P.x[i] = 0.0;
    pv[i] = 0.0;
    P.r[i] = bi;
    if (top_sb.two) top_sb.oth[i] = bi * __ldg(top_sb.idg + i);
    part += bi * bi;
  }
  const double bb = grid_sum2(part, slot0, P.bar);
  // multi-GPU: no peer store before every rank is inside this launch (a peer may still be running the kernels in front of
  // it -- the power iteration uses the level vectors of the exchange arena as scratch)
  if (top_sh) scx.sync();
  prof_mark(P.prof, PK_INIT);
  int it = 0;
  double rr = bb, status = 1.0, e_tot = 0.0, e_last4 = 0.0;
  if (bb > 0.0 && isfinite(bb)) {
    const double target = rtol2 * bb;
    double rz_old = 1.0, best = bb;
    int since_best = 0;
    // energy bookkeeping: for CG from x = 0, b.x_k = |x_k|_A^2 = sum_j alpha_j (r.z)_j grows monotonically to b.A^-1 b -- the
    // Newton decrement the caller needs; e_m4 is its value four iterations ago
    // (kept by thread 0 in shared memory: registers are scarce at 1024 threads per CTA)
    if (threadIdx.x == 0) s_e[0] = s_e[1] = s_e[2] = s_e[3] = s_e[4] = 0.0;
    const Pcg2Level &top = P.lev[0];
    SellMat Atop = top.A;
    Atop.valf = nullptr;   // the PCG operator is always FP64
    while (it < maxit) {
      // z = M^{-1} r, with r.z accumulated in the last smoothing sweep of the top level
      const bool single = (P.nlev == 1);
      double prz = vcycle<true, DIST>(VA, P.lev, sc, scx, ol, ox, nshard, 0, P.nbig, P.r, single ? nullptr : P.r, tail);
      const double *z = top.x;
      if (single) {   // one-level "hierarchy": no up-sweep ran, take the dot here
        prz = 0.0;
        for (int64_t i = tid; i < m; i += nthr) prz += P.r[i] * __ldcg(z + i);
      }
      const double rz = xsum(prz, slot1);
      prof_mark(P.prof, PK_RZSUM);
      const double beta = rz / rz_old;
      rz_old = rz;
      // p2 = z + beta p;  Ap = A p2 (neighbour values formed on the fly);  p2.Ap
      double ppap = 0.0;
      {
        int s0, s1;
        (top_sh ? scx : sc).range(Atop, s0, s1);
        const GatherAxpy<true> g{z, pv, beta};
        for (int s = s0 + warp; s < s1; s += nwarps) {
          bool lead;
          const int row = sell_rowof(Atop, s, lane, lead);
          const double acc = sell_row<true, false>(Atop, s, lane, g);
          if (lead) {
            const double pn = __ldcg(z + row) + beta * __ldcg(pv + row);
            if (top_sh) ox.st(pv2, row, pn);   // the next iteration's mat-vec gathers p from every rank's rows
            else pv2[row] = pn;
            P.Ap[row] = acc;
            ppap += pn * acc;
          }
        }
      }
      const double pAp = xsum(ppap, slot2);
      prof_mark(P.prof, PK_MATVEC);
      {
        double *t = pv;
        pv = pv2;
        pv2 = t;
      }
      ++it;
      if (!(pAp > 0.0) || !isfinite(pAp)) {
        status = -1.0;
        break;
      }
      const double alpha = rz / pAp;
      if (threadIdx.x == 0) {
        s_e[(it - 1) & 3] = s_e[4];   // total before this iteration; the slot it overwrites is four iterations old
        s_e[4] += alpha * rz;
      }
      double prr = 0.0;
      if (top_sh) {
        for (int i = own0 + (int)threadIdx.x; i < own1; i += (int)blockDim.x) {
          P.x[i] += alpha * __ldcg(pv + i);
          const double ri = P.r[i] - alpha * __ldcg(P.Ap + i);
          P.r[i] = ri;
          if (top_sb.two) ox.st(top_sb.oth, i, ri * __ldg(top_sb.idg + i));
          prr += ri * ri;
        }
      } else {
        for (int64_t i = tid; i < m; i += nthr) {
          P.x[i] += alpha * __ldcg(pv + i);
          const double ri = P.r[i] - alpha * __ldcg(P.Ap + i);
          P.r[i] = ri;
          if (top_sb.two) top_sb.oth[i] = ri * __ldg(top_sb.idg + i);
          prr += ri * ri;
        }
      }
      rr = xsum(prr, slot0);
      prof_mark(P.prof, PK_UPDATE);
      if (!isfinite(rr)) {
        status = -1.0;
        break;
      }
      if (rr <= target) break;
      if (rr < best * 0.999) {
        best = rr;
        since_best = 0;
      } else if (++since_best >= stall_window) {
        status = 2.0;   // stagnation at the attainable accuracy (above the requested tolerance)
        break;
      }
    }
    if (status == 1.0 && rr > target) status = 3.0;   // iteration limit
    if (threadIdx.x == 0) {
      e_tot = s_e[4];
      e_last4 = s_e[4] - (it >= 4 ? s_e[it & 3] : 0.0);   // slot (it & 3) holds the total before iteration it - 3
    }
  }
  if (top_sh) {   // every rank needs the whole direction: owners publish their rows of x
    for (int i = own0 + (int)threadIdx.x; i < own1; i += (int)blockDim.x) ox.st(P.x, i, P.x[i]);
    scx.sync();
    if (s_xrt.aborted) status = -3.0;   // a peer never arrived at a cross-GPU barrier
  }
  if (tid == 0) {
    P.out[kPcg2OutIters] = (double)it;
    P.out[kPcg2OutRR] = rr;
    P.out[kPcg2OutStatus] = status;
    P.out[kPcg2OutBB] = bb;
    P.out[kPcg2OutEnergy] = e_tot;
    P.out[kPcg2OutEnergyLast4] = e_last4;
  }
}

// ---- lambda_max(D^-1 A) by power iteration, all levels of a plan in ONE cooperative launch ---------------------------------
// The levels are independent, so one phase serves them all: y = D^-1 A v (+ this CTA's share of |y|^2 per level), grid barrier,
// every CTA adds the partials in the same order, v = y / |y|, grid barrier.  The vector v (Pcg2Level::pw) persists between
// launches (warm start across Newton iterations).  lam <- min(lam, safety |D^-1 A v|): the Gershgorin bound k_l1diag left in
// lam stays an upper clamp.
__global__ void __launch_bounds__(kPcg2Threads, 1) k_lambda_power(const Pcg2Plan *plan_g, int iters, double safety) {
  __shared__ Pcg2Plan P;
  {
    const uint64_t *src = reinterpret_cast<const uint64_t *>(plan_g);
    uint64_t *dst = reinterpret_cast<uint64_t *>(&P);
    for (int i = threadIdx.x; i < (int)(sizeof(Pcg2Plan) / sizeof(uint64_t)); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const Scope<true> sc{(int)blockIdx.x, (int)gridDim.x, warp, nwarps, lane, P.bar};
  const int nl = P.nlev - (P.bottom_dense ? 1 : 0);   // a dense bottom level has no smoother
  for (int it = 0; it < iters; ++it) {
    for (int q = 0; q < nl; ++q) {
      const Pcg2Level &Lv = P.lev[q];
      SellMat A = Lv.A;
      A.valf = nullptr;
      // every level is shared by the whole grid here, whatever the solve kernel does with it
      const int spc = (A.nslices + (int)gridDim.x - 1) / (int)gridDim.x;
      const int s0 = (int)blockIdx.x * spc, s1 = min(A.nslices, s0 + spc);
      const GatherX<true> g{Lv.pw};
      double part = 0.0;
      for (int s = s0 + warp; s < s1; s += nwarps) {
        bool lead;
        const int row = sell_rowof(A, s, lane, lead);
        const double acc = sell_row<true, false>(A, s, lane, g);
        if (lead) {
          const double y = acc * __ldg(Lv.idiag + row);
          Lv.r[row] = y;
          part += y * y;
        }
      }
      const double bs = block_sum_bcast2(part);
      if (threadIdx.x == 0) P.partials[(size_t)q * gridDim.x + blockIdx.x] = bs;
    }
    grid_barrier2(P.bar);
    for (int q = 0; q < nl; ++q) {
      const Pcg2Level &Lv = P.lev[q];
      double v = 0.0;
      for (unsigned int b = threadIdx.x; b < gridDim.x; b += blockDim.x) v += __ldcg(P.partials + (size_t)q * gridDim.x + b);
      const double nrm = sqrt(block_sum_bcast2(v));
      const double inv = nrm > 0.0 ? 1.0 / nrm : 0.0;
      for (int i = (int)(blockIdx.x * blockDim.x + threadIdx.x); i < Lv.m; i += (int)(gridDim.x * blockDim.x)) Lv.pw[i] = __ldcg(Lv.r + i) * inv;
      if (it == iters - 1 && blockIdx.x == 0 && threadIdx.x == 0 && nrm > 0.0 && isfinite(nrm)) {
        double *lam = const_cast<double *>(Lv.lam);
        const double est = safety * nrm;
        if (est < *lam) *lam = est;
      }
    }
    grid_barrier2(P.bar);
  }
}

// ---- sliced-ELL construction ---------------------------------------------------------------------------------------
__global__ void k_sell_widths(int64_t rows, int lpr, const int64_t *__restrict__ ptr, int *width) {
  const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // one warp per slice
  const int lane = threadIdx.x & 31;
  const int rps = 32 / lpr;
  const int64_t nsl = (rows + rps - 1) / rps;
  if (gw >= nsl) return;
  const int64_t row = gw * rps + lane / lpr;
  int len = row < rows ? (int)(ptr[row + 1] - ptr[row]) : 0;
  len = (len + lpr - 1) / lpr;   // entries per lane of the row's group
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
  if (lane == 0) width[gw] = len;
}

__global__ void k_sell_pattern(int64_t rows, int lpr, const int64_t *__restrict__ ptr, const int32_t *__restrict__ cidx, const int *__restrict__ soff,
                               int *idx, int *src) {
  const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int rps = 32 / lpr, sub = lane % lpr;
  const int64_t nsl = (rows + rps - 1) / rps;
  if (gw >= nsl) return;
  const int64_t row = gw * rps + lane / lpr;
  const int b = soff[gw], w = (soff[gw + 1] - b) / 32;
  const int64_t p0 = row < rows ? ptr[row] : 0;
  const int len = row < rows ? (int)(ptr[row + 1] - p0) : 0;
  const int pad = len > 0 ? cidx[p0] : 0;
  for (int j = 0; j < w; ++j) {
    const int e = b + 32 * j + lane;
    const int k = j * lpr + sub;   // the row's entries are dealt round-robin to the lanes of its group
    if (k < len) {
      idx[e] = cidx[p0 + k];
      src[e] = (int)(p0 + k);
    } else {
      idx[e] = pad;   // a column the row (or the matrix) really has: the gather stays in bounds for rectangular matrices too
      src[e] = -1;
    }
  }
}

__global__ void k_sell_values(int entries, const int *__restrict__ src, const double *__restrict__ cval, double *val, float *valf) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= entries) return;
  const int q = src[e];
  const double v = q >= 0 ? cval[q] : 0.0;
  val[e] = v;
  if (valf) valf[e] = (float)v;
}

}  // namespace

size_t pcg2_tail_bytes(const Pcg2Plan &P) {
  auto al = [](size_t b) { return (b + 15) & ~(size_t)15; };
  auto sell = [&](const SellMat &M) -> size_t {
    if (M.nslices == 0) return 0;
    return al(sizeof(int) * (M.nslices + 1)) + al(sizeof(int) * (size_t)M.entries) + al(sizeof(float) * (size_t)M.entries);
  };
  size_t tot = 0;
  for (int k = P.nbig; k < P.nlev; ++k) {
    const Pcg2Level &L = P.lev[k];
    const bool dense_bottom = (k == P.nlev - 1) && P.bottom_dense;
    tot += (dense_bottom ? 0 : sell(L.A)) + sell(L.T) + sell(L.Tt) + 6 * al(sizeof(double) * (size_t)L.m);
  }
  return tot;
}

static int g_pcg2_grid[64] = {0};

int pcg2_grid(int device) {
  if (device < 0 || device >= 64) return 0;
  if (g_pcg2_grid[device]) return g_pcg2_grid[device];
  int nsm = 0, coop = 0, per_sm = 0, optin = 0;
  if (cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return 0;
  cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
  cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  if (!coop) return 0;
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, k_pcg2<true>) != cudaSuccess) return 0;   // the larger of the two instantiations
  const int dyn = optin - (int)fa.sharedSizeBytes - 1024;
  if (dyn > 0) {
    cudaFuncSetAttribute(k_pcg2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn);
    cudaFuncSetAttribute(k_pcg2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn);
  }
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pcg2<true>, kPcg2Threads, dyn > 0 ? dyn : 0) != cudaSuccess || per_sm < 1) return 0;
  g_pcg2_grid[device] = nsm < kPcg2MaxGrid ? nsm : kPcg2MaxGrid;
  return g_pcg2_grid[device];
}

size_t pcg2_max_tail_bytes(int device);
size_t pcg2_max_tail_bytes(int device) {
  int optin = 0;
  cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, k_pcg2<true>) != cudaSuccess) return 0;
  const int dyn = optin - (int)fa.sharedSizeBytes - 1024;
  return dyn > 0 ? (size_t)dyn : 0;
}

cudaError_t pcg2_launch(const Pcg2Plan *dev_plan, int grid, size_t smem_bytes, double rtol2, int maxit, int stall_window, bool dist, cudaStream_t s) {
  void *args[] = {(void *)&dev_plan, (void *)&rtol2, (void *)&maxit, (void *)&stall_window};
  const void *fn = dist ? (const void *)k_pcg2<true> : (const void *)k_pcg2<false>;
  return cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kPcg2Threads), args, smem_bytes, s);
}

cudaError_t pcg2_lambda_power(const Pcg2Plan *dev_plan, int grid, int iters, double safety, cudaStream_t s) {
  void *args[] = {(void *)&dev_plan, (void *)&iters, (void *)&safety};
  return cudaLaunchCooperativeKernel((const void *)k_lambda_power, dim3(grid), dim3(kPcg2Threads), args, 0, s);
}

cudaError_t sell_slice_widths(int64_t rows, int lpr, const int64_t *ptr, int *width, cudaStream_t s) {
  const int rps = 32 / lpr;
  const int64_t nsl = (rows + rps - 1) / rps;
  if (nsl == 0) return cudaSuccess;
  k_sell_widths<<<(unsigned int)((nsl * 32 + 255) / 256), 256, 0, s>>>(rows, lpr, ptr, width);
  return cudaGetLastError();
}
cudaError_t sell_fill_pattern(int64_t rows, int lpr, const int64_t *ptr, const int32_t *csr_idx, const int *soff, int *idx, int *src, cudaStream_t s) {
  const int rps = 32 / lpr;
  const int64_t nsl = (rows + rps - 1) / rps;
  if (nsl == 0) return cudaSuccess;
  k_sell_pattern<<<(unsigned int)((nsl * 32 + 255) / 256), 256, 0, s>>>(rows, lpr, ptr, csr_idx, soff, idx, src);
  return cudaGetLastError();
}
cudaError_t sell_fill_values(int entries, const int *src, const double *csr_val, double *val, float *valf, cudaStream_t s) {
  if (entries == 0) return cudaSuccess;
  k_sell_values<<<(entries + 255) / 256, 256, 0, s>>>(entries, src, csr_val, val, valf);
  return cudaGetLastError();
}

}  // namespace mgbx
