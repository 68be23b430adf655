// pcg2.hpp -- interface of the persistent solve kernel k_pcg2 (pcg2.cu, its own translation unit).
//
// Replaces the reference's `solve(Symmetric(H), g)` (src/utils.jl:142-145: CHOLMOD; cuDSS in
// ext/MultiGridBarrierCUDAExt/cudss_solver.jl:264-381) by ONE cooperative launch that runs the whole V-cycle-preconditioned CG:
// every smoother sweep, residual, grid transfer, dot product and the convergence test, phases separated by grid barriers.
// Design:
//   * every level matrix (A, T, T') is stored as sliced ELL, 32 rows per slice, column-major inside a slice: a warp owns a slice,
//     lane = row, so index / value loads are coalesced and a row's loads are independent of each other (no row-pointer ->
//     entry chain; the only dependent load left is the gather of the vector entry);
//   * rows are OWNED: CTA c works on the same contiguous block of slices of a level in every phase, warps take the block's
//     slices round-robin -- the mapping the multi-GPU row partition extends (a rank owns a block of CTAs' blocks);
//   * the single-CTA tail levels keep their matrices in CTA 0's shared memory (copied once per launch);
//   * distinct exit states (converged / stagnated / iteration limit / breakdown).
// Row sums run over a row's entries in column order: results are deterministic.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mgbx {

constexpr int kPcg2Threads = 1024;
constexpr int kPcg2MaxGrid = 2048;        // partial-sum slots per reduction (CTAs of all ranks of a multi-GPU solve)
constexpr int kPcg2MaxRanks = 8;
constexpr int kPcg2MaxLevels = 32;
constexpr int kPcg2ProfCap = 1 << 16;   // phase-profile records per launch (debugging aid)

// sliced-ELL matrix: slice s holds rows [rps s, rps s + rps), rps = 32 / lpr; lane l of the owning warp reads the entries
// idx/val[soff[s] + 32 j + l], j < width(s).
// Padding entries carry val = 0 and idx = the first column of their row (a valid gather for rectangular matrices too).
// lpr lanes share a row (1, 2, 4 or 8; a slice then holds 32 / lpr rows): entry k of a row sits with lane (k mod lpr) of the
// row's lane group, so that short levels still occupy the whole grid and a long row's dependent loads are split.
// slices of a level each CTA owns when `ncta` CTAs (of one GPU, or of all ranks of a row-sharded level) share it
inline int pcg2_slices_per_cta(int64_t nslices, int64_t ncta) { return (int)((nslices + ncta - 1) / (ncta > 0 ? ncta : 1)); }
// rows [r0, r1) of a level with `rows` rows and `lpr` lanes per row that rank `rank` of `nranks` owns in a row-sharded solve
// with `grid` CTAs per rank (CTA c of rank r is CTA r * grid + c of the joint grid)
inline void pcg2_rank_rows(int64_t rows, int lpr, int grid, int nranks, int rank, int64_t &r0, int64_t &r1) {
  const int64_t rps = 32 / lpr, nsl = (rows + rps - 1) / rps;
  const int64_t spc = pcg2_slices_per_cta(nsl, (int64_t)grid * nranks);
  const int64_t s0 = (int64_t)rank * grid * spc, s1 = (int64_t)(rank + 1) * grid * spc;
  r0 = s0 * rps < rows ? s0 * rps : rows;
  r1 = s1 * rps < rows ? s1 * rps : rows;
}

struct SellMat {
  int rows = 0, nslices = 0;
  int lpr = 1;                 // lanes per row
  int spc = 0;                 // slices per CTA (grid-wide levels): CTA c owns slices [c spc, (c+1) spc)
  int entries = 0;             // padded entries (soff[nslices])
  const int *soff = nullptr;   // nslices + 1
  const int *idx = nullptr;
  const double *val = nullptr;
  const float *valf = nullptr; // FP32 copy of the values: used instead of val when set (preconditioner passes; always by the tail)
};

struct Pcg2Level {
  int m = 0;
  SellMat A, T, Tt;            // T: rows of this level <- next coarser active level; Tt: rows of the coarser level <- this level
  const double *idiag = nullptr;   // 1 / a_ii (Chebyshev)
  const double *dinv = nullptr;    // l1-Jacobi 1 / sum_j |a_ij|
  const double *lam = nullptr;     // bound of lambda_max(D^-1 A) (device scalar, refreshed with the values)
  double *b = nullptr, *x = nullptr, *x2 = nullptr, *r = nullptr;
  double *pw = nullptr;            // power-iteration vector for lambda_max(D^-1 A) (pcg2_lambda_power), kept between launches
};

// Multi-GPU solve (one process per GPU): levels [0, nshard) are row-sharded over the ranks.  Everything a peer writes lives in
// this rank's exchange arena (one cudaMalloc block, identical layout on every rank, mapped into the peers by CUDA IPC):
// peer_off[q] = (rank q's arena base) - (this rank's arena base) in this process's address space.
struct Pcg2Dist {
  int nranks = 1, rank = 0, nshard = 0;
  long long peer_off[kPcg2MaxRanks] = {0};
  unsigned long long *flags = nullptr;     // [nranks] epochs published by the peers' CTA 0 (in the arena)
  unsigned int *xarrive = nullptr;         // local arrival counter of the cross barrier (monotonic)
  unsigned long long *xrelease = nullptr;  // local release epoch (~0: abort)
};

struct Pcg2Plan {
  int nlev = 0, nbig = 0;      // active levels: [0, nbig) by the whole grid, [nbig, nlev) by CTA 0 alone
  int bottom_dense = 0;        // the last level is applied through dense_inv (m x m, row-major)
  int nu = 2, nu_bottom = 30;
  int smoother = 1;            // 1 Chebyshev(nu) on [lam/ratio, lam], 0 l1-Jacobi
  double cheb_ratio = 8.0;
  int tail_smem_bytes = 0;     // shared-memory bytes holding the tail levels' matrices (0: tail reads global memory)
  Pcg2Level lev[kPcg2MaxLevels];
  const double *dense_inv = nullptr;
  double *r = nullptr, *p = nullptr, *p2 = nullptr, *Ap = nullptr, *x = nullptr;
  const double *b = nullptr;
  double *partials = nullptr;  // 3 x kPcg2MaxGrid
  unsigned int *bar = nullptr;
  Pcg2Dist dist;
  unsigned long long *prof = nullptr;   // optional phase profile: [0] count, then (tag, globaltimer ns) pairs; tag = level * 16 + kind
  double *out = nullptr;       // result record, kPcg2OutCount slots (below)
};

// slots of Pcg2Plan::out, written by k_pcg2 once per launch
enum {
  kPcg2OutIters = 0,   // iterations
  kPcg2OutRR,          // |r|^2
  kPcg2OutStatus,      // 1 converged, 2 stagnated above the tolerance, 3 iteration limit, -1 breakdown,
                       // -3 a peer never arrived at a cross-GPU barrier
  kPcg2OutBB,          // |b|^2
  kPcg2OutEnergy,      // b.x = |x|_A^2
  kPcg2OutEnergyLast4, // the part of kPcg2OutEnergy gained in the last four iterations
  kPcg2OutCount
};

// shared memory the tail needs: indices + FP32 values of A, T, Tt of the levels >= nbig, their diagonals and work vectors
size_t pcg2_tail_bytes(const Pcg2Plan &P);
// one-time attribute setup + occupancy check; returns the number of CTAs to launch (<= SM count), 0 if the device cannot run it
int pcg2_grid(int device);
size_t pcg2_max_tail_bytes(int device);   // dynamic shared memory available to the tail
// `iters` power iterations on D^-1 A for every level of the plan in one cooperative launch; lam <- min(lam, safety |D^-1 A v|)
// (needs nlev * grid <= 3 * kPcg2MaxGrid partial slots and Pcg2Level::pw initialised to a non-zero vector)
cudaError_t pcg2_lambda_power(const Pcg2Plan *dev_plan, int grid, int iters, double safety, cudaStream_t s);
cudaError_t pcg2_launch(const Pcg2Plan *dev_plan, int grid, size_t smem_bytes, double rtol2, int maxit, int stall_window, bool dist, cudaStream_t s);

// ---- sliced-ELL construction from a device CSR (int64 row pointers, int32 columns), once per pattern
struct SellBuild {
  SellMat M;
  int *soff = nullptr, *idx = nullptr, *src = nullptr;   // src: CSR position of every padded entry, -1 = padding
  double *val = nullptr;
  float *valf = nullptr;
};
// width[s] = longest row of slice s (device array of nslices ints)
cudaError_t sell_slice_widths(int64_t rows, int lpr, const int64_t *ptr, int *width, cudaStream_t s);
// fills idx / src from the CSR pattern (soff already on the device)
cudaError_t sell_fill_pattern(int64_t rows, int lpr, const int64_t *ptr, const int32_t *csr_idx, const int *soff, int *idx, int *src, cudaStream_t s);
// val[e] = src[e] >= 0 ? csr_val[src[e]] : 0  (and the FP32 copy if valf != nullptr); called whenever the matrix values change
cudaError_t sell_fill_values(int entries, const int *src, const double *csr_val, double *val, float *valf, cudaStream_t s);

}  // namespace mgbx
