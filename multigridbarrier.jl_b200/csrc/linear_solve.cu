// linear_solve.cu -- dir = H^{-1} g for one Newton system: preconditioner setup after each assembly, the dense direct
// solves, and the V-cycle-preconditioned CG, which runs as one cooperative launch of k_pcg2 (pcg2.hpp / pcg2.cu).
//   utils.jl:142-145           solve           -> Engine::solve (dense Cholesky or V-cycle PCG)
#include "engine.hpp"
#include "solver_kernels.cuh"

namespace mgbx {

void solve_kernels_init() {
  CK(cudaFuncSetAttribute(k_coarse_inverse, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)coarse_inverse_smem(kCoarseMaxDense)));
  CK(cudaFuncSetAttribute(k_dense_solve_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dense_solve_small_smem(kCoarseMaxDense)));
  CK(cudaFuncSetAttribute(k_chol_diag_inv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCholDiagSmem));
  CK(cudaFuncSetAttribute(k_chol_solve_blocked, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(double) * kDenseMaxUnknowns)));
}

// FP32 copies of the level matrices for the preconditioner passes: on, off, or (2) automatic -- only when the top matrix
// is far larger than the L2 cache, i.e. when the V-cycle is HBM-bound (measured -12% per PCG iteration at 26 M non-zeros,
// neutral at 2 M)
bool Engine::precond_fp32(const System &S) const {
  if (h->cfg.precond_fp32 != 2) return h->cfg.precond_fp32 == 1;
  int64_t tot = 0;                       // automatic: the level matrices together (12 B per entry) no longer fit the 126 MB L2
  for (const SysLevel &Lv : S.lev) tot += Lv.A.nnz;
  return tot >= 10000000;
}
// power iterations per level and assembly for lambda_max(D^-1 A): cfg.lambda_power, or automatic (-1): 6 when the top
// matrix has long rows (3-D stencils: the Gershgorin bound overestimates 1.3-2.5x there and misplaces the Chebyshev
// interval -- measured on fem3d 32^3: 14 194 -> 8 294 PCG iterations per solve), none on 2-D meshes (bound within 4 %)
int Engine::lambda_power_its(const System &S) const {
  if (h->cfg.lambda_power >= 0) return h->cfg.lambda_power;
  if (S.lev.empty() || S.lev[0].A.rows == 0) return 0;
  return ((double)S.lev[0].A.nnz / (double)S.lev[0].A.rows > 16.0) ? 6 : 0;
}
// Systems with at most dense_direct_max unknowns are solved directly (shared-memory solve with pivoted fallback up to
// 128, blocked DMMA Cholesky above): faster than PCG at these sizes and robust for the systems that could not be
// condensed (e.g. a :broken_P1 slack), whose 1/slack^2 entries make them too ill-conditioned for an iterative solve.
bool Engine::use_direct(const System &S, const SysLevel &Lv) const {
  return S.dense || Lv.m <= h->cfg.dense_direct_max;   // dense (spectral) systems have no hierarchy: always direct
}
std::vector<int> Engine::active_levels(const System &S, int ktop) const {
  const int nlev = (int)S.lev.size();
  const int kend = (S.cut >= 0) ? std::max(S.cut, ktop) : nlev - 1;
  std::vector<int> act;
  for (int k = ktop; k <= kend; ++k) {
    if (k < kend && S.lev[k].T_identity) continue;   // same matrix as the next level
    act.push_back(k);
  }
  return act;
}

void Engine::setup_hierarchy(Amg &A, System &S, int ktop) {
  const int nlev = (int)S.lev.size();
  SysLevel &Ltop = S.lev[ktop];
  const bool direct = use_direct(S, Ltop);
  int kend = ktop;
  if (!direct) kend = (S.cut >= 0) ? std::max(S.cut, ktop) : nlev - 1;
  galerkin(S, kend);
  if (direct) {
    if (Ltop.m > kCoarseMaxDense) dense_factor(Ltop);   // tiny systems are factorised inside k_dense_solve_small
    return;
  }
  for (int k = ktop; k <= kend; ++k) {
    SysLevel &Lv = S.lev[k];
    CK(cudaMemsetAsync(Lv.lam, 0, sizeof(double), s));
    LAUNCH(KC_VEC, k_l1diag<<<nblk(Lv.m), 256, 0, s>>>(Lv.A, Lv.dinv, Lv.diag, (unsigned long long *)Lv.lam));
    if (precond_fp32(S)) {
      if (!Lv.val32) Lv.val32 = h->pool.alloc<float>(Lv.A.nnz);
      LAUNCH(KC_VEC, k_f64_to_f32<<<nblk(Lv.A.nnz), 256, 0, s>>>(Lv.A.nnz, Lv.A.val, Lv.val32));
    }
  }
  if (S.cut >= 0 && S.cut >= ktop) {
    SysLevel &Lc = S.lev[S.cut];
    const int m = (int)Lc.m;
    if (!Lc.dense_inv) Lc.dense_inv = h->pool.alloc<double>((size_t)m * m);
    LAUNCH(KC_DENSE, k_coarse_inverse<<<1, 1024, coarse_inverse_smem(m), s>>>(Lc.A, Lc.dense_inv));
  }
  sell_prepare(S, ktop);
  if (lambda_power_its(S) > 0) {   // all levels' power iterations in one cooperative launch
    System::Pcg2Dev &D = pcg2_plan(S, ktop);
    if ((int64_t)D.host.nlev * h->pcg2_grid > 3 * (int64_t)kPcg2MaxGrid) throw std::runtime_error("internal: too many levels for the power-iteration kernel");
    LAUNCH(KC_VEC, CK(pcg2_lambda_power(D.dev, h->pcg2_grid, lambda_power_its(S), 1.2, s)));
  }
}

void Engine::dense_factor(SysLevel &Lv) {
  const int m = (int)Lv.m;
  if (m == 0) return;
  const int npan = (m + kCholNB - 1) / kCholNB;
  if (!Lv.dense) {
    Lv.dense = h->pool.alloc<double>((size_t)m * m);
    Lv.dscale = h->pool.alloc<double>(m);
    Lv.dense_inv = h->pool.alloc<double>((size_t)npan * kCholNB * kCholNB);   // inverses of the diagonal blocks
  }
  zero(Lv.dense, (int64_t)m * m);
  LAUNCH(KC_DENSE, k_dense_scale_diag<<<nblk(m), 256, 0, s>>>(Lv.A, Lv.dscale));
  LAUNCH(KC_DENSE, k_csr_to_dense<<<nblk(m), 256, 0, s>>>(Lv.A, Lv.dscale, Lv.dense));
  // blocked right-looking Cholesky, panel width 64: diagonal block in shared memory, panel and trailing update as DMMA GEMMs
  for (int p = 0; p < npan; ++p) {
    const int k0 = p * kCholNB, nb = std::min(kCholNB, m - k0), rem = m - k0 - nb;
    double *Li = Lv.dense_inv + (size_t)p * kCholNB * kCholNB;
    LAUNCH(KC_DENSE, k_chol_diag_inv<<<1, 1024, kCholDiagSmem, s>>>(Lv.dense, m, k0, Li));
    if (rem > 0) {
      double *A21 = Lv.dense + (size_t)(k0 + nb) * m + k0;
      dgemm_nt(rem, nb, nb, A21, m, Li, kCholNB, nullptr, A21, m, false);                                   // L21 = A21 inv(L11)' (in place: one tile column)
      dgemm_nt(rem, rem, nb, A21, m, A21, m, nullptr, Lv.dense + (size_t)(k0 + nb) * m + k0 + nb, m, true, -1.0);   // A22 -= L21 L21'
    }
  }
}

// x = A^{-1} b through the scaled Cholesky factor (one right-hand side), uses Lv.r as scratch
void Engine::dense_apply(SysLevel &Lv, const double *b, double *x) {
  const int m = (int)Lv.m;
  LAUNCH(KC_DENSE, k_chol_solve_blocked<<<1, 1024, sizeof(double) * m, s>>>(Lv.dense, m, Lv.dense_inv, Lv.dscale, b, x));
}

// x = A^{-1} b by the dense direct solve (factorised by dense_factor above kCoarseMaxDense unknowns) and one step of
// iterative refinement against the CSR operator; uses Lv.r and Lv.x2 as scratch
void Engine::direct_solve(SysLevel &Lv, const double *b, double *x) {
  const bool small = Lv.m <= kCoarseMaxDense;
  auto apply = [&](const double *rhs, double *out) {
    if (small) LAUNCH(KC_DENSE, k_dense_solve_small<<<1, 1024, dense_solve_small_smem((int)Lv.m), s>>>(Lv.A, rhs, out, nullptr));
    else dense_apply(Lv, rhs, out);
  };
  apply(b, x);
  spmv(Lv.A, x, b, -1.0, Lv.r, Lv.spmv_group);
  apply(Lv.r, Lv.x2);
  axpby(Lv.m, 1.0, x, 1.0, Lv.x2, x);
}

// sliced-ELL copy of a device CSR pattern (32 rows per slice, slices-per-CTA for the grid the kernel is launched with)
SellBuild Engine::make_sell(const DevCsr &A, int64_t nthreads) {
  SellBuild B;
  h->pool.cat = "solve kernel: sliced-ELL level matrices";
  if (A.rows >= INT32_MAX / 2) throw std::runtime_error("persistent solve kernel: a level matrix exceeds 32-bit indexing");
  // lanes per row: widen while the level leaves at least half of the threads that share its phases idle and the rows
  // still give every lane two entries (measured, tools/micro/bench_spmv_phase: one lane per row wins on the two finest
  // levels of C2, four lanes on the 32 k-row level)
  int lpr = 1;
  const double avg = A.rows ? (double)A.nnz / (double)A.rows : 0.0;
  // up to a whole warp per row: the near-dense coarse Galerkin levels of 3-D hierarchies (fem3d 64^3: 544 rows of ~500 entries)
  // otherwise leave 8 lanes walking 60+ dependent rounds each -- 141 us per PCG iteration on a 544-row level
  // (profiles/r02h_pcg2_phase_profile_fem3d_64cubed.txt)
  while (lpr < 32 && A.rows * (int64_t)lpr * 2 <= nthreads && avg / lpr >= 2.0) lpr *= 2;
  const int rps = 32 / lpr;
  const int nsl = (int)((A.rows + rps - 1) / rps);
  B.M.rows = (int)A.rows;
  B.M.lpr = lpr;
  B.M.nslices = nsl;
  B.M.spc = pcg2_slices_per_cta(nsl, std::max(1, h->pcg2_grid));
  if (nsl == 0) return B;
  int *width = tmp_alloc<int>(nsl, s);
  CK(sell_slice_widths(A.rows, lpr, A.ptr, width, s));
  std::vector<int> hw(nsl);
  CK(cudaMemcpyAsync(hw.data(), width, sizeof(int) * nsl, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  tmp_free(width, s);
  std::vector<int> soff(nsl + 1, 0);
  int64_t tot = 0;
  for (int q = 0; q < nsl; ++q) {
    tot += 32 * (int64_t)hw[q];
    if (tot > INT32_MAX) throw std::runtime_error("persistent solve kernel: sliced-ELL level matrix exceeds 32-bit indexing");
    soff[q + 1] = (int)tot;
  }
  B.M.entries = (int)tot;
  B.soff = h->pool.upload<int>(soff.data(), soff.size(), s);
  B.idx = h->pool.alloc<int>((size_t)tot);
  B.src = h->pool.alloc<int>((size_t)tot);
  B.val = h->pool.alloc<double>((size_t)tot);
  B.valf = h->pool.alloc<float>((size_t)tot);
  CK(sell_fill_pattern(A.rows, lpr, A.ptr, A.idx, B.soff, B.idx, B.src, s));
  h->launches += 2;
  B.M.soff = B.soff;
  B.M.idx = B.idx;
  B.M.val = B.val;
  B.M.valf = nullptr;
  CK(cudaStreamSynchronize(s));   // soff (host vector) has been consumed
  return B;
}

// Build (once) the sliced-ELL structures of the active levels below lev[ktop] and refresh the values of the level matrices.
// Called from setup_hierarchy after every assembly, i.e. before every solve.
void Engine::sell_prepare(System &S, int ktop) {
  const std::vector<int> act = active_levels(S, ktop);
  const int64_t grid_threads = (int64_t)h->pcg2_grid * kPcg2Threads;
  for (size_t q = 0; q < act.size(); ++q) {
    SysLevel &Lv = S.lev[act[q]];
    // threads that share this level's phases: the whole grid, or CTA 0 alone for the tail (q > 0 and small)
    const int64_t nthr = (q > 0 && Lv.m <= h->cfg.tail_max) ? kPcg2Threads : grid_threads;
    if (!Lv.sell_A) {
      Lv.sA = make_sell(Lv.A, nthr);
      Lv.sell_A = true;
    }
    if (Lv.sA.M.entries) LAUNCH(KC_VEC, CK(sell_fill_values(Lv.sA.M.entries, Lv.sA.src, Lv.A.val, Lv.sA.val, Lv.sA.valf, s)));
    if (q + 1 < act.size() && !Lv.sell_T) {
      const int64_t nthr_c = (S.lev[act[q + 1]].m <= h->cfg.tail_max) ? kPcg2Threads : grid_threads;
      Lv.sT = make_sell(Lv.T, nthr);
      Lv.sTt = make_sell(Lv.Tt, nthr_c);
      if (Lv.sT.M.entries) LAUNCH(KC_VEC, CK(sell_fill_values(Lv.sT.M.entries, Lv.sT.src, Lv.T.val, Lv.sT.val, Lv.sT.valf, s)));
      if (Lv.sTt.M.entries) LAUNCH(KC_VEC, CK(sell_fill_values(Lv.sTt.M.entries, Lv.sTt.src, Lv.Tt.val, Lv.sTt.val, Lv.sTt.valf, s)));
      Lv.sell_T = true;
    }
  }
}

System::Pcg2Dev &Engine::pcg2_plan(System &S, int ktop) {
  auto it = S.pplans2.find(ktop);
  if (it != S.pplans2.end()) return it->second;
  System::Pcg2Dev &D = S.pplans2[ktop];
  Pcg2Plan &P = D.host;
  P = Pcg2Plan();
  const std::vector<int> act = active_levels(S, ktop);
  if ((int)act.size() > kPcg2MaxLevels) throw std::runtime_error("persistent solve kernel: too many levels");
  P.nlev = (int)act.size();
  P.bottom_dense = (S.cut >= 0 && act.back() == S.cut) ? 1 : 0;
  P.nu = std::max(1, h->cfg.smoother_sweeps);
  P.nu_bottom = 30;
  P.smoother = h->cfg.smoother;
  P.cheb_ratio = h->cfg.cheb_ratio > 1.0 ? h->cfg.cheb_ratio : 8.0;
  const bool f32 = precond_fp32(S);
  for (int q = 0; q < P.nlev; ++q) {
    SysLevel &Lv = S.lev[act[q]];
    Pcg2Level &pl = P.lev[q];
    if (Lv.m > INT32_MAX / 2) throw std::runtime_error("persistent solve kernel: level exceeds 32-bit indexing");
    pl.m = (int)Lv.m;
    pl.A = Lv.sA.M;
    pl.A.valf = Lv.sA.valf;       // narrowed below for the grid-wide levels
    if (q + 1 < P.nlev) {
      pl.T = Lv.sT.M;
      pl.T.valf = Lv.sT.valf;
      pl.Tt = Lv.sTt.M;
      pl.Tt.valf = Lv.sTt.valf;
    }
    pl.idiag = Lv.diag;
    pl.dinv = Lv.dinv;
    pl.lam = Lv.lam;
    pl.b = Lv.b;
    pl.x = Lv.x;
    pl.x2 = Lv.x2;
    pl.r = Lv.r;
    if (!Lv.pw) {   // power-iteration vector (warm-started across Newton iterations)
      Lv.pw = h->pool.alloc<double>(Lv.m);
      LAUNCH(KC_VEC, k_pw_init<<<nblk(Lv.m), 256, 0, s>>>(Lv.m, Lv.pw));
    }
    pl.pw = Lv.pw;
  }
  // the tail [nbig, nlev): levels with <= tail_max unknowns, as many as fit into CTA 0's shared memory
  int dev = 0;
  CK(cudaGetDevice(&dev));
  const size_t cap = pcg2_max_tail_bytes(dev);
  P.nbig = 0;
  for (int q = 0; q < P.nlev; ++q)
    if (S.lev[act[q]].m > h->cfg.tail_max) P.nbig = q + 1;
  P.nbig = std::max(P.nbig, 1);
  while (P.nbig < P.nlev && (pcg2_tail_bytes(P) > cap || P.nlev - P.nbig > 12)) P.nbig++;
  D.smem = (P.nbig < P.nlev) ? pcg2_tail_bytes(P) : 0;
  P.tail_smem_bytes = (int)D.smem;
  for (int q = 0; q < P.nbig; ++q) {   // grid-wide levels read FP32 values only when the FP32 preconditioner is on
    if (!f32) P.lev[q].A.valf = P.lev[q].T.valf = P.lev[q].Tt.valf = nullptr;
  }
  P.dense_inv = P.bottom_dense ? S.lev[S.cut].dense_inv : nullptr;
  P.r = S.pc_r;
  P.p = S.pc_p;
  P.p2 = S.pc_p2;
  P.Ap = S.pc_Ap;
  P.x = S.pc_x;
  P.b = S.pc_b;
  P.partials = S.pcg_partials;
  P.bar = S.pcg_bar;
  P.out = S.pcg_out;
  if (getenv("MGBX_PCG_PROF")) P.prof = h->pool.zeros<unsigned long long>(1 + 2 * (size_t)kPcg2ProfCap, s);
  if (dist() && h->cfg.shard_solve && P.nlev >= 2) {
    // multi-GPU: the leading levels with at least shard_min_rows unknowns are row-sharded over the ranks (pcg2.hpp)
    // A cross-GPU barrier costs several microseconds more than the local grid barrier, so a level is sharded only when a phase
    // over it is long enough to pay for that: T (1 - 1/N) > B with T ~ 12 B nnz / 3 TB/s and B ~ 10 us (measured on 2 GPUs:
    // profiles/r02f_*), i.e. nnz (1 - 1/N) >= shard_min_nnz (default 4 M).  C2's 2-D levels (1.8 M non-zeros) stay replicated.
    int nshard = 0;
    const std::vector<int> act = active_levels(S, ktop);
    for (int q = 0; q < P.nbig && q < P.nlev - 1; ++q) {
      const double nnzq = (double)S.lev[act[q]].A.nnz * (1.0 - 1.0 / (double)h->nranks);
      if (P.lev[q].m < h->cfg.shard_min_rows || nnzq < (double)h->cfg.shard_min_nnz) break;
      nshard = q + 1;
    }
    if (nshard > 0) pcg2_setup_dist(D, nshard);
  }
  D.dev = h->pool.upload<Pcg2Plan>(&P, 1, s);
  CK(cudaStreamSynchronize(s));
  if (h->cfg.verbose > 0)
    fprintf(stderr, "[mgbx] persistent PCG plan: %d levels (%d grid-wide, %d in CTA 0 from %zu bytes of shared memory), dense bottom %d, grid %d x %d\n",
            P.nlev, P.nbig, P.nlev - P.nbig, D.smem, P.bottom_dense, h->pcg2_grid, kPcg2Threads);
  return D;
}

// Exchange arena of one sharded solve plan: every vector a peer writes into (the work vectors of the sharded levels, p, x, the
// partial-sum slots, the barrier flags) is carved out of ONE cudaMalloc block with the same layout on every rank; the blocks
// are exported with CUDA IPC, the handles all-gathered with NCCL, and each rank maps its peers' blocks.
void Engine::pcg2_setup_dist(System::Pcg2Dev &D, int nshard) {
  Pcg2Plan &P = D.host;
  const int nr = h->nranks;
  if (nr > kPcg2MaxRanks) throw std::runtime_error("row-sharded solve: more than 8 ranks");
  if ((int64_t)nr * h->pcg2_grid > kPcg2MaxGrid) throw std::runtime_error("row-sharded solve: too many CTAs for the partial-sum slots");
  size_t bytes = 0;
  auto take = [&](size_t n) {
    const size_t off = bytes;
    bytes += (n + 255) & ~(size_t)255;
    return off;
  };
  const size_t o_flags = take(sizeof(unsigned long long) * kPcg2MaxRanks), o_arr = take(sizeof(unsigned int)), o_rel = take(sizeof(unsigned long long));
  const size_t o_part = take(sizeof(double) * 3 * (size_t)kPcg2MaxGrid);
  const size_t m0 = (size_t)P.lev[0].m;
  const size_t o_p = take(8 * m0), o_p2 = take(8 * m0), o_x = take(8 * m0);
  std::vector<size_t> o_lev(4 * (size_t)nshard);
  for (int q = 0; q < nshard; ++q)
    for (int v = 0; v < 4; ++v) o_lev[4 * q + v] = take(8 * (size_t)P.lev[q].m);
  CK(cudaMalloc((void **)&D.arena, bytes));
  CK(cudaMemsetAsync(D.arena, 0, bytes, s));
  // export / all-gather / import
  cudaIpcMemHandle_t mine;
  CK(cudaIpcGetMemHandle(&mine, D.arena));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  char *dsend = tmp_alloc<char>(64, s), *dall = tmp_alloc<char>(64 * (size_t)nr, s);
  CK(cudaMemcpyAsync(dsend, &mine, 64, cudaMemcpyHostToDevice, s));
  NCK(nccl_api().AllGather(dsend, dall, 8, kNcclInt64, h->comm, s));
  std::vector<cudaIpcMemHandle_t> all(nr);
  CK(cudaMemcpyAsync(all.data(), dall, 64 * (size_t)nr, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  tmp_free(dsend, s);
  tmp_free(dall, s);
  P.dist = Pcg2Dist();
  P.dist.nranks = nr;
  P.dist.rank = h->rank;
  P.dist.nshard = nshard;
  for (int q = 0; q < nr; ++q) {
    if (q == h->rank) {
      P.dist.peer_off[q] = 0;
      continue;
    }
    CK(cudaIpcOpenMemHandle(&D.peer[q], all[q], cudaIpcMemLazyEnablePeerAccess));
    P.dist.peer_off[q] = (long long)((char *)D.peer[q] - D.arena);
  }
  P.dist.flags = (unsigned long long *)(D.arena + o_flags);
  P.dist.xarrive = (unsigned int *)(D.arena + o_arr);
  P.dist.xrelease = (unsigned long long *)(D.arena + o_rel);
  P.partials = (double *)(D.arena + o_part);
  P.p = (double *)(D.arena + o_p);
  P.p2 = (double *)(D.arena + o_p2);
  P.x = (double *)(D.arena + o_x);
  const int64_t gcta = (int64_t)nr * h->pcg2_grid;
  auto respc = [&](SellMat &M) { M.spc = pcg2_slices_per_cta(M.nslices, gcta); };
  for (int q = 0; q < nshard; ++q) {
    Pcg2Level &pl = P.lev[q];
    pl.x = (double *)(D.arena + o_lev[4 * q + 0]);
    pl.x2 = (double *)(D.arena + o_lev[4 * q + 1]);
    pl.r = (double *)(D.arena + o_lev[4 * q + 2]);
    pl.b = (double *)(D.arena + o_lev[4 * q + 3]);
    respc(pl.A);              // rows of level q: owned by the CTAs of all ranks together
    respc(pl.T);
    if (q > 0) respc(P.lev[q - 1].Tt);
  }
  if (h->cfg.verbose > 0)
    fprintf(stderr, "[mgbx] rank %d: row-sharded solve over %d ranks, %d of %d levels sharded, exchange arena %.1f MB\n", h->rank, nr, nshard, P.nlev, bytes / 1e6);
}

// Preconditioned CG on lev[ktop], the whole solve in one cooperative launch of k_pcg2
SolveResult Engine::pcg(System &S, int ktop, const double *b, double *x, const SolveTol &tol) {
  SysLevel &Lv = S.lev[ktop];
  const int64_t m = Lv.m;
  System::Pcg2Dev &D = pcg2_plan(S, ktop);
  if (b != S.pc_b) copy(S.pc_b, b, m);
  pre_launch(KC_PCG);
  CK(pcg2_launch(D.dev, h->pcg2_grid, D.smem, tol.rtol2, h->cfg.pcg_maxit, tol.window, D.host.dist.nshard > 0, s));
  post_launch(KC_PCG);
  if (D.host.prof) {   // debugging aid: accumulate the per-phase durations of this launch
    h->prof_host.resize(1 + 2 * (size_t)kPcg2ProfCap);
    CK(cudaMemcpyAsync(h->prof_host.data(), D.host.prof, sizeof(unsigned long long) * h->prof_host.size(), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (h->prof_ns.empty()) {
      h->prof_ns.assign(kPcg2MaxLevels * 16, 0.0);
      h->prof_cnt.assign(kPcg2MaxLevels * 16, 0);
    }
    const size_t nrec = (size_t)h->prof_host[0];
    for (size_t q = 1; q < nrec; ++q) {
      const int tag = (int)h->prof_host[1 + 2 * q];
      if (tag < 0 || tag >= kPcg2MaxLevels * 16) continue;
      h->prof_ns[tag] += (double)(h->prof_host[2 + 2 * q] - h->prof_host[2 + 2 * (q - 1)]);
      h->prof_cnt[tag]++;
    }
  }
  CK(cudaMemcpyAsync(h->hscal + kScalPcgOut, S.pcg_out, sizeof(double) * kPcg2OutCount, cudaMemcpyDeviceToHost, s));
  sync();
  const double *o = h->hscal + kScalPcgOut;
  const int it = (int)o[kPcg2OutIters];
  const double status = o[kPcg2OutStatus];
  if (status == -3.0) throw std::runtime_error("row-sharded solve: a peer rank never arrived at a cross-GPU barrier (ranks out of step?)");
  if (x != D.host.x) copy(x, D.host.x, m);
  SolveResult r;
  r.iters = status < 0 ? -std::max(it, 1) : it;
  r.status = (int)status;
  r.rel = (o[kPcg2OutBB] > 0.0) ? std::sqrt(o[kPcg2OutRR] / o[kPcg2OutBB]) : 0.0;
  r.erel = (o[kPcg2OutEnergy] > 0.0) ? o[kPcg2OutEnergyLast4] / o[kPcg2OutEnergy] : 0.0;
  return r;
}

SolveResult Engine::solve_compact(System &S, int ktop, const double *b, double *x, const SolveTol &tol) {
  SysLevel &Lv = S.lev[ktop];
  if (use_direct(S, Lv)) {
    direct_solve(Lv, b, x);
    return SolveResult();
  }
  // Loud, not slow: an un-condensable slack above the dense fallback size would grind through thousands of failing PCG solves
  // (kappa -> sqrt(kappa) ~50 times per barrier step) before mgb_core gives up.  The reference's direct solve has no such
  // regime; refuse it up front unless the caller opts in (cfg.uncondensed_pcg).
  if (S.uncondensed_slack && !h->cfg.uncondensed_pcg && Lv.m > kDenseMaxUnknowns)
    throw UnsupportedError("Newton system with a slack variable that can be eliminated neither node-locally nor element-locally and " +
                           std::to_string((long long)Lv.m) + " unknowns: above the dense direct solver's size (8192) only the V-cycle PCG is available, "
                           "which is not reliable for these systems (set cfg.uncondensed_pcg = 1 to try anyway)");
  // The same rule after an element-local elimination (e.g. a slack in :broken_P1): the condensed systems keep the late-ramp
  // conditioning that stalls the V-cycle PCG (400 iterations without convergence from t max|f| ~ 3e5 on pure P2, CPU
  // experiment tools/pure_p2_lab.py), so above the dense solver's size they are refused as well.
  if (S.elem_local && !h->cfg.uncondensed_pcg && Lv.m > kDenseMaxUnknowns)
    throw UnsupportedError("Newton system with an element-local slack variable (e.g. a slack in :broken_P1), eliminated exactly: the condensed "
                           "system still has " + std::to_string((long long)Lv.m) + " unknowns, above the dense direct solver's size (8192); the V-cycle PCG "
                           "is not reliable for these systems late in the t-ramp (set cfg.uncondensed_pcg = 1 to try anyway)");
  SolveResult r = pcg(S, ktop, b, x, tol);
  // PCG first, direct second: a solve that broke down or stayed inexact is redone by the dense Cholesky when the system is
  // small enough to hold as a dense matrix (the un-condensable families, the last steps of a parabolic ramp)
  const bool bad = r.status < 0 || (r.rel > h->cfg.pcg_fail_rtol && r.erel > h->cfg.pcg_fail_etol);
  if (bad && h->cfg.direct_fallback && Lv.m <= kDenseMaxUnknowns) {
    if (h->cfg.verbose > 0)
      fprintf(stderr, "[mgbx] PCG on %lld unknowns ended with status %d, |r|/|b| = %.3g: falling back to the dense direct solve\n", (long long)Lv.m,
              r.status, r.rel);
    if (Lv.m > kCoarseMaxDense) dense_factor(Lv);
    direct_solve(Lv, b, x);
    r.status = 1;
    r.rel = r.erel = 0.0;
    if (h->res) h->res->direct_fallbacks++;
  }
  return r;
}

// dir = H_J^{-1} g  (full level-J vectors).  With a condensed system the node-local variables are
// eliminated exactly first and recovered by back-substitution.
SolveResult Engine::solve(Amg &A, System &S, int J, const double *g, double *dir, const SolveTol &tol) {
  cudaEvent_t st = stage_begin();
  const int ktop = S.ltop - J;
  SysLevel &Lv = S.lev[ktop];
  SolveResult r;
  if (S.nE == 0) {
    r = solve_compact(S, ktop, g, dir, tol);
  } else {
    // (only at the fine level)  rhs_K = g_K + R_K' sum_j D_j' gt_j
    CondParams C;
    memset(&C, 0, sizeof(C));
    C.n = A.n;
    C.nD = A.nD;
    C.nK = S.nK;
    C.nE = S.nE;
    for (int j = 0; j < S.nK; ++j) C.Krow[j] = S.Krow[j];
    for (int e = 0; e < S.nE; ++e) C.Eoff[e] = A.voff[A.L - 1][S.elim[e]];
    C.hEEinv = A.hEEinv;
    C.hKE = A.hKE;
    if (S.elem_local) LAUNCH(KC_COND, k_condense_rhs_elem<<<nblk(A.N), 256, 0, s>>>(C, S.el, A.N, A.p, g, A.G));
    else LAUNCH(KC_COND, k_condense_rhs<<<nblk(A.n), 256, 0, s>>>(C, g, A.G));
    ElemParams E = elem_params(A);
    E.nK = S.nK;
    for (int j = 0; j < S.nK; ++j) E.Krow[j] = S.Krow[j];
    blockgrad(A, E);
    if (!dist()) {
      spmv(A.RLt, A.gb, g, 1.0, A.tmp);               // tmp = g + R' gb   (entries of eliminated variables unused)
    } else {
      spmv(A.RLt, A.gb, nullptr, 1.0, A.tmp);         // this rank's part of R' gb, summed over the ranks, then + g
      allreduce_shared(A, J, A.tmp);
      axpby(A.m[J], 1.0, A.tmp, 1.0, g, A.tmp);
    }
    for (size_t q = 0; q < S.kept.size(); ++q)
      copy(S.pc_b + Lv.off[q], A.tmp + A.voff[A.L - 1][S.kept[q]], Lv.off[q + 1] - Lv.off[q]);
    r = solve_compact(S, ktop, S.pc_b, S.pc_x, tol);
    zero(dir, A.m[A.L - 1]);
    for (size_t q = 0; q < S.kept.size(); ++q)
      copy(dir + A.voff[A.L - 1][S.kept[q]], S.pc_x + Lv.off[q], Lv.off[q + 1] - Lv.off[q]);
    // broken image of the kept part, then back-substitution
    spmv(A.RL, dir, nullptr, 1.0, A.gb);
    NodeParams NP = node_params(A, 0.0);
    NP.zf = A.gb;
    if (S.elem_local) LAUNCH(KC_COND, k_backsubst_elem<<<nblk(A.N), 256, 0, s>>>(C, S.el, NP, A.N, g, dir));
    else LAUNCH(KC_COND, k_backsubst<<<nblk(A.n), 256, 0, s>>>(C, NP, g, dir));
  }
  stage_end(STAGE_SOLVE, st);
  r.dg = dot2(A, J, dir, g);
  if (h->res) {
    h->res->linear_solves++;
    h->res->pcg_iters += r.iters > 0 ? r.iters : -r.iters;
  }
  return r;
}

}  // namespace mgbx
