// evaluate.cu -- barrier evaluation (f0, f1) and Hessian assembly at one level, the level chain between a level and the
// fine broken space, and the vector helpers the other units launch through Engine.
//   convex.jl:155-202          f0 / f1 / f2    -> Engine::eval_f01 / assemble
//   BlockMatrices.jl:322-555   assembly plan   -> k_elem* / k_sell_gather over the plans of setup.cu
#include "engine.hpp"
#include "kernels.cuh"
#include "dense_kernels.cuh"

namespace mgbx {
namespace {

// per-node kernel, instantiated for array bounds NDT in {4, 6, 8, 12}
template <int MODE>
void launch_node(const NodeParams &P, unsigned int grid, cudaStream_t s) {
  if (P.nD <= 4) k_node<MODE, 4><<<grid, kRedThreads, 0, s>>>(P);
  else if (P.nD <= 6) k_node<MODE, 6><<<grid, kRedThreads, 0, s>>>(P);
  else if (P.nD <= 8) k_node<MODE, 8><<<grid, kRedThreads, 0, s>>>(P);
  else k_node<MODE, MGBX_MAX_ND><<<grid, kRedThreads, 0, s>>>(P);
}

// Fused element kernels walk persistent tiles: exactly one wave of resident CTAs (grid = SMs x occupancy), never more than
// the reduction slots.  The dynamic shared-memory limit of each kernel is raised once per device.
template <auto K, class Params>
void launch_wave(const Params &Q, unsigned int grid, size_t smem, cudaStream_t s) {
  static int nsm[64] = {0};   // per device ordinal: SM count, 0 until K's limit has been raised there
  int dev = 0;
  CK(cudaGetDevice(&dev));
  if (!nsm[dev]) {
    CK(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    CK(cudaDeviceGetAttribute(&nsm[dev], cudaDevAttrMultiProcessorCount, dev));
  }
  int occ = 1;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, K, 256, smem));
  const unsigned int wave = (unsigned int)std::min(std::max(1, occ) * nsm[dev], kRedBlocks);
  K<<<std::min(grid, wave), 256, smem, s>>>(Q);
}

// generic fused element kernel (k_elem), same NDT dispatch as launch_node
template <int MODE>
void launch_elem(const ElemFused &Q, unsigned int grid, size_t smem, cudaStream_t s) {
  if (Q.np.nD <= 4) launch_wave<k_elem<MODE, 4>>(Q, grid, smem, s);
  else if (Q.np.nD <= 6) launch_wave<k_elem<MODE, 6>>(Q, grid, smem, s);
  else if (Q.np.nD <= 8) launch_wave<k_elem<MODE, 8>>(Q, grid, smem, s);
  else launch_wave<k_elem<MODE, MGBX_MAX_ND>>(Q, grid, smem, s);
}

// specialised fused kernel of the default problem family (k_elem_plap)
template <int MODE>
void launch_plap(int dim, bool cond, const PlapParams &Q, unsigned int grid, size_t smem, cudaStream_t s) {
  if (cond || MODE == NODE_F01) {
    if (dim == 1) launch_wave<k_elem_plap<MODE, 1, true>>(Q, grid, smem, s);
    else if (dim == 2) launch_wave<k_elem_plap<MODE, 2, true>>(Q, grid, smem, s);
    else launch_wave<k_elem_plap<MODE, 3, true>>(Q, grid, smem, s);
  } else {
    if (dim == 1) launch_wave<k_elem_plap<NODE_F2, 1, false>>(Q, grid, smem, s);
    else if (dim == 2) launch_wave<k_elem_plap<NODE_F2, 2, false>>(Q, grid, smem, s);
    else launch_wave<k_elem_plap<NODE_F2, 3, false>>(Q, grid, smem, s);
  }
}

// the result of k_dot2 from its slots, and of k_dot2_seg: the local part (summed over the ranks) plus the shared part
Dot2 dot2_slots(const double *d) { return {d[0], d[1], d[2]}; }
Dot2 dot2_seg_slots(const double *local, const double *shared) {
  return {local[0] + shared[0], local[1] + shared[1], local[2] + shared[2]};
}

}  // namespace

void kron_w_init(size_t smem) { CK(cudaFuncSetAttribute(k_kron_w, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); }

void Engine::spmv(const DevCsr &A, const double *x, const double *y0, double alpha, double *y, int G) {
  if (A.rows == 0) return;
  if (G == 0) G = group_for(A);
  pre_launch(KC_SPMV);
  if (G == 32) k_spmv<32><<<nblk(A.rows * 32), 256, 0, s>>>(A, x, y0, alpha, y);
  else if (G == 4) k_spmv<4><<<nblk(A.rows * 4), 256, 0, s>>>(A, x, y0, alpha, y);
  else k_spmv<1><<<nblk(A.rows), 256, 0, s>>>(A, x, y0, alpha, y);
  post_launch(KC_SPMV);
}

void Engine::axpby(int64_t m, double a, const double *x, double b, const double *y, double *out) {
  LAUNCH(KC_VEC, k_axpby<<<nblk(m), 256, 0, s>>>(m, a, x, b, y, out));
}

// ---------------------------------------------------------------- level chain
// zf = z + R_L * T_{L-2} ... T_J * x
void Engine::prolong_to_fine(Amg &A, int J, const double *x, const double *zbase, double *zf) {
  const double *v = x;
  for (int l = J; l < A.L - 1; ++l) {
    spmv(A.T[l], v, nullptr, 1.0, A.chain[l + 1]);
    v = A.chain[l + 1];
  }
  spmv(A.RL, v, zbase, 1.0, zf);
}
// g_J = T_J' ... T_{L-2}' R_L' gb
void Engine::restrict_from_fine(Amg &A, int J, const double *gb, double *gJ) {
  if (J == A.L - 1) {
    spmv(A.RLt, gb, nullptr, 1.0, gJ);
    return;
  }
  spmv(A.RLt, gb, nullptr, 1.0, A.chain2[A.L - 1]);
  const double *v = A.chain2[A.L - 1];
  for (int l = A.L - 2; l >= J; --l) {
    double *out = (l == J) ? gJ : A.chain2[l];
    spmv(A.Tt[l], v, nullptr, 1.0, out);
    v = out;
  }
}


SegList Engine::seglist(Amg &A, int J) {
  SegList S;
  memset(&S, 0, sizeof(S));
  if (J == A.L - 1) {
    S.n = A.nu;
    for (int v = 0; v < A.nu; ++v) {
      S.off[v] = A.voff[J][v];
      S.local[v] = A.var_local[v];
    }
    S.off[A.nu] = A.voff[J][A.nu];
  } else {
    S.n = 1;
    S.off[0] = 0;
    S.off[1] = A.m[J];
  }
  return S;
}
// sum the shared segments of a level-J vector over the ranks (the local segments are already complete)
void Engine::allreduce_shared(Amg &A, int J, double *v, double *extra, int64_t nextra) {
  const SegList S = seglist(A, J);
  NCK(nccl_api().GroupStart());
  for (int q = 0; q < S.n; ++q)
    if (!S.local[q]) allreduce(v + S.off[q], S.off[q + 1] - S.off[q]);
  if (extra) allreduce(extra, nextra);
  NCK(nccl_api().GroupEnd());
}
// {a.b, a.a, #non-finite(a)} over a level-J vector (all ranks obtain the same values)
Dot2 Engine::dot2(Amg &A, int J, const double *a, const double *b) {
  const int64_t m = A.m[J];
  if (!dist()) {
    LAUNCH(KC_VEC, k_dot2<<<red_grid(m), kRedThreads, 0, s>>>(m, a, b, h->partials, h->ticket, h->dscal + kScalDot));
    fetch(kScalSingle);
    return dot2_slots(h->hscal + kScalDot);
  }
  LAUNCH(KC_VEC, k_dot2_seg<<<red_grid(m), kRedThreads, 0, s>>>(seglist(A, J), m, a, b, h->partials, h->ticket, h->dscal + kScalDotSeg));
  allreduce(h->dscal + kScalDotSeg, 3);   // the local part; the shared part is already the same on every rank
  fetch(kScalSlots);
  return dot2_seg_slots(h->hscal + kScalDotSeg, h->hscal + kScalDotSeg + 3);
}

// {max, max|.|, #non-finite} of a node vector (over all ranks)
MaxAbs Engine::maxabs(int64_t n, const double *v) {
  LAUNCH(KC_VEC, k_maxabs<<<red_grid(n), kRedThreads, 0, s>>>(n, v, h->partials, h->ticket, h->dscal + kScalMaxAbs));
  if (dist()) allreduce(h->dscal + kScalMaxAbs, 3, kNcclMax);
  fetch(kScalMaxAbs + 3);
  const double *d = h->hscal + kScalMaxAbs;
  return {d[0], d[1], d[2]};
}

// f0 / f1 at the level-J trial point A.xn = A.x - sigma A.dir (gradient into A.gn)
TrialOut Engine::eval_trial(Amg &A, int J, double t, double sigma) {
  const int64_t m = A.m[J];
  if (!dist()) LAUNCH(KC_VEC, k_trial<<<red_grid(m), kRedThreads, 0, s>>>(m, A.x, A.dir, sigma, A.xn, h->partials, h->ticket, h->dscal + kScalTrial));
  else LAUNCH(KC_VEC, k_trial_seg<<<red_grid(m), kRedThreads, 0, s>>>(seglist(A, J), m, A.x, A.dir, sigma, A.xn, h->partials, h->ticket, h->dscal + kScalTrialSeg));
  double step2 = 0.0;
  const EvalOut e = eval_f01(A, J, t, A.z, A.xn, A.gn, true, &step2);
  return {e, step2};
}

// phase-I start of the feasibility AMG F: [z0, slack] with slack_i = 2*max(slack_fn(D z0), 1) (src/mgb.jl:437-445);
// A.zf holds z0 from the feasibility probe
void Engine::phase1_slack(Amg &A, Amg &F) {
  NodeParams P = node_params(A, 0.0);
  LAUNCH(KC_NODE_F01, launch_node<NODE_SLACK>(P, red_grid(A.n), s));
  LAUNCH(KC_VEC, k_phase1_slack<<<nblk(A.n), 256, 0, s>>>(A.n, A.slack, F.zinit + (int64_t)A.nu * A.n));
  copy(F.zinit, A.z, (int64_t)A.nu * A.n);
  copy(F.z, F.zinit, (int64_t)F.nu * F.n);
}

// A.gb = sum_k D_k' A.G_k over the rows E.Krow
void Engine::blockgrad(Amg &A, const ElemParams &E) {
  LAUNCH(KC_BLOCKGRAD, k_blockgrad<<<nblk((int64_t)A.nu * A.n), 256, 0, s>>>(E, A.G, A.gb, A.nu));
}

NodeParams Engine::node_params(Amg &A, double t) {
  NodeParams P;
  memset(&P, 0, sizeof(P));
  P.n = A.n;
  P.p = A.p;
  P.nu = A.nu;
  P.nD = A.nD;
  for (int j = 0; j < A.nD; ++j) {
    P.D_var[j] = A.D_var[j];
    P.D_op[j] = A.D_op[j];
  }
  for (int o = 0; o < A.nops; ++o) P.ops[o] = A.ops[o];
  P.zf = A.zf;
  P.w = A.w;
  P.f = A.f;
  P.bw = A.bw;
  P.t = t;
  P.inv_n = 1.0 / (double)A.n_global;
  P.cd = A.cd;
  P.G = A.G;
  P.partials = h->partials;
  P.ticket = h->ticket;
  P.red_out = h->dscal + kScalEval;
  P.slack = A.slack;
  return P;
}
ElemParams Engine::elem_params(Amg &A) {
  ElemParams P;
  memset(&P, 0, sizeof(P));
  P.n = A.n;
  P.N = A.N;
  P.p = A.p;
  P.nD = A.nD;
  for (int j = 0; j < A.nD; ++j) {
    P.D_var[j] = A.D_var[j];
    P.D_op[j] = A.D_op[j];
  }
  for (int o = 0; o < A.nops; ++o) P.ops[o] = A.ops[o];
  P.nK = A.nD;
  for (int j = 0; j < A.nD; ++j) P.Krow[j] = j;
  return P;
}

// tile geometry of the fused element kernel; false: fall back to the separate node / block kernels
// (operator blocks too large for shared memory, e.g. the dense spectral "element")
bool Engine::elem_fused_setup(Amg &A, const NodeParams &NP, int nex, ElemFused &Q, size_t &smem, unsigned int &grid) {
  if (!h->cfg.fused || A.p > 256) return false;
  memset(&Q, 0, sizeof(Q));
  Q.np = NP;
  Q.N = A.N;
  Q.nops = A.nops;
  Q.p1 = A.p | 1;
  Q.ES = (A.p * Q.p1) | 1;
  Q.nex = nex;
  int epb = std::max(1, 256 / A.p);
  const size_t cap = 216 * 1024;
  while (epb > 1 && elem_fused_smem(A.nops, epb, Q.ES, A.nu, nex, A.p) > cap) epb = (epb + 1) / 2;
  smem = elem_fused_smem(A.nops, epb, Q.ES, A.nu, nex, A.p);
  if (smem > cap) return false;
  Q.epb = epb;
  const int64_t ntiles = (A.N + epb - 1) / epb;
  grid = (unsigned int)std::max<int64_t>(1, std::min<int64_t>(ntiles, kRedBlocks));
  return true;
}

// The default problem family (state (u, s), D = [u:id; u:d_1..d_dim; s:id], one Euclidean-power cone on rows 1..dim+1
// with identity A, zero b, uniform p and mu): returns dim (1..3) if the specialised kernel applies, else 0.
int Engine::plap_dim(const Amg &A) const {
  if (h->cfg.fused != 1 || A.nu != 2 || A.p >= 256) return 0;
  const int dim = A.nD - 2;
  if (dim < 1 || dim > 3) return 0;
  const int vu = A.D_var[0], vs = A.D_var[dim + 1];
  if (vu == vs || A.D_op[0] >= 0 || A.D_op[dim + 1] >= 0) return 0;
  for (int a = 1; a <= dim; ++a)
    if (A.D_var[a] != vu || A.D_op[a] < 0) return 0;
  const ConvexDev &cd = A.cd;
  if (cd.feas || cd.npieces != 1 || cd.select) return 0;
  const PieceDev &pc = cd.pc[0];
  if (pc.kind != MGBX_PIECE_EP || pc.ni != dim + 1 || pc.nc != dim + 1 || pc.A || pc.b || pc.p || pc.mu) return 0;
  for (int c = 0; c <= dim; ++c)
    if (pc.idx[c] != c + 1) return 0;
  return dim;
}
bool Engine::plap_setup(Amg &A, int dim, double t, bool use_bw, PlapParams &Q, size_t &smem, unsigned int &grid, bool cond) {
  memset(&Q, 0, sizeof(Q));
  Q.n = A.n;
  Q.N = A.N;
  Q.p = A.p;
  Q.p1 = A.p | 1;
  Q.ES = (A.p * Q.p1) | 1;
  // bulk staging (cfg.elem_bulk): operator slabs and node columns arrive by cp.async.bulk instead of one 8-byte cp.async per
  // double.  Odd p: the padded layout already equals the contiguous one (p1 == p, ES == p*p) -> one copy per operator slab;
  // even p: columns are padded to p + 2 (16-byte aligned, conflict-free transposed reads) -> one copy per block column.
  Q.bulk = 0;
  if (h->cfg.elem_bulk) {
    if (A.p & 1) {
      if (Q.p1 == A.p && Q.ES == A.p * A.p) Q.bulk = 1;
    } else {
      Q.p1 = A.p + 2;
      Q.ES = A.p * Q.p1;
      if (Q.ES % 16 == 0) Q.ES += 8;
      Q.bulk = 2;
    }
  }
  int epb = std::max(1, 256 / A.p);
  const size_t cap = 216 * 1024, want = 72 * 1024;   // aim at 3 resident CTAs per SM (double-buffered tiles)
  while (epb > 1 && elem_plap_smem(dim, epb, Q.ES, A.p, cond) > want && epb * A.p > 128) epb = (epb + 1) / 2;
  while (epb > 1 && elem_plap_smem(dim, epb, Q.ES, A.p, cond) > cap) epb = (epb + 1) / 2;
  if (Q.bulk && (epb & 1) && epb > 1) --epb;         // even tiles keep every slab a multiple of 16 bytes and 16-byte aligned
  if (Q.bulk && (epb & 1) && (A.p & 1)) Q.bulk = 0;  // a one-element tile of an odd element cannot be bulk-copied
  smem = elem_plap_smem(dim, epb, Q.ES, A.p, cond);
  if (smem > cap) return false;
  Q.epb = epb;
  Q.dp = make_fastdiv((unsigned int)A.p);
  Q.dpp = make_fastdiv((unsigned int)(A.p * A.p));
  for (int a = 0; a < dim; ++a) Q.ops[a] = A.ops[A.D_op[a + 1]];
  Q.zu = A.zf + (int64_t)A.D_var[0] * A.n;
  Q.zs = A.zf + (int64_t)A.D_var[dim + 1] * A.n;
  Q.w = A.w;
  Q.f = A.f;
  Q.bw = use_bw ? A.bw : nullptr;
  Q.t = t;
  Q.inv_n = 1.0 / (double)A.n_global;
  Q.pexp = A.cd.pc[0].p_uniform;
  Q.mu = A.cd.pc[0].mu_uniform;
  Q.partials = h->partials;
  Q.ticket = h->ticket;
  Q.red_out = h->dscal + (dist() ? kScalEvalDist : kScalEval);
  if (Q.bulk) {   // bulk copies need 16-byte aligned sources: every base pointer, and the column stride n of f / the state blocks
    auto al16 = [](const void *q) { return q == nullptr || ((uintptr_t)q & 15) == 0; };
    bool ok = al16(Q.zu) && al16(Q.zs) && al16(Q.w) && al16(Q.bw) && al16(Q.f) && (A.n % 2 == 0);
    for (int a = 0; a < dim; ++a) ok = ok && al16(Q.ops[a]);
    if (!ok) {   // fall back to the per-double staging with its own padding
      Q.bulk = 0;
      Q.p1 = A.p | 1;
      Q.ES = (A.p * Q.p1) | 1;
      smem = elem_plap_smem(dim, epb, Q.ES, A.p, cond);
      if (smem > cap) return false;
    }
  }
  const int64_t ntiles = (A.N + epb - 1) / epb;
  grid = (unsigned int)std::max<int64_t>(1, std::min<int64_t>(ntiles, kRedBlocks));
  return true;
}
// ---------------------------------------------------------------- f0 + f1 at level J
// zbase: broken state the level correction is added to; x: level-J coefficients; gout: level-J gradient
// step2: |xn - x|^2 of the trial launch that produced x (eval_trial)
EvalOut Engine::eval_f01(Amg &A, int J, double t, const double *zbase, const double *x, double *gout, bool use_bw, double *step2) {
  cudaEvent_t st = stage_begin();
  prolong_to_fine(A, J, x, zbase, A.zf);
  NodeParams P = node_params(A, t);
  if (!use_bw) P.bw = nullptr;
  if (dist()) P.red_out = h->dscal + kScalEvalDist;
  ElemFused Q;
  PlapParams PQ;
  size_t smem = 0;
  unsigned int grid = 0;
  const int pdim = plap_dim(A);
  if (pdim && plap_setup(A, pdim, t, use_bw, PQ, smem, grid)) {
    PQ.gbu = A.gb + (int64_t)A.D_var[0] * A.n;
    PQ.gbs = A.gb + (int64_t)A.D_var[pdim + 1] * A.n;
    LAUNCH(KC_ELEM_F01, launch_plap<NODE_F01>(pdim, true, PQ, grid, smem, s));
  } else if (elem_fused_setup(A, P, A.nD, Q, smem, grid)) {
    Q.gb = A.gb;
    LAUNCH(KC_ELEMG_F01, launch_elem<NODE_F01>(Q, grid, smem, s));
  } else {
    LAUNCH(KC_NODE_F01, launch_node<NODE_F01>(P, red_grid(A.n), s));
    blockgrad(A, elem_params(A));
  }
  restrict_from_fine(A, J, A.gb, gout);
  const double *red;   // red_out: {sum bw F0 (or sum F0), sum w c.Dz, #non-finite F0, max slack}
  Dot2 gg;             // {0, |gout|^2, #non-finite(gout)}
  if (!dist()) {
    LAUNCH(KC_VEC, k_dot2<<<red_grid(A.m[J]), kRedThreads, 0, s>>>(A.m[J], gout, nullptr, h->partials, h->ticket, h->dscal + kScalDot));
    stage_end(STAGE_F01, st);
    fetch(kScalSingle);
    red = h->hscal + kScalEval;
    gg = dot2_slots(h->hscal + kScalDot);
    if (step2) *step2 = h->hscal[kScalTrial];
  } else {
    // partial sums over this rank's elements -> all ranks: the shared part of R'g, the objective scalars, and the
    // local-part norms (one grouped all-reduce); the shared-part norm is then formed identically on every rank
    const SegList SG = seglist(A, J);
    LAUNCH(KC_VEC, k_dot2_seg<<<red_grid(A.m[J]), kRedThreads, 0, s>>>(SG, A.m[J], gout, nullptr, h->partials, h->ticket, h->dscal + kScalDotSeg));
    // the local trial norm, the node sums and the local dot
    allreduce_shared(A, J, gout, h->dscal + kScalTrialSeg + 1, kScalDotSeg + 3 - (kScalTrialSeg + 1));
    LAUNCH(KC_VEC, k_dot2_seg<<<red_grid(A.m[J]), kRedThreads, 0, s>>>(SG, A.m[J], gout, nullptr, h->partials, h->ticket, h->dscal + kScalDotSeg2));
    stage_end(STAGE_F01, st);
    fetch(kScalSlots);
    red = h->hscal + kScalEvalDist;
    gg = dot2_seg_slots(h->hscal + kScalDotSeg, h->hscal + kScalDotSeg2 + 3);
    if (step2) *step2 = h->hscal[kScalTrialSeg] + h->hscal[kScalTrialSeg + 1];
    CK(cudaMemsetAsync(h->dscal + kScalTrialSeg, 0, 2 * sizeof(double), s));   // the trial norms are consumed
  }
  if (h->res) h->res->f01_evals++;
  EvalOut o;
  const double bar = (use_bw && A.bw) ? red[0] : red[0] * (1.0 / (double)A.n_global);
  o.lin = red[1];
  o.y = bar + red[1];
  o.nonfinite_nodes = red[2];
  o.gnorm = std::sqrt(gg.aa);
  o.finite = std::isfinite(o.y) && (gg.nonfinite == 0.0) && std::isfinite(gg.aa);
  return o;
}
// Which Euclidean-power pieces can be condensed analytically (node_barrier.cuh piece_eval): identity A, not under the phase-I
// wrapper, the piece's slack row belongs to a node-locally eliminated variable that has no other D row and that no other piece
// (nor another input of this piece) touches, and none of its q rows is eliminated.  Then H_EE is diagonal in that variable and its
// Schur complement is the piece's own.
void Engine::schur_masks(const Amg &A, const System &S, unsigned &pieces, unsigned &elim) const {
  pieces = elim = 0u;
  if (!h->cfg.analytic_schur || S.nE == 0 || A.cd.feas) return;
  const ConvexDev &cd = A.cd;
  for (int k = 0; k < cd.npieces && k < 32; ++k) {
    const PieceDev &pc = cd.pc[k];
    if (pc.kind != MGBX_PIECE_EP || pc.A != nullptr || pc.nc < 2 || pc.ni != pc.nc) continue;
    const int nq = pc.nc - 1, js = pc.idx[nq];
    if (js < 0 || js >= A.nD) continue;
    const int ev = S.Erow[js];
    if (ev < 0) continue;
    bool ok = true;
    for (int r = 0; r < nq; ++r) ok = ok && pc.idx[r] != js && S.Erow[pc.idx[r]] < 0;
    for (int j = 0; j < A.nD; ++j) ok = ok && (j == js || S.Erow[j] != ev);          // the variable's only row
    for (int k2 = 0; k2 < cd.npieces; ++k2)
      if (k2 != k)
        for (int c = 0; c < cd.pc[k2].ni; ++c) ok = ok && cd.pc[k2].idx[c] != js;     // no other piece reads it
    if (ok) {
      pieces |= 1u << k;
      elim |= 1u << ev;
    }
  }
}

// Evaluate the node Hessians at zbase + R_J x and fill the system matrices from the top level down to
// level index ktop (= L-1-J), then the preconditioner hierarchy below it.
void Engine::assemble(Amg &A, System &S, int J, double t, const double *zbase, const double *x) {
  cudaEvent_t st = stage_begin();
  prolong_to_fine(A, J, x, zbase, A.zf);
  NodeParams P = node_params(A, t);
  P.nK = S.nK;
  P.nE = S.nE;
  for (int j = 0; j < MGBX_MAX_ND; ++j) {
    P.Krow[j] = S.Krow[j];
    P.Erow[j] = S.Erow[j];
  }
  P.Hn = A.Hn;
  P.hEEinv = A.hEEinv;
  P.hKE = A.hKE;
  schur_masks(A, S, P.schur_pieces, P.schur_elim);
  if (S.dense) {
    assemble_dense(A, S, P);
    stage_end(STAGE_F2, st);
    if (h->res) h->res->f2_evals++;
    return;
  }
  ElemFused Q;
  PlapParams PQ;
  size_t smem = 0;
  unsigned int grid = 0;
  const int pdim = plap_dim(A);
  // the specialised kernel needs exactly: s eliminated node-locally, u kept with all of its rows
  const bool plap_ok = pdim && S.nE == 1 && S.kept.size() == 1 && S.kept[0] == A.D_var[0] && S.elim[0] == A.D_var[pdim + 1] &&
                       S.nK == pdim + 1 && S.pl.npairs == 1 && plap_setup(A, pdim, t, true, PQ, smem, grid);
  // ... or nothing eliminated and the four pairs (u,u), (u,s), (s,u), (s,s) in this order (coarse-level systems)
  const bool plap_unc = !plap_ok && pdim && S.nE == 0 && S.kept.size() == 2 && S.nK == pdim + 2 && S.pl.npairs == 4 &&
                        S.pl.va[0] == A.D_var[0] && S.pl.vb[0] == A.D_var[0] && S.pl.va[1] == A.D_var[0] && S.pl.vb[1] == A.D_var[pdim + 1] &&
                        S.pl.va[2] == A.D_var[pdim + 1] && S.pl.vb[2] == A.D_var[0] && S.pl.va[3] == A.D_var[pdim + 1] &&
                        S.pl.vb[3] == A.D_var[pdim + 1] && plap_setup(A, pdim, t, true, PQ, smem, grid, false);
  if (plap_ok || plap_unc) {
    PQ.hEEinv = A.hEEinv;
    PQ.hKE = A.hKE;
    PQ.Hblk = S.Hblk;
    LAUNCH(KC_ELEM_F2, launch_plap<NODE_F2>(pdim, plap_ok, PQ, grid, smem, s));
  } else if (elem_fused_setup(A, P, std::max(A.nD, S.nK * (S.nK + 1) / 2), Q, smem, grid)) {
    Q.pl = S.pl;
    Q.Hblk = S.Hblk;
    LAUNCH(KC_ELEMG_F2, launch_elem<NODE_F2>(Q, grid, smem, s));
  } else {
    LAUNCH(KC_NODE_F2, launch_node<NODE_F2>(P, red_grid(A.n), s));
    ElemParams E = elem_params(A);
    E.nK = S.nK;
    for (int j = 0; j < S.nK; ++j) E.Krow[j] = S.Krow[j];
    LAUNCH(KC_BLOCKHESS, k_blockhess<<<nblk(S.hblk_size), 256, 0, s>>>(E, S.pl, A.Hn, S.Hblk));
  }
  if (S.elem_local) {   // the element-local part of the slack's Schur complement, on top of the node-local one
    ElemParams E = elem_params(A);
    E.nK = S.nK;
    for (int j = 0; j < S.nK; ++j) E.Krow[j] = S.Krow[j];
    LAUNCH(KC_COND, k_elem_local_schur<<<nblk(A.N, 128), 128, 0, s>>>(E, S.pl, S.el, A.hEEinv, A.hKE, S.Hblk));
  }
  SysLevel &top = S.lev[0];
  LAUNCH(KC_GATHER, k_sell_gather<<<nblk(top.A.nnz), 256, 0, s>>>(S.top, S.Hblk, top.A.val));
  if (dist()) allreduce(top.A.val, top.A.nnz);   // sum of the ranks' element contributions (identical pattern on every rank)
  const int ktop = S.ltop - J;
  setup_hierarchy(A, S, ktop);
  stage_end(STAGE_F2, st);
  if (h->res) h->res->f2_evals++;
}

// Galerkin products A_{k+1} = T_k' (A_k T_k) for the levels k < kend, one fixed-order gather each
void Engine::galerkin(System &S, int kend) {
  for (int k = 0; k < kend; ++k) {
    SysLevel &Lv = S.lev[k];
    SysLevel &Lc = S.lev[k + 1];
    if (Lv.T_identity) continue;   // an identity transfer aliases the same matrix
    LAUNCH(KC_SPGEMM, k_sell_gather<<<nblk(Lv.AT.nnz), 256, 0, s>>>(Lv.s1, Lv.A.val, Lv.AT.val));
    LAUNCH(KC_SPGEMM, k_sell_gather<<<nblk(Lc.A.nnz), 256, 0, s>>>(Lv.s2, Lv.AT.val, Lc.A.val));
  }
}

// Uncondensed Hessian of the sparse system S at level J, by the separate node and block kernels: the parity reference
// the fused element kernels are checked against (mgbx_hessian_values).  Leaves it in S.lev[ltop - J].A.
void Engine::assemble_unfused(Amg &A, System &S, int J, double t, const double *x) {
  prolong_to_fine(A, J, x, A.z, A.zf);
  NodeParams P = node_params(A, t);
  P.nK = S.nK;
  P.nE = 0;
  for (int j = 0; j < MGBX_MAX_ND; ++j) {
    P.Krow[j] = S.Krow[j];
    P.Erow[j] = -1;
  }
  P.Hn = A.Hn;
  LAUNCH(KC_NODE_F2, launch_node<NODE_F2>(P, red_grid(A.n), s));
  LAUNCH(KC_BLOCKHESS, k_blockhess<<<nblk(S.hblk_size), 256, 0, s>>>(elem_params(A), S.pl, A.Hn, S.Hblk));
  LAUNCH(KC_GATHER, k_sell_gather<<<nblk(S.lev[0].A.nnz), 256, 0, s>>>(S.top, S.Hblk, S.lev[0].A.val));
  if (dist()) allreduce(S.lev[0].A.val, S.lev[0].A.nnz);
  galerkin(S, S.ltop - J);
}


void Engine::dgemm_nt(int M, int N, int K, const double *Am, int64_t lda, const double *Bm, int64_t ldb, const double *sc, double *C, int64_t ldc,
                      bool acc, double alpha) {
  if (M <= 0 || N <= 0) return;
  // in place (C = A, e.g. L21 = A21 inv(L11)' in dense_factor) is correct only while one CTA owns whole rows of C: it reads
  // all K columns of its rows of A before it writes any of them, and no other CTA reads those rows
  if (C == Am && (N > kGemmBN || ldc != lda)) throw std::runtime_error("internal: in-place dgemm_nt needs N <= 64 and ldc == lda");
  dim3 grid((N + kGemmBN - 1) / kGemmBN, (M + kGemmBM - 1) / kGemmBM);
  LAUNCH(KC_DGEMM, k_dgemm_nt<<<grid, 128, 0, s>>>(M, N, K, Am, lda, Bm, ldb, sc, C, ldc, acc ? 1 : 0, alpha));
  h->dgemm_flops += 2.0 * M * (double)N * K;
}

// Dense (spectral) assembly: per pair of state variables  Hd = sum_jk D_j' diag(h_jk) D_k  (n x n),  then
// A_top[a-block, b-block] = R_a' Hd R_b  by two GEMMs, written straight into the full row-major top matrix.
void Engine::assemble_dense(Amg &A, System &S, const NodeParams &P) {
  LAUNCH(KC_NODE_F2, launch_node<NODE_F2>(P, red_grid(A.n), s));
  SysLevel &top = S.lev[0];
  const int64_t m = top.m;
  const int n = (int)A.n, nK = S.nK;
  zero(top.A.val, m * m);
  if (S.kron) {
    // sum-factorised: per block of kept variables one small contraction over the fast index (k_kron_w), ONE DMMA GEMM over
    // (operator pair, slow index) against the constant factor table, and the index permutation into the system matrix
    const int n1 = A.kron_n1;
    for (const System::KronPair &kp : S.kp) {
      KronWArgs W;
      memset(&W, 0, sizeof(W));
      W.n1 = n1;
      W.c2a = kp.c2a;
      W.c2b = kp.c2b;
      W.ncombo = kp.ncombo;
      W.K = kp.ncombo * n1;
      for (int c = 0; c < kp.ncombo; ++c) {
        W.c[c].Qj = kp.Qj[c];
        W.c[c].Qk = kp.Qk[c];
        W.c[c].h = A.Hn + (int64_t)kp.hidx[c] * A.n;
      }
      const size_t smem = sizeof(double) * ((size_t)n1 + (size_t)n1 * kp.c2a + (size_t)n1 * kp.c2b);
      LAUNCH(KC_DENSE, k_kron_w<<<kp.ncombo * n1, 256, smem, s>>>(W, S.Wcat));
      const int Mr = kp.c1a * kp.c1b, Nc = kp.c2a * kp.c2b;
      dgemm_nt(Mr, Nc, W.K, kp.AA, W.K, S.Wcat, W.K, nullptr, S.Hd, Nc, false);
      LAUNCH(KC_DENSE, k_kron_scatter<<<nblk((int64_t)Mr * Nc), 256, 0, s>>>(kp.c1a, kp.c2a, kp.c1b, kp.c2b, S.Hd, top.A.val, m, kp.offa, kp.offb));
    }
    setup_hierarchy(A, S, 0);
    return;
  }
  for (size_t qa = 0; qa < S.kept.size(); ++qa)
    for (size_t qb = 0; qb < S.kept.size(); ++qb) {
      const int va = S.kept[qa], vb = S.kept[qb];
      bool any = false;
      zero(S.Hd, (int64_t)n * n);
      for (int ja = 0; ja < nK; ++ja) {
        const int j = S.Krow[ja];
        if (A.D_var[j] != va) continue;
        for (int kb = 0; kb < nK; ++kb) {
          const int k = S.Krow[kb];
          if (A.D_var[k] != vb) continue;
          any = true;
          const int a = std::min(ja, kb), b = std::max(ja, kb);
          const double *hv = A.Hn + (int64_t)(a * nK - (a * (a - 1)) / 2 + (b - a)) * A.n;
          const int oj = A.D_op[j], ok = A.D_op[k];
          if (oj < 0 && ok < 0) LAUNCH(KC_DENSE, k_dense_hess_ident<<<nblk(n), 256, 0, s>>>(n, 0, hv, nullptr, S.Hd));
          else if (oj < 0) LAUNCH(KC_DENSE, k_dense_hess_ident<<<nblk((int64_t)n * n), 256, 0, s>>>(n, 1, hv, A.ops[ok], S.Hd));
          else if (ok < 0) LAUNCH(KC_DENSE, k_dense_hess_ident<<<nblk((int64_t)n * n), 256, 0, s>>>(n, 2, hv, A.ops[oj], S.Hd));
          else dgemm_nt(n, n, n, A.ops[oj], n, A.ops[ok], n, hv, S.Hd, n, true);
        }
      }
      if (!any) continue;
      const int ma = (int)(top.off[qa + 1] - top.off[qa]), mb = (int)(top.off[qb + 1] - top.off[qb]);
      dgemm_nt(mb, n, n, S.Rt[qb], n, S.Hd, n, nullptr, S.Wt, n, false);                                   // Wt = (Hd R_b)'
      dgemm_nt(ma, mb, n, S.Rt[qa], n, S.Wt, n, nullptr, top.A.val + top.off[qa] * m + top.off[qb], m, false);   // R_a' Hd R_b
    }
  setup_hierarchy(A, S, 0);
}

}  // namespace mgbx
