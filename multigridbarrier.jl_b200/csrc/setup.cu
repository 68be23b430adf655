// setup.cu -- construction of everything the Newton iterations reuse: the AMG state and the convex set uploaded from
// the ABI structs, and per linear-system family the top-level assembly plan and the Galerkin hierarchy, built on the
// device (setup_kernels.cuh).
#include "engine.hpp"
#include "setup_kernels.cuh"

namespace mgbx {

DevCsr upload_csr(Pool &pool, const HostCsr &H, cudaStream_t s, bool with_values = true) {
  DevCsr D;
  D.rows = H.rows;
  D.cols = H.cols;
  D.nnz = H.nnz();
  D.ptr = pool.upload<int64_t>(H.ptr.data(), H.ptr.size(), s);
  D.idx = pool.upload<int32_t>(H.idx.data(), H.idx.size(), s);
  if (with_values && !H.val.empty()) D.val = pool.upload<double>(H.val.data(), H.val.size(), s);
  else D.val = pool.zeros<double>(H.idx.size(), s);
  return D;
}


// temporary device CSR (plan construction only), freed explicitly
struct TempCsr {
  DevCsr d;
  cudaStream_t s = nullptr;
  void free_all() {
    if (d.ptr) cudaFreeAsync(d.ptr, s);
    if (d.idx) cudaFreeAsync(d.idx, s);
    if (d.val) cudaFreeAsync(d.val, s);
    d = DevCsr();
  }
};
TempCsr upload_csr_temp(const HostCsr &H, cudaStream_t s, bool with_values) {
  TempCsr T;
  T.s = s;
  T.d.rows = H.rows;
  T.d.cols = H.cols;
  T.d.nnz = H.nnz();
  CK(cudaMallocAsync((void **)&T.d.ptr, sizeof(int64_t) * (H.rows + 1), s));
  CK(cudaMallocAsync((void **)&T.d.idx, sizeof(int32_t) * std::max<int64_t>(1, H.nnz()), s));
  CK(cudaMemcpyAsync(T.d.ptr, H.ptr.data(), sizeof(int64_t) * (H.rows + 1), cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(T.d.idx, H.idx.data(), sizeof(int32_t) * H.nnz(), cudaMemcpyHostToDevice, s));
  if (with_values && !H.val.empty()) {
    CK(cudaMallocAsync((void **)&T.d.val, sizeof(double) * std::max<int64_t>(1, H.nnz()), s));
    CK(cudaMemcpyAsync(T.d.val, H.val.data(), sizeof(double) * H.nnz(), cudaMemcpyHostToDevice, s));
  }
  CK(cudaStreamSynchronize(s));
  return T;
}
// (row << 32 | col) keys (unsorted, duplicates allowed) -> CSR pattern with sorted columns; consumes `keys`.
// drop_sentinel: keys equal to ~0 (padding of the multi-GPU all-gather) are discarded.
DevCsr csr_from_keys(Pool &pool, unsigned long long *keys, int64_t total, int64_t rows, int64_t cols, bool drop_sentinel, cudaStream_t s) {
  DevCsr C;
  C.rows = rows;
  C.cols = cols;
  if (total > INT32_MAX) throw std::runtime_error("csr_from_keys: more than 2^31 candidate entries");
  unsigned long long *keys2 = tmp_alloc<unsigned long long>(total, s);
  int *nsel = tmp_alloc<int>(1, s);
  int nnz = 0;
  if (total > 0) {
    size_t tmp_bytes = 0;
    const int end_bit = 64;
    CK(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, keys, keys2, (int)total, 0, end_bit, s));
    char *tmp = tmp_alloc<char>(tmp_bytes, s);
    CK(cub::DeviceRadixSort::SortKeys(tmp, tmp_bytes, keys, keys2, (int)total, 0, end_bit, s));
    tmp_free(tmp, s);
    CK(cub::DeviceSelect::Unique(nullptr, tmp_bytes, keys2, keys, nsel, (int)total, s));
    tmp = tmp_alloc<char>(tmp_bytes, s);
    CK(cub::DeviceSelect::Unique(tmp, tmp_bytes, keys2, keys, nsel, (int)total, s));
    tmp_free(tmp, s);
    CK(cudaMemcpyAsync(&nnz, nsel, sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (drop_sentinel && nnz > 0) {
      unsigned long long last = 0;
      CK(cudaMemcpyAsync(&last, keys + (nnz - 1), sizeof(last), cudaMemcpyDeviceToHost, s));
      CK(cudaStreamSynchronize(s));
      if (last == ~0ull) --nnz;
    }
  }
  C.nnz = nnz;
  C.ptr = pool.alloc<int64_t>(C.rows + 1);
  C.idx = pool.alloc<int32_t>(C.nnz);
  C.val = pool.zeros<double>(C.nnz, s);
  k_sym_finish<<<nblk(std::max<int64_t>(C.nnz, C.rows + 1)), 256, 0, s>>>(keys, C.nnz, C.rows, C.ptr, C.idx);
  CK(cudaGetLastError());
  tmp_free(keys, s);
  tmp_free(keys2, s);
  tmp_free(nsel, s);
  CK(cudaStreamSynchronize(s));
  return C;
}

// Multi-GPU: the union over the ranks of the local top-level patterns (each rank sees only its elements), so that
// every rank assembles into the SAME CSR structure and the values can be all-reduced.
DevCsr global_pattern(int nranks, void *comm, Pool &pool, const HostCsr &pat, cudaStream_t s) {
  NcclApi &N = nccl_api();
  const int64_t nloc = pat.nnz();
  std::vector<unsigned long long> hk(nloc);
  for (int64_t i = 0; i < pat.rows; ++i)
    for (int64_t k = pat.ptr[i]; k < pat.ptr[i + 1]; ++k) hk[k] = ((unsigned long long)i << 32) | (unsigned int)pat.idx[k];
  int64_t *dcnt = tmp_alloc<int64_t>(nranks + 1, s);
  CK(cudaMemcpyAsync(dcnt + nranks, &nloc, sizeof(int64_t), cudaMemcpyHostToDevice, s));
  NCK(N.AllGather(dcnt + nranks, dcnt, 1, kNcclInt64, comm, s));
  std::vector<int64_t> cnt(nranks);
  CK(cudaMemcpyAsync(cnt.data(), dcnt, sizeof(int64_t) * nranks, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  tmp_free(dcnt, s);
  const int64_t maxc = *std::max_element(cnt.begin(), cnt.end());
  unsigned long long *send = tmp_alloc<unsigned long long>(maxc, s);
  unsigned long long *all = tmp_alloc<unsigned long long>(maxc * nranks, s);
  CK(cudaMemsetAsync(send, 0xff, sizeof(unsigned long long) * std::max<int64_t>(1, maxc), s));
  CK(cudaMemcpyAsync(send, hk.data(), sizeof(unsigned long long) * nloc, cudaMemcpyHostToDevice, s));
  NCK(N.AllGather(send, all, (size_t)maxc, kNcclUint64, comm, s));
  CK(cudaStreamSynchronize(s));
  tmp_free(send, s);
  return csr_from_keys(pool, all, maxc * nranks, pat.rows, pat.cols, true, s);
}

// Sparsity pattern of A*B on the device: candidate keys (row << 32 | col) -> radix sort -> unique -> CSR.
DevCsr device_symbolic(Pool &pool, const DevCsr &A, const DevCsr &B, cudaStream_t s) {
  if (A.cols != B.rows) throw std::runtime_error("device_symbolic: inner dimensions differ");
  DevCsr C;
  C.rows = A.rows;
  C.cols = B.cols;
  int64_t *cand = tmp_alloc<int64_t>(A.rows + 1, s), *offs = tmp_alloc<int64_t>(A.rows + 1, s);
  k_sym_count<<<nblk(A.rows + 1), 256, 0, s>>>(A, B, cand);
  CK(cudaGetLastError());
  size_t tmp_bytes = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, cand, offs, (int)(A.rows + 1), s));
  char *tmp = tmp_alloc<char>(tmp_bytes, s);
  CK(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, cand, offs, (int)(A.rows + 1), s));
  int64_t total = 0;
  CK(cudaMemcpyAsync(&total, offs + A.rows, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  tmp_free(tmp, s);
  if (total > INT32_MAX) {
    tmp_free(cand, s);
    tmp_free(offs, s);
    throw std::runtime_error("device_symbolic: more than 2^31 candidate entries");
  }
  unsigned long long *keys = tmp_alloc<unsigned long long>(total, s);
  if (total > 0) {
    k_sym_fill<<<nblk(A.rows), 256, 0, s>>>(A, B, offs, keys);
    CK(cudaGetLastError());
  }
  tmp_free(cand, s);
  tmp_free(offs, s);
  return csr_from_keys(pool, keys, total, C.rows, C.cols, false, s);
}

// two-pass sliced-ELL construction shared by the device plan builders: COUNT(P, width) then FILL(P)
template <class CountFn, class FillFn>
SellPlan build_sell_two_pass(Pool &pool, int64_t nout, bool with_weights, cudaStream_t s, CountFn count, FillFn fill) {
  SellPlan P;
  P.nout = nout;
  P.nslices = (nout + 31) / 32;
  if (nout == 0) return P;
  int32_t *width = tmp_alloc<int32_t>(P.nslices, s);
  P.cnt = pool.alloc<int32_t>(nout);
  count(P, width);
  CK(cudaGetLastError());
  std::vector<int32_t> hwid(P.nslices);
  CK(cudaMemcpyAsync(hwid.data(), width, sizeof(int32_t) * P.nslices, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  std::vector<int64_t> sptr(P.nslices + 1, 0);
  for (int64_t sl = 0; sl < P.nslices; ++sl) sptr[sl + 1] = sptr[sl] + 32 * (int64_t)hwid[sl];
  P.nterms = sptr[P.nslices];
  P.sptr = pool.upload<int64_t>(sptr.data(), sptr.size(), s);
  P.src = pool.zeros<int32_t>(P.nterms, s);
  P.w = with_weights ? pool.zeros<double>(P.nterms, s) : nullptr;
  fill(P, width);
  CK(cudaGetLastError());
  tmp_free(width, s);
  CK(cudaStreamSynchronize(s));
  return P;
}

// Term list of the sparse product C = Lm * Rm, built on the device (one thread per non-zero of C; two passes).
SellPlan device_product_plan(Pool &pool, const DevCsr &Lm, const DevCsr &Rm, const DevCsr &C, bool variable_left, cudaStream_t s) {
  if (Lm.nnz > INT32_MAX || Rm.nnz > INT32_MAX || C.rows > INT32_MAX) throw std::runtime_error("product plan: index exceeds 32 bits");
  if (C.nnz == 0) return SellPlan();
  int32_t *rowof = tmp_alloc<int32_t>(C.nnz, s);
  k_csr_rows<<<nblk(C.rows), 256, 0, s>>>(C, rowof);
  const unsigned int g = nblk(((C.nnz + 31) / 32) * 32);
  const int vl = variable_left ? 1 : 0;
  SellPlan P = build_sell_two_pass(
      pool, C.nnz, true, s, [&](SellPlan &Q, int32_t *width) { k_prod_plan<0><<<g, 256, 0, s>>>(Lm, Rm, C, rowof, vl, Q, width); },
      [&](SellPlan &Q, int32_t *width) { k_prod_plan<1><<<g, 256, 0, s>>>(Lm, Rm, C, rowof, vl, Q, width); });
  tmp_free(rowof, s);
  return P;
}
// Is the prolongation block B (rows: the variable's n = N p broken nodes, cols: its fine-level coefficients) element-local?
// Every column must be supported inside one element's node range, every element must own the same number nc <= kElemMaxNc
// of consecutive columns.  Returns nc (0: not element-local) and fills c0 (first column per element) and P (N x p x nc).
static int element_local_blocks(const HostCsr &B, int64_t N, int p, std::vector<int64_t> &c0, std::vector<double> &P) {
  const HostCsr Bt = transpose(B);
  std::vector<int64_t> elem_of(Bt.rows, -1);
  for (int64_t c = 0; c < Bt.rows; ++c) {
    if (Bt.ptr[c] == Bt.ptr[c + 1]) return 0;
    const int64_t e = Bt.idx[Bt.ptr[c]] / p;
    for (int64_t k = Bt.ptr[c]; k < Bt.ptr[c + 1]; ++k)
      if (Bt.idx[k] / p != e) return 0;
    elem_of[c] = e;
  }
  c0.assign(N, -1);
  std::vector<int> cnt(N, 0);
  for (int64_t c = 0; c < Bt.rows; ++c) {
    const int64_t e = elem_of[c];
    if (c0[e] < 0) c0[e] = c;
    else if (c != c0[e] + cnt[e]) return 0;   // the element's columns must be consecutive
    cnt[e]++;
  }
  const int nc = N > 0 ? cnt[0] : 0;
  for (int64_t e = 0; e < N; ++e)
    if (cnt[e] != nc) return 0;
  if (nc < 1 || nc > kElemMaxNc) return 0;
  P.assign((size_t)N * p * nc, 0.0);
  for (int64_t i = 0; i < B.rows; ++i)
    for (int64_t k = B.ptr[i]; k < B.ptr[i + 1]; ++k) {
      const int64_t e = i / p;
      P[(size_t)i * nc + (B.idx[k] - c0[e])] = B.val.empty() ? 1.0 : B.val[k];
    }
  return nc;
}

// -------------------------------------------------------------------------------------------------
// host-side plan construction
// -------------------------------------------------------------------------------------------------
// Build the index plans of one linear-system family.  ltop: the AMG level the top matrix lives on.  The top
// matrix is assembled directly from the element blocks with R_top = R_fine[ltop] (= R_fine[L-1] * T[L-2] ... T[ltop]),
// every coarser level by Galerkin gather plans.
std::unique_ptr<System> build_system(mgbx_handle *h, Amg &A, bool condensed, int ltop) {
  auto S = std::make_unique<System>();
  Pool &pool = h->pool;
  pool.cat = "system: patterns, gather plans, level vectors";
  cudaStream_t s = h->stream;
  const int L = ltop + 1;            // levels 0..ltop take part
  S->condensed = condensed;
  S->ltop = ltop;
  if (condensed && ltop != A.L - 1) throw std::runtime_error("internal: condensation only at the fine level");
  // prolongation from the top level of this system to the broken fine space
  HostCsr Rtop_store;
  const HostCsr *Rtop_p = &A.hRL;
  if (ltop != A.L - 1) {
    Rtop_store = A.hRL;
    for (int l = A.L - 2; l >= ltop; --l) Rtop_store = spgemm_numeric_host(Rtop_store, A.hT[l]);
    Rtop_p = &Rtop_store;
  }
  const HostCsr &Rtop = *Rtop_p;
  // which variables can be eliminated node-locally at the fine level: R block == identity and every D row is :id
  std::vector<char> is_elim(A.nu, 0);
  if (condensed) {
    for (int v = 0; v < A.nu; ++v) {
      const int64_t c0 = A.voff[L - 1][v], c1 = A.voff[L - 1][v + 1];
      if (c1 - c0 != A.n) continue;
      bool idonly = true, any = false;
      for (int j = 0; j < A.nD; ++j)
        if (A.D_var[j] == v) {
          any = true;
          if (A.D_op[j] >= 0) idonly = false;
        }
      if (!any || !idonly) continue;
      HostCsr blk = submatrix(Rtop, (int64_t)v * A.n, (int64_t)(v + 1) * A.n, c0, c1);
      if (is_identity(blk)) is_elim[v] = 1;
    }
    int ne = 0;
    for (int v = 0; v < A.nu; ++v) ne += is_elim[v];
    if (ne > 4) {   // keep at most 4 eliminated variables (register budget of the node kernel)
      for (int v = A.nu - 1; v >= 0 && ne > 4; --v)
        if (is_elim[v]) {
          is_elim[v] = 0;
          --ne;
        }
    }
    if (ne == A.nu) is_elim[0] = 0;   // keep at least one variable in the reduced system
    // otherwise, an element-local variable (single GPU): eliminated exactly element by element (elem_schur.cuh)
    if (ne == 0 && A.nu > 1 && h->nranks == 1 && A.p <= kElemMaxP)
      for (int v = 0; v < A.nu && !S->elem_local; ++v) {
        bool idonly = true, any = false;
        for (int j = 0; j < A.nD; ++j)
          if (A.D_var[j] == v) {
            any = true;
            if (A.D_op[j] >= 0) idonly = false;
          }
        int coupled = 0;   // kept variables with D rows: Y has one p-column block per such variable
        for (int u = 0; u < A.nu; ++u) {
          bool rows = false;
          for (int j = 0; j < A.nD; ++j) rows = rows || (u != v && A.D_var[j] == u);
          coupled += rows ? 1 : 0;
        }
        if (!any || !idonly || coupled > 2) continue;
        std::vector<int64_t> c0;
        std::vector<double> Pe;
        const int nc = element_local_blocks(submatrix(Rtop, (int64_t)v * A.n, (int64_t)(v + 1) * A.n, A.voff[L - 1][v], A.voff[L - 1][v + 1]),
                                            A.N, A.p, c0, Pe);
        if (nc == 0) continue;
        is_elim[v] = 1;
        S->elem_local = true;
        S->el.nc = nc;
        S->el.c0 = pool.upload<int64_t>(c0.data(), c0.size(), s);
        S->el.P = pool.upload<double>(Pe.data(), Pe.size(), s);
        S->el.R = pool.zeros<double>((size_t)A.N * elem_rsize(nc), s);
      }
  }
  for (int v = 0; v < A.nu; ++v) (is_elim[v] ? S->elim : S->kept).push_back(v);
  S->nE = (int)S->elim.size();
  if (condensed)
    for (int v = 0; v < A.nu; ++v) {
      bool idonly = true, any = false;
      for (int j = 0; j < A.nD; ++j)
        if (A.D_var[j] == v) {
          any = true;
          if (A.D_op[j] >= 0) idonly = false;
        }
      if (any && idonly && !is_elim[v] && A.nu > 1) S->uncondensed_slack = true;
    }
  // row classification
  S->nK = 0;
  for (int j = 0; j < A.nD; ++j) {
    S->Erow[j] = -1;
    for (int e = 0; e < S->nE; ++e)
      if (S->elim[e] == A.D_var[j]) S->Erow[j] = e;
    if (S->Erow[j] < 0) S->Krow[S->nK++] = j;
  }
  // variables of the kept set that own at least one D row form the block pairs
  std::vector<int> used;
  for (int v : S->kept) {
    bool any = false;
    for (int j = 0; j < A.nD; ++j) any = any || (A.D_var[j] == v);
    if (any) used.push_back(v);
  }
  if ((int)(used.size() * used.size()) > 16) throw ArgError("too many coupled state variables (max 4 kept variables)");
  S->pl.npairs = 0;
  for (int a : used)
    for (int b : used) {
      S->pl.va[S->pl.npairs] = a;
      S->pl.vb[S->pl.npairs] = b;
      S->pl.npairs++;
    }
  // levels
  const int nlev = L;
  S->lev.resize(nlev);
  for (int k = 0; k < nlev; ++k) {
    const int l = L - 1 - k;
    SysLevel &Lv = S->lev[k];
    Lv.off.assign(1, 0);
    for (int v : S->kept) Lv.off.push_back(Lv.off.back() + (A.voff[l][v + 1] - A.voff[l][v]));
    Lv.m = Lv.off.back();
  }
  if (dense_mode(A)) {
    // ---- dense (spectral) system: full m x m matrix assembled by GEMMs, solved directly; no plans, no hierarchy
    S->dense = true;
    S->lev.resize(1);
    SysLevel &Lv = S->lev[0];
    const int64_t m = Lv.m;
    if (m > kDenseMaxUnknowns) throw std::runtime_error("dense (spectral) Newton systems are limited to 8192 unknowns in this build");
    HostCsr full;
    full.rows = full.cols = m;
    full.ptr.resize(m + 1);
    full.idx.resize((size_t)m * m);
    for (int64_t i = 0; i <= m; ++i) full.ptr[i] = i * m;
    for (int64_t i = 0; i < m; ++i)
      for (int64_t j = 0; j < m; ++j) full.idx[i * m + j] = (int32_t)j;
    Lv.A = upload_csr(pool, full, s, false);
    Lv.spmv_group = 32;
    Lv.x2 = pool.alloc<double>(m);   // scratch of the direct solve (Engine::direct_solve)
    Lv.r = pool.alloc<double>(m);
    TempCsr rt = upload_csr_temp(Rtop, s, true);
    int64_t mvmax = 1;
    for (size_t q = 0; q < S->kept.size(); ++q) {
      const int v = S->kept[q];
      const int64_t mv = Lv.off[q + 1] - Lv.off[q];
      mvmax = std::max(mvmax, mv);
      double *d = pool.zeros<double>((size_t)mv * A.n, s);
      k_csr_block_to_dense_t<<<nblk(A.n), 256, 0, s>>>(rt.d, (int64_t)v * A.n, (int)A.n, A.voff[L - 1][v], (int)mv, d);
      CK(cudaGetLastError());
      S->Rt.push_back(d);
    }
    CK(cudaStreamSynchronize(s));
    rt.free_all();
    S->Hd = pool.alloc<double>((size_t)A.n * A.n);
    S->Wt = pool.alloc<double>((size_t)mvmax * A.n);
    S->cut = -1;
    // ---- sum-factorised assembly when every operator and every prolongation block is a Kronecker product
    if (h->cfg.spectral_kron && A.kron_n1 > 0 && S->nE == 0) {
      const int n1 = A.kron_n1;
      const size_t nk = S->kept.size();
      std::vector<std::vector<double>> R1a(nk), R1b(nk);
      std::vector<int> cq(nk, 0);
      bool ok = true;
      for (size_t q = 0; q < nk && ok; ++q) {
        const int v = S->kept[q];
        const int64_t mv = Lv.off[q + 1] - Lv.off[q];
        const int c = isqrt_exact(mv);
        if (c <= 0 || c > n1) {
          ok = false;
          break;
        }
        std::vector<double> dense((size_t)A.n * mv, 0.0);
        const int64_t c0 = A.voff[L - 1][v];
        for (int64_t i = 0; i < A.n; ++i)
          for (int64_t k = Rtop.ptr[(int64_t)v * A.n + i]; k < Rtop.ptr[(int64_t)v * A.n + i + 1]; ++k) {
            const int64_t cc = Rtop.idx[k] - c0;
            if (cc >= 0 && cc < mv) dense[(size_t)i * mv + cc] = Rtop.val[k];
          }
        cq[q] = c;
        ok = kron_factor([&](int64_t r, int64_t cc) { return dense[(size_t)r * mv + cc]; }, n1, n1, c, c, R1a[q], R1b[q]);
      }
      if (ok) {
        // per D row j: P_j = A_j R1a_v, Q_j = B_j R1b_v  (n1 x c_v); identity operators have A_j = B_j = I
        std::vector<std::vector<double>> Pj(S->nK), Qj(S->nK);
        std::vector<const double *> Qdev(S->nK, nullptr);
        std::vector<int> qof(S->nK, -1);
        auto mul = [&](const std::vector<double> *F, const std::vector<double> &Rm, int c) {
          if (!F) return Rm;
          std::vector<double> out((size_t)n1 * c, 0.0);
          for (int e = 0; e < n1; ++e)
            for (int g = 0; g < n1; ++g) {
              const double f = (*F)[(size_t)e * n1 + g];
              if (f != 0.0)
                for (int i = 0; i < c; ++i) out[(size_t)e * c + i] += f * Rm[(size_t)g * c + i];
            }
          return out;
        };
        for (int a = 0; a < S->nK; ++a) {
          const int j = S->Krow[a], v = A.D_var[j], o = A.D_op[j];
          for (size_t q = 0; q < nk; ++q)
            if (S->kept[q] == v) qof[a] = (int)q;
          if (qof[a] < 0) continue;
          Pj[a] = mul(o >= 0 ? &A.kronA[o] : nullptr, R1a[qof[a]], cq[qof[a]]);
          Qj[a] = mul(o >= 0 ? &A.kronB[o] : nullptr, R1b[qof[a]], cq[qof[a]]);
          Qdev[a] = pool.upload<double>(Qj[a].data(), Qj[a].size(), s);
        }
        size_t wmax = 0;
        for (size_t qa = 0; qa < nk && ok; ++qa)
          for (size_t qb = 0; qb < nk && ok; ++qb) {
            System::KronPair kp;
            kp.c1a = kp.c2a = cq[qa];
            kp.c1b = kp.c2b = cq[qb];
            kp.offa = Lv.off[qa];
            kp.offb = Lv.off[qb];
            std::vector<std::pair<int, int>> combos;
            for (int ja = 0; ja < S->nK; ++ja)
              for (int kb = 0; kb < S->nK; ++kb)
                if (qof[ja] == (int)qa && qof[kb] == (int)qb) combos.push_back({ja, kb});
            if (combos.empty()) continue;
            if ((int)combos.size() > kKronMaxCombos) {
              ok = false;
              break;
            }
            kp.ncombo = (int)combos.size();
            const int64_t Mr = (int64_t)kp.c1a * kp.c1b, K = (int64_t)kp.ncombo * n1;
            std::vector<double> AA((size_t)Mr * K);
            for (int c = 0; c < kp.ncombo; ++c) {
              const int ja = combos[c].first, kb = combos[c].second;
              const int lo = std::min(ja, kb), hi = std::max(ja, kb);
              kp.hidx[c] = lo * S->nK - (lo * (lo - 1)) / 2 + (hi - lo);
              kp.Qj[c] = Qdev[ja];
              kp.Qk[c] = Qdev[kb];
              for (int i = 0; i < kp.c1a; ++i)
                for (int l = 0; l < kp.c1b; ++l)
                  for (int e = 0; e < n1; ++e)
                    AA[((size_t)i * kp.c1b + l) * K + (size_t)c * n1 + e] = Pj[ja][(size_t)e * kp.c1a + i] * Pj[kb][(size_t)e * kp.c1b + l];
            }
            kp.AA = pool.upload<double>(AA.data(), AA.size(), s);
            wmax = std::max(wmax, (size_t)kp.c2a * kp.c2b * (size_t)K);
            S->kp.push_back(kp);
          }
        if (ok && !S->kp.empty()) {
          S->Wcat = pool.alloc<double>(wmax);
          S->kron = true;
          const size_t smem = sizeof(double) * ((size_t)n1 + 2 * (size_t)n1 * n1);
          kron_w_init(smem);
        } else {
          S->kp.clear();
        }
      }
      if (h->cfg.verbose > 0) fprintf(stderr, "[mgbx] build_system(dense, level %d): sum-factorised (Kronecker) assembly %s\n", ltop, S->kron ? "on" : "not applicable");
    }
    CK(cudaStreamSynchronize(s));
    if (h->cfg.verbose > 0) fprintf(stderr, "[mgbx] build_system(dense, level %d): m=%lld, n=%lld\n", ltop, (long long)m, (long long)A.n);
    return S;
  }
  // top pattern = reference plan pattern restricted to the kept variables
  const int64_t mtop = S->lev[0].m;
  std::vector<int64_t> colmap(A.m[L - 1], -1);
  for (size_t q = 0; q < S->kept.size(); ++q) {
    const int v = S->kept[q];
    for (int64_t c = A.voff[L - 1][v]; c < A.voff[L - 1][v + 1]; ++c) colmap[c] = S->lev[0].off[q] + (c - A.voff[L - 1][v]);
  }
  HostTimer tm;
  const bool vb = h->cfg.verbose > 0;
  HostCsr Einc = element_incidence(Rtop, A.N, A.p, used, A.n, colmap, mtop);
  HostCsr pat = plan_pattern(Einc);
  if (vb) fprintf(stderr, "[mgbx] build_system(cond=%d): pattern m=%lld nnz=%lld %.3fs\n", (int)condensed, (long long)mtop, (long long)pat.nnz(), tm.lap());   // (local pattern on a multi-GPU rank)
  // gather plan, built on the device: for each nz of the pattern, the Hblk entries (and weights) that sum into it
  const int p = A.p;
  const int64_t pp = (int64_t)p * p;
  S->hblk_size = (int64_t)S->pl.npairs * A.N * pp;
  if (S->hblk_size > INT32_MAX) throw std::runtime_error("element block array exceeds 32-bit gather indices");
  // multi-GPU: each rank sees only its own elements; the CSR structure is the union over the ranks
  S->lev[0].A = (h->nranks > 1) ? global_pattern(h->nranks, h->comm, pool, pat, s) : upload_csr(pool, pat, s, false);
  const int64_t top_nnz = S->lev[0].A.nnz;
  {
    bool unit = true;
    for (double v : Rtop.val)
      if (v != 1.0) {
        unit = false;
        break;
      }
    TempCsr einct = upload_csr_temp(transpose(Einc), s, false);
    TempCsr rtmp;
    TopPlanParams Q;
    memset(&Q, 0, sizeof(Q));
    if (ltop == A.L - 1) Q.R = A.RL;
    else {
      rtmp = upload_csr_temp(Rtop, s, true);
      Q.R = rtmp.d;
    }
    Q.EincT = einct.d;
    Q.pat = S->lev[0].A;
    Q.n = A.n;
    Q.N = A.N;
    Q.p = p;
    Q.unit = unit ? 1 : 0;
    Q.nkept = (int)S->kept.size();
    for (int q = 0; q < Q.nkept; ++q) {
      Q.kept[q] = S->kept[q];
      Q.off[q] = S->lev[0].off[q];
      Q.rcol0[q] = A.voff[L - 1][S->kept[q]];
    }
    Q.off[Q.nkept] = S->lev[0].off[Q.nkept];
    for (int qa = 0; qa < Q.nkept; ++qa)
      for (int qb = 0; qb < Q.nkept; ++qb) {
        int pr = -1;
        for (int k = 0; k < S->pl.npairs; ++k)
          if (S->pl.va[k] == S->kept[qa] && S->pl.vb[k] == S->kept[qb]) pr = k;
        Q.pair_of[qa * Q.nkept + qb] = pr;
      }
    int32_t *rowof = tmp_alloc<int32_t>(top_nnz, s);
    k_csr_rows<<<nblk(pat.rows), 256, 0, s>>>(S->lev[0].A, rowof);
    Q.rowof = rowof;
    const unsigned int g = nblk(((top_nnz + 31) / 32) * 32);
    S->top = build_sell_two_pass(
        pool, top_nnz, !unit, s, [&](SellPlan &P, int32_t *width) { k_top_plan<0><<<g, 256, 0, s>>>(Q, P, width); },
        [&](SellPlan &P, int32_t *width) { k_top_plan<1><<<g, 256, 0, s>>>(Q, P, width); });
    tmp_free(rowof, s);
    einct.free_all();
    if (rtmp.d.ptr) rtmp.free_all();
  }
  pool.cat = "system: element block Hessians";
  S->Hblk = pool.alloc<double>(S->hblk_size);
  pool.cat = "system: Galerkin patterns and term lists";
  if (vb) fprintf(stderr, "[mgbx]   gather plan (%lld padded terms) %.3fs\n", (long long)S->top.nterms, tm.lap());
  // hierarchy patterns (device symbolic products) and Galerkin gather plans
  for (int k = 0; k < nlev; ++k) {
    SysLevel &Lv = S->lev[k];
    const int l = L - 1 - k;
    Lv.spmv_group = Engine::group_for(Lv.A);
    Lv.dinv = pool.alloc<double>(Lv.m);
    Lv.diag = pool.alloc<double>(Lv.m);
    Lv.lam = pool.zeros<double>(1, s);
    Lv.b = pool.alloc<double>(Lv.m);
    Lv.x = pool.alloc<double>(Lv.m);
    Lv.x2 = pool.alloc<double>(Lv.m);
    Lv.r = pool.alloc<double>(Lv.m);
    if (k + 1 < nlev) {
      // transfer from level l-1 to level l restricted to the kept variables
      std::vector<HostCsr> blocks;
      for (int v : S->kept)
        blocks.push_back(submatrix(A.hT[l - 1], A.voff[l][v], A.voff[l][v + 1], A.voff[l - 1][v], A.voff[l - 1][v + 1]));
      HostCsr Tk = block_diag(blocks);
      Lv.T_identity = is_identity(Tk);
      HostCsr Ttk = transpose(Tk);
      Lv.T = upload_csr(pool, Tk, s);
      Lv.Tt = upload_csr(pool, Ttk, s);
      if (Lv.T_identity) {
        S->lev[k + 1].A = Lv.A;   // same matrix: the coarser level aliases this one
      } else {
        const double t_host = tm.lap();
        Lv.AT = device_symbolic(pool, Lv.A, Lv.T, s);
        S->lev[k + 1].A = device_symbolic(pool, Lv.Tt, Lv.AT, s);
        const double t_sym = tm.lap();
        Lv.s1 = device_product_plan(pool, Lv.A, Lv.T, Lv.AT, true, s);
        Lv.s2 = device_product_plan(pool, Lv.Tt, Lv.AT, S->lev[k + 1].A, false, s);
        if (vb)
          fprintf(stderr, "[mgbx]   level %d: m=%lld -> %lld, nnz(A_c)=%lld, plan entries %lld + %lld, host %.3fs symbolic %.3fs plans %.3fs\n", k,
                  (long long)Lv.m, (long long)S->lev[k + 1].m, (long long)S->lev[k + 1].A.nnz, (long long)Lv.s1.nterms, (long long)Lv.s2.nterms,
                  t_host, t_sym, tm.lap());
      }
    }
  }
  // V-cycle cut: the first level small enough for the shared-memory dense inverse
  S->cut = -1;
  for (int k = 0; k < nlev; ++k)
    if (S->lev[k].m <= h->cfg.coarse_max) {
      S->cut = k;
      break;
    }
  const int64_t mx = S->lev[0].m;
  S->pc_r = pool.alloc<double>(mx);
  S->pc_p = pool.alloc<double>(mx);
  S->pc_p2 = pool.alloc<double>(mx);
  S->pc_Ap = pool.alloc<double>(mx);
  S->pc_x = pool.alloc<double>(mx);
  S->pc_b = pool.alloc<double>(mx);
  S->pcg_partials = pool.zeros<double>(3 * (size_t)kPcg2MaxGrid, s);
  S->pcg_out = pool.zeros<double>(8, s);
  S->pcg_bar = pool.zeros<unsigned int>(4, s);
  CK(cudaStreamSynchronize(s));
  return S;
}

System &Engine::system_for(Amg &A, int J) {
  if (dense_mode(A)) {
    auto &p = A.sys_dense[J];
    if (!p) p = build_system(h, A, false, J);
    return *p;
  }
  const bool fine = (J == A.L - 1);
  if (fine) {
    if (h->cfg.condense) {
      if (!A.sys_cond) A.sys_cond = build_system(h, A, true, A.L - 1);
      return *A.sys_cond;
    }
    if (!A.sys_hook) A.sys_hook = build_system(h, A, false, A.L - 1);
    return *A.sys_hook;
  }
  // coarse Newton levels (the recovery path of mgb_step): assembled directly at level L-2, Galerkin below
  if (!A.sys_coarse) A.sys_coarse = build_system(h, A, false, A.L - 2);
  return *A.sys_coarse;
}
// -------------------------------------------------------------------------------------------------
// create
// -------------------------------------------------------------------------------------------------
void upload_convex(mgbx_handle *h, const mgbx_convex &Q, int64_t n, int nD_user, ConvexDev &cd) {
  Pool &pool = h->pool;
  cudaStream_t s = h->stream;
  memset(&cd, 0, sizeof(cd));
  if (Q.npieces < 0 || Q.npieces > MGBX_MAX_PIECES) throw ArgError("convex set: unsupported number of pieces");
  cd.npieces = Q.npieces;
  for (int k = 0; k < Q.npieces; ++k) {
    const mgbx_piece &q = Q.pieces[k];
    PieceDev &d = cd.pc[k];
    if (q.kind != MGBX_PIECE_EP && q.kind != MGBX_PIECE_LINEAR) throw ArgError("convex piece: unknown kind");
    if (q.ni < 1 || q.ni > MGBX_MAX_NI || q.nc < 1 || q.nc > MGBX_MAX_NC) throw ArgError("convex piece: ni / nc out of range");
    if (q.kind == MGBX_PIECE_EP && q.nc != q.ni) throw ArgError("EP piece needs a square A (nc == ni == nz)");
    if (q.kind == MGBX_PIECE_EP && q.nc < 1) throw ArgError("EP piece needs nz >= 1");
    d.kind = q.kind;
    d.ni = q.ni;
    d.nc = q.nc;
    for (int c = 0; c < q.ni; ++c) {
      d.idx[c] = q.idx ? q.idx[c] : c;
      if (d.idx[c] < 0 || d.idx[c] >= nD_user) throw ArgError("convex piece indexes a D row that does not exist");
    }
    // grid compression: identity A / zero b / uniform p, mu are passed as constants (no HBM traffic)
    bool Aid = (q.nc == q.ni);
    if (Aid && q.A)
      for (int c = 0; c < q.ni && Aid; ++c)
        for (int r = 0; r < q.nc && Aid; ++r) {
          const double want = (r == c) ? 1.0 : 0.0;
          const double *col = q.A + (int64_t)(c * q.nc + r) * n;
          for (int64_t i = 0; i < n; ++i)
            if (col[i] != want) {
              Aid = false;
              break;
            }
        }
    if (!q.A && !(q.nc == q.ni)) throw ArgError("convex piece: A missing");
    d.A = (Aid || !q.A) ? nullptr : pool.upload<double>(q.A, (size_t)n * q.nc * q.ni, s);
    bool bz = true;
    if (q.b)
      for (int64_t i = 0; i < n * q.nc; ++i)
        if (q.b[i] != 0.0) {
          bz = false;
          break;
        }
    d.b = (bz || !q.b) ? nullptr : pool.upload<double>(q.b, (size_t)n * q.nc, s);
    d.p_uniform = 2.0;
    d.mu_uniform = 0.0;
    d.p = d.mu = nullptr;
    if (q.kind == MGBX_PIECE_EP) {
      if (!q.p || !q.mu) throw ArgError("EP piece: p / mu grids missing");
      bool pu = true, mu_u = true;
      for (int64_t i = 1; i < n; ++i) {
        if (q.p[i] != q.p[0]) pu = false;
        if (q.mu[i] != q.mu[0]) mu_u = false;
      }
      if (pu) d.p_uniform = q.p[0];
      else d.p = pool.upload<double>(q.p, n, s);
      if (mu_u) d.mu_uniform = q.mu[0];
      else d.mu = pool.upload<double>(q.mu, n, s);
    }
  }
  cd.select = nullptr;
  if (Q.select) {
    bool all = true;
    for (int64_t i = 0; i < n * Q.npieces; ++i)
      if (Q.select[i] == 0.0) {
        all = false;
        break;
      }
    if (!all) cd.select = pool.upload<double>(Q.select, (size_t)n * Q.npieces, s);
  }
  cd.feas = 0;
  cd.NC = nD_user + 1;
  cd.NF = nD_user;
}

void create_amg(mgbx_handle *h, const mgbx_amg &in, Amg &A) {
  Pool &pool = h->pool;
  cudaStream_t s = h->stream;
  if (in.n <= 0 || in.N <= 0 || in.p <= 0 || in.n != in.N * (int64_t)in.p) throw ArgError("amg: n must equal p*N");
  if (in.nu < 1 || in.nu > MGBX_MAX_ND) throw ArgError("amg: nu out of range");
  if (in.nD < 1 || in.nD > MGBX_MAX_ND) throw ArgError("amg: nD out of range (MGBX_MAX_ND)");
  if (in.L < 1 || in.L > MGBX_MAX_LEVELS) throw ArgError("amg: L out of range");
  if (in.nops < 0 || in.nops > MGBX_MAX_OPS) throw ArgError("amg: too many distinct operators");
  A.n = in.n;
  A.N = in.N;
  A.p = in.p;
  A.nu = in.nu;
  A.nD = in.nD;
  A.L = in.L;
  A.nops = in.nops;
  A.n_global = in.n_global > 0 ? in.n_global : in.n;
  A.var_local.assign(in.nu, 0);
  for (int v = 0; v < in.nu; ++v) A.var_local[v] = (in.var_local && in.var_local[v]) ? 1 : 0;
  A.any_local = false;
  for (char c : A.var_local) A.any_local = A.any_local || c;
  for (int j = 0; j < in.nD; ++j) {
    A.D_var[j] = in.D_var[j];
    A.D_op[j] = in.D_op[j];
    if (A.D_var[j] < 0 || A.D_var[j] >= in.nu) throw ArgError("amg: D row references a state variable that does not exist");
    if (A.D_op[j] >= in.nops) throw ArgError("amg: D row references an operator that does not exist");
  }
  const size_t ppN = (size_t)in.p * in.p * in.N;
  for (int o = 0; o < in.nops; ++o) A.ops[o] = pool.upload<double>(in.op_data[o], ppN, s);
  // dense (spectral) discretisation on a tensor grid: are all operators Kronecker products kron(A1, B1) of n1 x n1 factors
  // (src/spectral2d.jl:28-35)?  Then the Hessian assembly is sum-factorised (build_system, dense_kernels.cuh).
  A.kron_n1 = 0;
  if (in.N == 1 && in.p > 64 && in.nops > 0) {
    const int n1 = isqrt_exact(in.n);
    bool ok = n1 > 1;
    A.kronA.assign(in.nops, {});
    A.kronB.assign(in.nops, {});
    for (int o = 0; o < in.nops && ok; ++o) {
      const double *D = in.op_data[o];   // column-major n x n
      const int64_t nn = in.n;
      ok = kron_factor([&](int64_t r, int64_t c) { return D[r + c * nn]; }, n1, n1, n1, n1, A.kronA[o], A.kronB[o]);
    }
    if (ok) A.kron_n1 = n1;
  }
  A.w = pool.upload<double>(in.w, in.n, s);
  A.voff.resize(in.L);
  A.m.resize(in.L);
  if (!in.R_fine) throw ArgError("amg: R_fine missing");
  for (int l = 0; l < in.L; ++l) {
    // var_offsets == NULL: read the per-variable column blocks off R_fine[l] (what a shim that only sees the reference's
    // `AMG` struct can provide, src/multigrid.jl:278-288)
    if (in.var_offsets) A.voff[l].assign(in.var_offsets + (size_t)l * (in.nu + 1), in.var_offsets + (size_t)(l + 1) * (in.nu + 1));
    else A.voff[l] = derive_var_offsets(in.R_fine[l], in.nu, in.n);
    A.m[l] = A.voff[l][in.nu];
    if (A.voff[l][0] != 0) throw ArgError("amg: var_offsets must start at 0");
    for (int v = 0; v < in.nu; ++v)
      if (A.voff[l][v + 1] < A.voff[l][v]) throw ArgError("amg: var_offsets must be non-decreasing");
    if (l == in.L - 1 && (in.R_fine[l].cols != A.m[l] || in.R_fine[l].rows != (int64_t)in.nu * in.n))
      throw ArgError("amg: R_fine dimension mismatch (rows must be nu*n, cols must match var_offsets)");
  }
  HostTimer tm;
  const bool vb = h->cfg.verbose > 0;
  if (vb) fprintf(stderr, "[mgbx] create_amg: operators + weights queued %.3fs\n", tm.lap());
  A.hRL = csr_from_abi(in.R_fine[in.L - 1]);
  if (vb) fprintf(stderr, "[mgbx]   R_fine[L-1] checked/converted (nnz=%lld) %.3fs\n", (long long)A.hRL.nnz(), tm.lap());
  A.RL = upload_csr(pool, A.hRL, s);
  A.RLt = upload_csr(pool, transpose(A.hRL), s);
  if (vb) fprintf(stderr, "[mgbx]   R, R' uploaded %.3fs\n", tm.lap());
  A.hT.resize(std::max(0, in.L - 1));
  A.T.resize(A.hT.size());
  A.Tt.resize(A.hT.size());
  for (int l = 0; l + 1 < in.L; ++l) {
    if (in.T) {
      if (in.T[l].rows != A.m[l + 1] || in.T[l].cols != A.m[l]) throw ArgError("amg: T dimension mismatch");
      A.hT[l] = csr_from_abi(in.T[l]);
    } else {
      // the reference discards the level transfers (src/multigrid.jl:166-170): recover them from R_fine[l] = R_fine[l+1] T[l]
      if (in.R_fine[l].cols != A.m[l] || in.R_fine[l + 1].cols != A.m[l + 1]) throw ArgError("amg: R_fine[l] columns do not match var_offsets");
      A.hT[l] = recover_transfer(in.R_fine[l + 1], in.R_fine[l]);
    }
    A.T[l] = upload_csr(pool, A.hT[l], s);
    A.Tt[l] = upload_csr(pool, transpose(A.hT[l]), s);
  }
  if (vb) fprintf(stderr, "[mgbx]   level transfers %.3fs\n", tm.lap());
  const int64_t nun = (int64_t)in.nu * in.n;
  A.z = pool.zeros<double>(nun, s);
  A.zsave = pool.zeros<double>(nun, s);
  A.zinit = pool.zeros<double>(nun, s);
  A.zunfin = pool.zeros<double>(nun, s);
  A.zf = pool.zeros<double>(nun, s);
  A.gb = pool.zeros<double>(nun, s);
  A.G = pool.zeros<double>((size_t)in.n * in.nD, s);
  A.f = pool.zeros<double>((size_t)in.n * in.nD, s);
  A.Hn = pool.alloc<double>((size_t)in.n * (in.nD * (in.nD + 1) / 2));
  A.hEEinv = pool.alloc<double>((size_t)in.n * 10);
  A.hKE = pool.alloc<double>((size_t)in.n * in.nD * 4);
  A.slack = pool.alloc<double>(in.n);
  A.chain.resize(in.L);
  A.chain2.resize(in.L);
  for (int l = 0; l < in.L; ++l) {
    A.chain[l] = pool.alloc<double>(A.m[l]);
    A.chain2[l] = pool.alloc<double>(A.m[l]);
  }
  int64_t mmax = 0;
  for (int l = 0; l < in.L; ++l) mmax = std::max(mmax, A.m[l]);
  A.x = pool.zeros<double>(mmax, s);
  A.xn = pool.zeros<double>(mmax, s);
  A.g = pool.zeros<double>(mmax, s);
  A.gn = pool.zeros<double>(mmax, s);
  A.dir = pool.zeros<double>(mmax, s);
  A.rhs = pool.zeros<double>(mmax, s);
  A.tmp = pool.zeros<double>(mmax, s);
  A.xbest = pool.zeros<double>(mmax, s);
  A.gbest = pool.zeros<double>(mmax, s);
  CK(cudaStreamSynchronize(s));
  if (vb) fprintf(stderr, "[mgbx]   work vectors + sync %.3fs\n", tm.lap());
}


// feasibility AMG (src/multigrid.jl:522-536): state [user..., slack], rows [user D...; slack:id; each component:id]
void attach_feasibility(mgbx_handle *h, const mgbx_amg &a1) {
  Amg &A = h->amg[0];
  if (h->has_feas) throw ArgError("feasibility AMG already attached");
  if (a1.n != A.n || a1.nu != A.nu + 1 || a1.nD != A.nD + 1 + A.nu)
    throw ArgError("feasibility AMG must have nu+1 state variables and nD+1+nu rows (src/multigrid.jl:522-536)");
  create_amg(h, a1, h->amg[1]);
  Amg &F = h->amg[1];
  F.cd = A.cd;          // same grids, wrapped
  F.cd.feas = 1;
  F.cd.NC = A.nD + 1;
  F.cd.NF = F.nD;
  F.cd.fb = 1.0;
  F.cd.fR = 10.0;
  // phase-I cost: integral of the slack = row nD of D (0-based) (src/mgb.jl:446-448)
  std::vector<double> c1((size_t)F.n * F.nD, 0.0);
  for (int64_t i = 0; i < F.n; ++i) c1[(size_t)A.nD * F.n + i] = 1.0;
  CK(cudaMemcpyAsync(F.f, c1.data(), sizeof(double) * c1.size(), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->has_feas = true;
}

}  // namespace mgbx
