// TEST-ONLY shim (never part of libmgbx.so, never on a product path): the element-local elimination of a slack
// (csrc/elem_schur.cuh) on the CPU, fed by the per-node barrier arithmetic of csrc/node_barrier.cuh, exactly as the element
// kernels chain them for the default problem family: one Euclidean-power cone on (D_1 u, ..., D_dim u, s), the slack s = P c
// eliminated element by element.  Built by tests/test_elem_math.py.
#include <cstring>

#include "../../multigridbarrier.jl_b200/csrc/elem_schur.cuh"

using namespace mgbx;

// Per node i: inputs y = (D_1 u .. D_dim u, s) = Z[i*(dim+1) + .], barrier weight sc[i] (0: masked node).
// D: dim operators, D_a[r][c] = D[(a*p + c)*p + r] (the kernels' column-major blocks); P: p x nc row-major.
// stable = 1: node-local closed form (piece_eval `schur`) + Y'Y (elem_condense)  -- what the kernels compute;
// stable = 0: H_uu - H_us H_ss^-1 H_su formed by subtraction in double precision.
// Out: H (p x p row-major), Rf (packed R factor, stable = 1 only).
static void node_hess(int dim, const double *y, double pexp, double mu, bool schur, double *F2) {
  PieceDev pc;
  memset(&pc, 0, sizeof(pc));
  pc.kind = MGBX_PIECE_EP;
  pc.ni = pc.nc = dim + 1;
  for (int c = 0; c <= dim; ++c) pc.idx[c] = c;
  pc.p_uniform = pexp;
  pc.mu_uniform = mu;
  double F1[MGBX_MAX_ND];
  for (int k = 0; k <= dim; ++k) F1[k] = 0.0;
  for (int k = 0; k < (dim + 1) * (dim + 1); ++k) F2[k] = 0.0;
  piece_eval(pc, 1, 0, y, dim + 1, 2, false, 0.0, 0, F1, F2, schur);
}

extern "C" int hostcheck_elem_schur(int p, int nc, int dim, const double *P, const double *D, const double *Z, const double *sc, double pexp,
                                    double mu, int stable, double *H, double *Rf) {
  if (p > kElemMaxP || nc > kElemMaxNc || dim > 3) return -1;
  const int ny = dim + 1;
  double hww[kElemMaxP][9], hws[kElemMaxP][3], hss[kElemMaxP];
  for (int i = 0; i < p; ++i) {
    double F2[16];
    node_hess(dim, Z + i * ny, pexp, mu, stable != 0, F2);
    for (int a = 0; a < dim; ++a) {
      for (int b = 0; b < dim; ++b) hww[i][a * dim + b] = sc[i] * F2[a * ny + b];
      hws[i][a] = sc[i] * F2[a * ny + dim];
    }
    hss[i] = sc[i] * F2[dim * ny + dim];
  }
  auto Dop = [&](int a, int r, int c) { return D[((size_t)a * p + c) * p + r]; };
  // H_uu (node-local Schur complement when stable): sum_i sum_ab D_a[i][r] h_ab D_b[i][c]
  for (int r = 0; r < p; ++r)
    for (int c = 0; c < p; ++c) {
      double s = 0.0;
      for (int i = 0; i < p; ++i)
        for (int a = 0; a < dim; ++a)
          for (int b = 0; b < dim; ++b) s += Dop(a, i, r) * hww[i][a * dim + b] * Dop(b, i, c);
      H[r * p + c] = s;
    }
  // X[i][c] = sum_a q_a,i D_a[i][c]
  double X[kElemMaxP * kElemMaxP];
  for (int i = 0; i < p; ++i)
    for (int c = 0; c < p; ++c) {
      double s = 0.0;
      for (int a = 0; a < dim; ++a) s += hws[i][a] * Dop(a, i, c);
      X[i * p + c] = s;
    }
  if (stable) {
    double hinv[kElemMaxP];
    for (int i = 0; i < p; ++i) hinv[i] = 1.0 / hss[i];   // 1/0 = inf on masked nodes, as the generic kernel stores it
    elem_condense(p, nc, P, hinv, X, p, Rf);
    for (int r = 0; r < p; ++r)
      for (int c = 0; c < p; ++c) {
        double s = 0.0;
        for (int i = 0; i < p; ++i) s += X[i * p + r] * X[i * p + c];
        H[r * p + c] += s;
      }
    return 0;
  }
  // plain: Hsu = P' X (nc x p), Hss = P' A P, H -= Hsu' Hss^-1 Hsu (Cholesky of Hss)
  double Hsu[kElemMaxNc * kElemMaxP], Hs[kElemMaxNc * kElemMaxNc], L[kElemMaxNc * kElemMaxNc];
  for (int k = 0; k < nc; ++k)
    for (int c = 0; c < p; ++c) {
      double s = 0.0;
      for (int i = 0; i < p; ++i) s += P[i * nc + k] * X[i * p + c];
      Hsu[k * p + c] = s;
    }
  for (int k = 0; k < nc; ++k)
    for (int l = 0; l < nc; ++l) {
      double s = 0.0;
      for (int i = 0; i < p; ++i) s += P[i * nc + k] * hss[i] * P[i * nc + l];
      Hs[k * nc + l] = s;
    }
  for (int i = 0; i < nc; ++i)
    for (int j = 0; j <= i; ++j) {
      double s = Hs[i * nc + j];
      for (int k = 0; k < j; ++k) s -= L[i * nc + k] * L[j * nc + k];
      L[i * nc + j] = (i == j) ? sqrt(s) : s / L[j * nc + j];
    }
  for (int c = 0; c < p; ++c) {   // column c of Hss^-1 Hsu, then the update of H's column c
    double v[kElemMaxNc];
    for (int k = 0; k < nc; ++k) {
      double s = Hsu[k * p + c];
      for (int l = 0; l < k; ++l) s -= L[k * nc + l] * v[l];
      v[k] = s / L[k * nc + k];
    }
    for (int k = nc - 1; k >= 0; --k) {
      double s = v[k];
      for (int l = k + 1; l < nc; ++l) s -= L[l * nc + k] * v[l];
      v[k] = s / L[k * nc + k];
    }
    for (int r = 0; r < p; ++r) {
      double s = 0.0;
      for (int k = 0; k < nc; ++k) s += Hsu[k * p + r] * v[k];
      H[r * p + c] -= s;
    }
  }
  return 0;
}

// back-substitution of one element: dc = H_ss^-1 (gc - P' sum_a q_a (D_a du)) through the factor Rf of hostcheck_elem_schur
extern "C" int hostcheck_elem_backsubst(int p, int nc, int dim, const double *P, const double *D, const double *Z, const double *sc, double pexp,
                                        double mu, const double *Rf, const double *gc, const double *du, double *dc) {
  const int ny = dim + 1;
  for (int k = 0; k < nc; ++k) dc[k] = gc[k];
  for (int i = 0; i < p; ++i) {
    double F2[16];
    node_hess(dim, Z + i * ny, pexp, mu, true, F2);
    double s = 0.0;
    for (int a = 0; a < dim; ++a) {
      double Ddu = 0.0;
      for (int c = 0; c < p; ++c) Ddu += D[((size_t)a * p + c) * p + i] * du[c];
      s += sc[i] * F2[a * ny + dim] * Ddu;
    }
    for (int k = 0; k < nc; ++k) dc[k] -= P[i * nc + k] * s;
  }
  elem_hss_solve(nc, Rf, dc);
  return 0;
}
