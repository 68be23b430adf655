// elem_schur.cuh -- exact elimination of an element-local slack variable (e.g. a slack in :broken_P1), element by element.
//
// On element e the slack at its p nodes is P_e c_e (P_e: the p x nc block of R_fine, nc <= 4 coefficients).  With the node
// slack Hessians a_i (A = diag(a)) and the couplings q_{j,i} of the kept D rows j to the slack row (Q_j = diag(q_j)), the
// slack block is H_ss = P' A P (nc x nc) and the coupling H_us = sum_j D_j' Q_j P.  The Schur complement of the slack is
//     H_uu - H_us H_ss^-1 H_su = [node-local Schur complement of every node] + Y'Y,   Y = (I - Pi_W) A^{-1/2} sum_j Q_j D_j,
// Pi_W the orthogonal projector onto range(W), W = A^{1/2} P.  The node-local part is formed in closed form by the element
// kernels (node_barrier.cuh piece_eval, `schur`), as for a node-local slack; the correction Y'Y is positive semi-definite and
// subtracts no large terms: q / sqrt(a) stays bounded as the slack approaches the cone, where the plain subtraction
// H_uu - H_us H_ss^-1 H_su cancels ~t^2-sized terms down to O(t) and loses every digit along the cone's axis.
// H_ss = Pi R'R Pi' with R the triangular factor of the column-pivoted QR factorisation W Pi = Q R, kept per element (with the
// pivot order) for the right-hand side and the back-substitution.
// A node of zero weight (masked barrier, a_i = 0 and q_{j,i} = 0) contributes a zero row to W and to A^{-1/2} Q D (0/0 := 0).
// __host__ __device__ so that tests can check the arithmetic on the CPU (tests/hostcheck/elem_check.cpp).
#pragma once
#include <math.h>

#include "node_barrier.cuh"

namespace mgbx {

constexpr int kElemMaxP = 12;                    // nodes per element
constexpr int kElemMaxNc = 4;                    // slack coefficients per element
constexpr int kElemMaxCols = 2 * kElemMaxP;      // columns of Y: at most two kept variables couple to the slack
// per element: the packed upper triangle of R by rows, then the pivot order (nc column indices, stored as doubles)
MGBX_HD int elem_rsize(int nc) { return nc * (nc + 1) / 2 + nc; }
MGBX_HD int elem_ridx(int nc, int k, int j) { return k * nc - (k * (k - 1)) / 2 + (j - k); }

// hinv: 1 / a_i as the element kernels store it (hEEinv); the node has zero weight unless it is a positive finite number
MGBX_HD double elem_isqrt_a(double hinv) { return (hinv > 0.0 && hinv < INFINITY) ? sqrt(hinv) : 0.0; }

// In:  P (p x nc, row-major), hinv (p), X (p x m, row-major) = sum_j Q_j D_j restricted to the element (the coupling rows).
// Out: X = Y = (I - Pi_W) A^{-1/2} X, and R with its pivot order (elem_rsize(nc)).  Householder QR with the rows ordered by
// decreasing weight and column pivoting (Powell-Reid: accurate when the weights spread over many orders of magnitude).  A zero
// remaining column gets a zero pivot (its direction carries no slack Hessian) and is not projected out.
MGBX_HD void elem_condense(int p, int nc, const double *P, const double *hinv, double *X, int m, double *R) {
  int ord[kElemMaxP];
  double w[kElemMaxP];
  for (int i = 0; i < p; ++i) {
    ord[i] = i;
    const double is = elem_isqrt_a(hinv[i]);
    w[i] = is > 0.0 ? 1.0 / is : 0.0;   // sqrt(a_i)
  }
  for (int i = 1; i < p; ++i)           // insertion sort, stable: decreasing sqrt(a)
    for (int k = i; k > 0 && w[ord[k]] > w[ord[k - 1]]; --k) {
      const int t = ord[k];
      ord[k] = ord[k - 1];
      ord[k - 1] = t;
    }
  double W[kElemMaxP * kElemMaxNc], V[kElemMaxP * kElemMaxNc], beta[kElemMaxNc];
  for (int r = 0; r < p; ++r)
    for (int k = 0; k < nc; ++k) W[r * nc + k] = w[ord[r]] * P[ord[r] * nc + k];
  // X <- A^{-1/2} X (0 on zero-weight nodes), read below in the sorted row order
  for (int i = 0; i < p; ++i) {
    const double is = elem_isqrt_a(hinv[i]);
    for (int c = 0; c < m; ++c) X[i * m + c] *= is;
  }
  auto Z = [&](int r, int c) -> double & { return X[ord[r] * m + c]; };
  int piv[kElemMaxNc];
  for (int k = 0; k < nc; ++k) piv[k] = k;
  for (int k = 0; k < nc; ++k) {
    int jb = k;   // column pivoting: the remaining column of largest norm below row k
    double best = -1.0;
    for (int j = k; j < nc; ++j) {
      double cn = 0.0;
      for (int r = k; r < p; ++r) cn += W[r * nc + j] * W[r * nc + j];
      if (cn > best) {
        best = cn;
        jb = j;
      }
    }
    if (jb != k) {
      for (int r = 0; r < p; ++r) {
        const double t = W[r * nc + k];
        W[r * nc + k] = W[r * nc + jb];
        W[r * nc + jb] = t;
      }
      for (int i = 0; i < k; ++i) {   // the already computed rows of R follow the swap
        const double t = R[elem_ridx(nc, i, k)];
        R[elem_ridx(nc, i, k)] = R[elem_ridx(nc, i, jb)];
        R[elem_ridx(nc, i, jb)] = t;
      }
      const int t = piv[k];
      piv[k] = piv[jb];
      piv[jb] = t;
    }
    double nrm2 = 0.0, amax = 0.0;
    for (int r = k; r < p; ++r) amax = fmax(amax, fabs(W[r * nc + k]));
    for (int r = 0; r < p; ++r) V[r * nc + k] = 0.0;
    beta[k] = 0.0;
    if (amax == 0.0) {
      for (int j = k; j < nc; ++j) R[elem_ridx(nc, k, j)] = (j == k) ? 0.0 : W[k * nc + j];
      continue;
    }
    for (int r = k; r < p; ++r) {
      const double v = W[r * nc + k] / amax;
      nrm2 += v * v;
    }
    const double x0 = W[k * nc + k];
    const double alpha = -copysign(amax * sqrt(nrm2), x0);   // H x = alpha e_k
    for (int r = k; r < p; ++r) V[r * nc + k] = W[r * nc + k];
    V[k * nc + k] = x0 - alpha;
    double vv = 0.0;
    for (int r = k; r < p; ++r) vv += V[r * nc + k] * V[r * nc + k];
    beta[k] = 2.0 / vv;
    R[elem_ridx(nc, k, k)] = alpha;
    for (int j = k + 1; j < nc; ++j) {
      double d = 0.0;
      for (int r = k; r < p; ++r) d += V[r * nc + k] * W[r * nc + j];
      d *= beta[k];
      for (int r = k; r < p; ++r) W[r * nc + j] -= d * V[r * nc + k];
      R[elem_ridx(nc, k, j)] = W[k * nc + j];
    }
  }
  for (int k = 0; k < nc; ++k) R[elem_rsize(nc) - nc + k] = (double)piv[k];
  // Y = Q_full diag(0 on the pivoted rows, 1 elsewhere) Q_full' Z,  Q_full = H_0 ... H_{nc-1}
  for (int c = 0; c < m; ++c) {
    for (int k = 0; k < nc; ++k) {
      if (beta[k] == 0.0) continue;
      double d = 0.0;
      for (int r = k; r < p; ++r) d += V[r * nc + k] * Z(r, c);
      d *= beta[k];
      for (int r = k; r < p; ++r) Z(r, c) -= d * V[r * nc + k];
    }
    for (int k = 0; k < nc; ++k)
      if (beta[k] != 0.0) Z(k, c) = 0.0;
    for (int k = nc - 1; k >= 0; --k) {
      if (beta[k] == 0.0) continue;
      double d = 0.0;
      for (int r = k; r < p; ++r) d += V[r * nc + k] * Z(r, c);
      d *= beta[k];
      for (int r = k; r < p; ++r) Z(r, c) -= d * V[r * nc + k];
    }
  }
}

// b <- H_ss^-1 b = Pi (R'R)^-1 Pi' b through the packed factor; a zero pivot leaves that coefficient's step at 0
MGBX_HD void elem_hss_solve(int nc, const double *R, double *bb) {
  const double *piv = R + elem_rsize(nc) - nc;
  double b[kElemMaxNc];
  for (int k = 0; k < nc; ++k) b[k] = bb[(int)piv[k]];
  for (int k = 0; k < nc; ++k) {   // R' u = Pi' b
    double s = b[k];
    for (int i = 0; i < k; ++i) s -= R[elem_ridx(nc, i, k)] * b[i];
    const double d = R[elem_ridx(nc, k, k)];
    b[k] = d != 0.0 ? s / d : 0.0;
  }
  for (int k = nc - 1; k >= 0; --k) {   // R x = u
    double s = b[k];
    for (int j = k + 1; j < nc; ++j) s -= R[elem_ridx(nc, k, j)] * b[j];
    const double d = R[elem_ridx(nc, k, k)];
    b[k] = d != 0.0 ? s / d : 0.0;
  }
  for (int k = 0; k < nc; ++k) bb[(int)piv[k]] = b[k];
}

}  // namespace mgbx
