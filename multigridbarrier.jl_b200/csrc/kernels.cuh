// kernels.cuh -- sm_100a device kernels of barrier evaluation and Hessian assembly (compiled by evaluate.cu only).
//
// What each kernel replaces in the reference (paths under /root/reference):
//   k_node            apply_D + map_rows_gpu(F0/F1/F2) + the (1/n)·y + w.*c combination
//                     src/convex.jl:125,155-202,213-257; ext/MultiGridBarrierCUDAExt/map_rows_gpu.jl:20-63,
//                     block_ops.jl:118-133 (_block_matvec_kernel!)
//   k_blockgrad       sum_k D_k' y_k                    src/convex.jl:173-178; block_ops.jl:135-148
//   k_blockhess       sum_{j,k} D_j' diag(y_jk) D_k     src/convex.jl:185-200; block_ops.jl:58-75 (called nD^2 times there)
//   k_sell_gather     R'HR into the fixed pattern and the numeric Galerkin products A_c = T'(A T) (north-star item 3),
//                     src/BlockMatrices.jl:506-555, as fixed-order gathers over a sliced-ELL term list (coalesced
//                     index/weight streams, deterministic; the reference CUDA ext uses FP64 atomics, block_ops.jl:229-249)
//   k_spmv*           R*s, R'*g                          CUSPARSE in the reference (src/convex.jl:156,178)
//   (solver_kernels.cuh: k_l1diag = smoother diagonals and the Gershgorin bound of every level of the solve kernel)
//   (pcg2.cu: k_pcg2 = the multigrid-preconditioned CG solve, replacing cuDSS LDL' (ext/.../cudss_solver.jl:264-381))
//   (dense_kernels.cuh: DMMA GEMM of the spectral path; solver_kernels.cuh: its blocked Cholesky)
// All reductions are fixed-order (block tree + last-block pass): results are run-to-run deterministic.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>


#include "device_common.cuh"

namespace mgbx {

// ------------------------------------------------------------------------------------------------
// sparse matrix-vector products.  G threads cooperate on one row (G = 1, 4, 32).
//   y = alpha * A x + (y0 ? y0 : 0)
// ------------------------------------------------------------------------------------------------
template <int G>
__global__ void __launch_bounds__(256) k_spmv(DevCsr A, const double *__restrict__ x, const double *y0, double alpha,
                                               double *y) {
  const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t row = gtid / G;
  const int sub = (int)(gtid % G);
  if (row >= A.rows) return;   // G divides 32 and the block size, so whole groups exit together
  const int64_t b = A.ptr[row], e = A.ptr[row + 1];
  double acc = 0.0;
  for (int64_t k = b + sub; k < e; k += G) acc += A.val[k] * x[A.idx[k]];
  if (G > 1) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o, G);
  }
  if (sub == 0) y[row] = alpha * acc + (y0 ? y0[row] : 0.0);
}

// NDT >= nD bounds the per-thread arrays (y, F1, F2 = NDT^2 doubles) so that they stay in registers / L1
template <int MODE, int NDT>
__global__ void __launch_bounds__(kRedThreads) k_node(NodeParams P) {
  double red[4] = {0.0, 0.0, 0.0, -INFINITY};
  const int op[4] = {0, 0, 0, 1};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P.n; i += (int64_t)gridDim.x * blockDim.x) {
    double y[NDT];
    node_Dz(P, i, y);
    if (MODE == NODE_SLACK) {
      const double s = node_slack(P.cd, P.n, i, y);
      P.slack[i] = s;
      red[3] = fmax(red[3], s);
      continue;
    }
    const int nD = P.nD;
    const double bwi = P.bw ? P.bw[i] : 1.0;
    const bool active = !(P.bw && bwi == 0.0);
    double F1[NDT];
    if (MODE == NODE_F01) {
      double F0 = 0.0;
      if (active) F0 = node_eval(P.cd, P.n, i, y, 1, F1, nullptr);
      else
        for (int j = 0; j < nD; ++j) F1[j] = 0.0;
      const double wi = P.w[i];
      double lin = 0.0;
      const double sc = P.bw ? bwi : P.inv_n;
      for (int j = 0; j < nD; ++j) {
        const double c = P.t * P.f[i + (int64_t)j * P.n];
        lin += c * y[j];
        P.G[i + (int64_t)j * P.n] = (active ? sc * F1[j] : 0.0) + wi * c;
      }
      red[0] += active ? (P.bw ? bwi * F0 : F0) : 0.0;
      red[1] += wi * lin;
      if (!isfinite(F0)) red[2] += 1.0;
    } else {   // NODE_F2
      double F2[NDT * NDT];
      const double sc = P.bw ? bwi : P.inv_n;
      if (active) {
        node_eval(P.cd, P.n, i, y, 2, F1, F2, nE_mask_guard(P));
        for (int k = 0; k < nD * nD; ++k) F2[k] *= sc;
      } else {
        for (int k = 0; k < nD * nD; ++k) F2[k] = 0.0;
      }
      const int nK = P.nK, nE = P.nE;
      if (nE == 0) {
        int q = 0;
        for (int a = 0; a < nK; ++a)
          for (int b = a; b < nK; ++b, ++q) P.Hn[i + (int64_t)q * P.n] = F2[P.Krow[a] * nD + P.Krow[b]];
      } else {
        double hEE[16], hKE[NDT * 4];
        for (int k = 0; k < nE * nE; ++k) hEE[k] = 0.0;
        for (int k = 0; k < nK * nE; ++k) hKE[k] = 0.0;
        for (int j = 0; j < nD; ++j) {
          const int ej = P.Erow[j];
          if (ej < 0) continue;
          for (int k = 0; k < nD; ++k) {
            const int ek = P.Erow[k];
            if (ek >= 0) hEE[ej * nE + ek] += F2[j * nD + k];
          }
          for (int a = 0; a < nK; ++a) hKE[a * nE + ej] += F2[P.Krow[a] * nD + j];
        }
        spd_inverse(hEE, nE);
        {
          int q = 0;
          for (int a = 0; a < nE; ++a)
            for (int b = a; b < nE; ++b, ++q) P.hEEinv[i + (int64_t)q * P.n] = hEE[a * nE + b];
        }
        for (int k = 0; k < nK * nE; ++k) P.hKE[i + (int64_t)k * P.n] = hKE[k];
        // W = hEEinv * hEK  (nE x nK);  Hn = hKK - hKE W
        int q = 0;
        for (int a = 0; a < nK; ++a)
          for (int b = a; b < nK; ++b, ++q) {
            double s = F2[P.Krow[a] * nD + P.Krow[b]];
            for (int ev = 0; ev < nE; ++ev) {
              if ((P.schur_elim >> ev) & 1u) continue;   // already condensed analytically inside node_eval
              double wv = 0.0;
              for (int ew = 0; ew < nE; ++ew) wv += hEE[ev * nE + ew] * hKE[b * nE + ew];
              s -= hKE[a * nE + ev] * wv;
            }
            P.Hn[i + (int64_t)q * P.n] = s;
          }
      }
    }
  }
  if (MODE != NODE_F2) grid_reduce<4>(red, op, P.partials, P.ticket, P.red_out);
}

// gb[v*n + e*p + c] = sum_{j in rows(v), j in Krow} sum_q D_j[q][c] * G[j*n + e*p + q]
// one thread per (variable slot, broken node)
__global__ void __launch_bounds__(256) k_blockgrad(ElemParams P, const double *__restrict__ G, double *gb, int nu) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= (int64_t)nu * P.n) return;
  const int v = (int)(tid / P.n);
  const int64_t i = tid - (int64_t)v * P.n;
  const int64_t e = i / P.p;
  const int c = (int)(i - e * P.p);
  double acc = 0.0;
  for (int jj = 0; jj < P.nK; ++jj) {
    const int j = P.Krow[jj];
    if (P.D_var[j] != v) continue;
    const int o = P.D_op[j];
    const double *g = G + (int64_t)j * P.n;
    if (o < 0) acc += g[i];
    else {
      const double *blk = P.ops[o] + e * (int64_t)(P.p * P.p) + (int64_t)c * P.p;
      const double *ge = g + e * P.p;
      for (int q = 0; q < P.p; ++q) acc += blk[q] * ge[q];
    }
  }
  gb[tid] = acc;
}

__global__ void __launch_bounds__(256) k_blockhess(ElemParams P, PairList PL, const double *__restrict__ Hn, double *Hblk) {
  const int pp = P.p * P.p;
  const int64_t total = (int64_t)PL.npairs * P.N * pp;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid >= total) return;
  const int c = (int)(tid % P.p);
  const int r = (int)((tid / P.p) % P.p);
  const int64_t e = (tid / pp) % P.N;
  const int pr = (int)(tid / ((int64_t)pp * P.N));
  const int va = PL.va[pr], vb = PL.vb[pr];
  const int nK = P.nK;
  const int64_t base = e * P.p;
  double acc = 0.0;
  for (int ja = 0; ja < nK; ++ja) {
    const int j = P.Krow[ja];
    if (P.D_var[j] != va) continue;
    const int oj = P.D_op[j];
    for (int kb = 0; kb < nK; ++kb) {
      const int k = P.Krow[kb];
      if (P.D_var[k] != vb) continue;
      const int ok = P.D_op[k];
      const int a = ja < kb ? ja : kb, b = ja < kb ? kb : ja;
      const double *h = Hn + (int64_t)(a * nK - (a * (a - 1)) / 2 + (b - a)) * P.n + base;
      if (oj < 0 && ok < 0) {
        if (r == c) acc += h[r];
      } else if (oj < 0) {
        acc += h[r] * P.ops[ok][e * (int64_t)pp + (int64_t)c * P.p + r];
      } else if (ok < 0) {
        acc += P.ops[oj][e * (int64_t)pp + (int64_t)r * P.p + c] * h[c];
      } else {
        const double *dj = P.ops[oj] + e * (int64_t)pp + (int64_t)r * P.p;
        const double *dk = P.ops[ok] + e * (int64_t)pp + (int64_t)c * P.p;
        double s = 0.0;
        for (int q = 0; q < P.p; ++q) s += dj[q] * h[q] * dk[q];
        acc += s;
      }
    }
  }
  Hblk[tid] = acc;
}

// ------------------------------------------------------------------------------------------------
// vector kernels (all scalars stay on the device)
// ------------------------------------------------------------------------------------------------
// out = {a.b, a.a, #non-finite entries of a}
__global__ void __launch_bounds__(kRedThreads) k_dot2(int64_t m, const double *__restrict__ a, const double *__restrict__ b,
                                                       double *partials, unsigned int *ticket, double *out) {
  double red[3] = {0.0, 0.0, 0.0};
  const int op[3] = {0, 0, 0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double x = a[i];
    red[0] += x * (b ? b[i] : 0.0);
    red[1] += x * x;
    if (!isfinite(x)) red[2] += 1.0;
  }
  grid_reduce<3>(red, op, partials, ticket, out);
}

// xn = x - s*d;  out = {|xn - x|^2} (exactly as evaluated in floating point: stall detection, src/newton.jl:141)
__global__ void __launch_bounds__(kRedThreads) k_trial(int64_t m, const double *__restrict__ x, const double *__restrict__ d, double s,
                                                        double *xn, double *partials, unsigned int *ticket, double *out) {
  double red[1] = {0.0};
  const int op[1] = {0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double xi = x[i];
    const double v = xi - s * d[i];
    xn[i] = v;
    const double df = v - xi;
    red[0] += df * df;
  }
  grid_reduce<1>(red, op, partials, ticket, out);
}

__global__ void k_axpby(int64_t m, double a, const double *__restrict__ x, double b, const double *__restrict__ y, double *out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) out[i] = a * x[i] + (y ? b * y[i] : 0.0);
}

// per-variable max and max|.| of the state: out[2k] = max, out[2k+1] = absmax  (one launch per variable)
__global__ void __launch_bounds__(kRedThreads) k_maxabs(int64_t m, const double *__restrict__ a, double *partials, unsigned int *ticket,
                                                         double *out) {
  double red[3] = {-INFINITY, -INFINITY, 0.0};
  const int op[3] = {1, 1, 0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double v = a[i];
    red[0] = fmax(red[0], v);
    red[1] = fmax(red[1], fabs(v));
    if (!isfinite(v)) red[2] += 1.0;
  }
  grid_reduce<3>(red, op, partials, ticket, out);
}

// sl[i] = 2*max(slack[i], 1)   (src/mgb.jl:437-440)
__global__ void k_phase1_slack(int64_t n, const double *slack, double *out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = 2.0 * fmax(slack[i], 1.0);
}

// out = {a.b, a.a, #non-finite entries of a} over the LOCAL segments, then the same three over the SHARED ones
__global__ void __launch_bounds__(kRedThreads) k_dot2_seg(SegList S, int64_t m, const double *__restrict__ a, const double *__restrict__ b,
                                                           double *partials, unsigned int *ticket, double *out) {
  double red[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  const int op[6] = {0, 0, 0, 0, 0, 0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double x = a[i];
    const int o = seg_is_local(S, i) ? 0 : 3;
    red[o] += x * (b ? b[i] : 0.0);
    red[o + 1] += x * x;
    if (!isfinite(x)) red[o + 2] += 1.0;
  }
  grid_reduce<6>(red, op, partials, ticket, out);
}

// xn = x - s*d;  out = {|xn - x|^2 over the SHARED segments, the same over the LOCAL ones}
__global__ void __launch_bounds__(kRedThreads) k_trial_seg(SegList S, int64_t m, const double *__restrict__ x, const double *__restrict__ d,
                                                            double s, double *xn, double *partials, unsigned int *ticket, double *out) {
  double red[2] = {0.0, 0.0};
  const int op[2] = {0, 0};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const double xi = x[i];
    const double v = xi - s * d[i];
    xn[i] = v;
    const double df = v - xi;
    red[seg_is_local(S, i) ? 1 : 0] += df * df;
  }
  grid_reduce<2>(red, op, partials, ticket, out);
}

template <int MODE, int NDT>
__global__ void __launch_bounds__(256) k_elem(ElemFused Q) {
  extern __shared__ double esm[];
  const NodeParams &P = Q.np;
  const int p = P.p, pp = p * p, p1 = Q.p1, ES = Q.ES, epb = Q.epb;
  const int TM = epb * p;                       // node slots per tile
  double *ops_s = esm;                          // [op][el][c][r] padded
  double *zs = ops_s + (size_t)Q.nops * epb * ES;   // [var][slot]
  double *ex = zs + (size_t)P.nu * TM;          // [row][slot]
  const int tid = threadIdx.x;
  double red[4] = {0.0, 0.0, 0.0, -INFINITY};
  const int op4[4] = {0, 0, 0, 1};
  const int64_t ntiles = (Q.N + epb - 1) / epb;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t e0 = tile * epb;
    const int ne = (int)min((int64_t)epb, Q.N - e0);
    const int T = ne * p;
    const int64_t node0 = e0 * p;
    __syncthreads();   // previous tile fully consumed
    for (int o = 0; o < Q.nops; ++o) {
      const double *src = P.ops[o] + e0 * (int64_t)pp;
      double *dst = ops_s + (size_t)o * epb * ES;
      for (int t = tid; t < ne * pp; t += blockDim.x) {
        const int el = t / pp, rem = t - el * pp;
        const int c = rem / p, r = rem - c * p;
        dst[el * ES + c * p1 + r] = src[t];
      }
    }
    for (int v = 0; v < P.nu; ++v)
      for (int t = tid; t < T; t += blockDim.x) zs[v * TM + t] = P.zf[(int64_t)v * P.n + node0 + t];
    __syncthreads();
    const int el = tid / p, q = tid - el * p;
    const bool on = tid < T;
    const int64_t i = node0 + tid;
    if (on) {
      double y[NDT];
      for (int j = 0; j < P.nD; ++j) {
        const int v = P.D_var[j], o = P.D_op[j];
        if (o < 0) y[j] = zs[v * TM + tid];
        else {
          const double *blk = ops_s + (size_t)o * epb * ES + el * ES + q;
          const double *ze = zs + v * TM + el * p;
          double acc = 0.0;
          for (int c = 0; c < p; ++c) acc += blk[c * p1] * ze[c];
          y[j] = acc;
        }
      }
      const int nD = P.nD;
      const double bwi = P.bw ? P.bw[i] : 1.0;
      const bool active = !(P.bw && bwi == 0.0);
      const double sc = P.bw ? bwi : P.inv_n;
      double F1[NDT];
      if (MODE == NODE_F01) {
        double F0 = 0.0;
        if (active) F0 = node_eval(P.cd, P.n, i, y, 1, F1, nullptr);
        else
          for (int j = 0; j < nD; ++j) F1[j] = 0.0;
        const double wi = P.w[i];
        double lin = 0.0;
        for (int j = 0; j < nD; ++j) {
          const double c = P.t * P.f[i + (int64_t)j * P.n];
          lin += c * y[j];
          ex[j * TM + tid] = (active ? sc * F1[j] : 0.0) + wi * c;
        }
        red[0] += active ? (P.bw ? bwi * F0 : F0) : 0.0;
        red[1] += wi * lin;
        if (!isfinite(F0)) red[2] += 1.0;
      } else {
        double F2[NDT * NDT];
        if (active) {
          node_eval(P.cd, P.n, i, y, 2, F1, F2, nE_mask_guard(P));
          for (int k = 0; k < nD * nD; ++k) F2[k] *= sc;
        } else {
          for (int k = 0; k < nD * nD; ++k) F2[k] = 0.0;
        }
        const int nK = P.nK, nE = P.nE;
        if (nE == 0) {
          int qq = 0;
          for (int a = 0; a < nK; ++a)
            for (int b = a; b < nK; ++b, ++qq) ex[qq * TM + tid] = F2[P.Krow[a] * nD + P.Krow[b]];
        } else {
          double hEE[16], hKE[NDT * 4];
          for (int k = 0; k < nE * nE; ++k) hEE[k] = 0.0;
          for (int k = 0; k < nK * nE; ++k) hKE[k] = 0.0;
          for (int j = 0; j < nD; ++j) {
            const int ej = P.Erow[j];
            if (ej < 0) continue;
            for (int k = 0; k < nD; ++k) {
              const int ek = P.Erow[k];
              if (ek >= 0) hEE[ej * nE + ek] += F2[j * nD + k];
            }
            for (int a = 0; a < nK; ++a) hKE[a * nE + ej] += F2[P.Krow[a] * nD + j];
          }
          spd_inverse(hEE, nE);
          {
            int qq = 0;
            for (int a = 0; a < nE; ++a)
              for (int b = a; b < nE; ++b, ++qq) P.hEEinv[i + (int64_t)qq * P.n] = hEE[a * nE + b];
          }
          for (int k = 0; k < nK * nE; ++k) P.hKE[i + (int64_t)k * P.n] = hKE[k];
          int qq = 0;
          for (int a = 0; a < nK; ++a)
            for (int b = a; b < nK; ++b, ++qq) {
              double s = F2[P.Krow[a] * nD + P.Krow[b]];
              for (int ev = 0; ev < nE; ++ev) {
                if ((P.schur_elim >> ev) & 1u) continue;   // already condensed analytically inside node_eval
                double wv = 0.0;
                for (int ew = 0; ew < nE; ++ew) wv += hEE[ev * nE + ew] * hKE[b * nE + ew];
                s -= hKE[a * nE + ev] * wv;
              }
              ex[qq * TM + tid] = s;
            }
        }
      }
    }
    __syncthreads();
    if (MODE == NODE_F01) {
      // gb[v][node0 + (el, c)] = sum_{j in rows(v)} sum_q D_j[q][c] G_j[q]
      if (on) {
        const int c = q;
        for (int v = 0; v < P.nu; ++v) {
          double acc = 0.0;
          for (int j = 0; j < P.nD; ++j) {
            if (P.D_var[j] != v) continue;
            const int o = P.D_op[j];
            const double *g = ex + j * TM + el * p;
            if (o < 0) acc += g[c];
            else {
              const double *blk = ops_s + (size_t)o * epb * ES + el * ES + c * p1;
              for (int k = 0; k < p; ++k) acc += blk[k] * g[k];
            }
          }
          Q.gb[(int64_t)v * P.n + i] = acc;
        }
      }
    } else {
      // Hblk[((pair*N + e)*p + r)*p + c] = sum_{ja in rows(va), kb in rows(vb)} sum_q D_ja[q][r] h[q] D_kb[q][c]
      const int nK = P.nK;
      const int per = ne * pp;
      for (int pr = 0; pr < Q.pl.npairs; ++pr) {
        const int va = Q.pl.va[pr], vb = Q.pl.vb[pr];
        double *out = Q.Hblk + ((int64_t)pr * Q.N + e0) * pp;
        for (int t = tid; t < per; t += blockDim.x) {
          const int e2 = t / pp, rem = t - e2 * pp;
          const int r = rem / p, c = rem - r * p;
          double acc = 0.0;
          for (int ja = 0; ja < nK; ++ja) {
            const int j = P.Krow[ja];
            if (P.D_var[j] != va) continue;
            const int oj = P.D_op[j];
            for (int kb = 0; kb < nK; ++kb) {
              const int k = P.Krow[kb];
              if (P.D_var[k] != vb) continue;
              const int ok = P.D_op[k];
              const int a = ja < kb ? ja : kb, b = ja < kb ? kb : ja;
              const double *h = ex + (a * nK - (a * (a - 1)) / 2 + (b - a)) * TM + e2 * p;
              if (oj < 0 && ok < 0) {
                if (r == c) acc += h[r];
              } else if (oj < 0) {
                acc += h[r] * ops_s[(size_t)ok * epb * ES + e2 * ES + c * p1 + r];
              } else if (ok < 0) {
                acc += ops_s[(size_t)oj * epb * ES + e2 * ES + r * p1 + c] * h[c];
              } else {
                const double *dj = ops_s + (size_t)oj * epb * ES + e2 * ES + r * p1;
                const double *dk = ops_s + (size_t)ok * epb * ES + e2 * ES + c * p1;
                double s = 0.0;
                for (int k2 = 0; k2 < p; ++k2) s += dj[k2] * h[k2] * dk[k2];
                acc += s;
              }
            }
          }
          out[t] = acc;
        }
      }
    }
  }
  if (MODE == NODE_F01) grid_reduce<4>(red, op4, P.partials, P.ticket, P.red_out);
}

// Tiles are software-pipelined: while tile k is evaluated, the operator blocks and node inputs of tile k+1 stream into the
// other shared-memory buffer with cp.async (LDGSTS), so the evaluation never waits on HBM latency after the first tile.
// COND: the slack is condensed node-locally (fine-level systems); !COND: nothing is eliminated and the four block pairs
// (u,u), (u,s), (s,u), (s,s) are written (the coarse-level systems of the mgb_step recovery path).
template <int MODE, int DIM, bool COND>
__global__ void __launch_bounds__(256, 3) k_elem_plap(PlapParams P) {
  extern __shared__ __align__(16) double esm[];
  constexpr int NH = (DIM * (DIM + 1)) / 2;
  constexpr int NEX = NH > DIM ? NH : DIM;
  constexpr int NF = DIM + 2;
  const int p = P.p, pp = p * p, p1 = P.p1, ES = P.ES, epb = P.epb;
  const int TM = epb * p;
  const size_t bufsz = (size_t)DIM * epb * ES + (size_t)(4 + NF) * TM;
  double *ex = esm + 2 * bufsz;                    // [row][slot]: F01 DIM rows, F2 NH rows
  (void)NEX;
  const int tid = threadIdx.x;
  double red[4] = {0.0, 0.0, 0.0, -INFINITY};
  const int op4[4] = {0, 0, 0, 1};
  const int64_t ntiles = (P.N + epb - 1) / epb;
  const double al = 2.0 / P.pexp;
  // completion barriers of the two input buffers (bulk staging); a tile arms its buffer's barrier with the bytes it will receive
  __shared__ __align__(8) unsigned long long mbar[2];
  unsigned int mphase = 0u;   // bit b: parity of buffer b's next completion
  if (P.bulk) {
    if (tid == 0) {
      mbar_init(&mbar[0], 1);
      mbar_init(&mbar[1], 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
  }
  // buffer layout: ops [a][el][c][r] padded | us | ss | ws | bws | fs[NF]
  auto issue = [&](int64_t tile, int b) {
    double *buf = esm + (size_t)b * bufsz;
    const int64_t e0 = tile * epb;
    const int ne = (int)min((int64_t)epb, P.N - e0);
    const int T = ne * p;
    const int64_t node0 = e0 * p;
    if (P.bulk) {
      // whole slabs move with one instruction each (UBLKCP); a ragged last tile (odd sizes break the 16-byte rule) falls through
      // to the per-double path below and arms the barrier with zero bytes
      const bool regular = ((ne & 1) == 0 || (p & 1) == 0) && ((T & 1) == 0);
      if (regular) {
        double *nd = buf + (size_t)DIM * epb * ES;
        const int narr = 3 + (P.bw ? 1 : 0) + NF;
        const unsigned int opbytes = (unsigned int)(ne * pp * 8), ndbytes = (unsigned int)(T * 8);
        if (tid == 0) {
          fence_proxy_async_smem();
          mbar_expect_tx(&mbar[b], DIM * opbytes + narr * ndbytes);
        }
        __syncwarp();
        if (P.bulk == 1) {
          if (tid < DIM) bulk_g2s(buf + (size_t)tid * epb * ES, P.ops[tid] + e0 * (int64_t)pp, opbytes, &mbar[b]);
        } else {
          for (int t = tid; t < DIM * ne * p; t += 256) {   // one block column (p doubles) per copy into the padded layout
            const int a = t / (ne * p), rem = t - a * ne * p;
            const int el = (int)fdiv((unsigned int)rem, P.dp), c = rem - el * p;
            bulk_g2s(buf + (size_t)a * epb * ES + el * ES + c * p1, P.ops[a] + (e0 + el) * (int64_t)pp + c * p, (unsigned int)(p * 8), &mbar[b]);
          }
        }
        if (tid >= 32 && tid < 32 + narr) {
          const int k = tid - 32;
          const double *src;
          double *dst;
          if (k == 0) { src = P.zu; dst = nd; }
          else if (k == 1) { src = P.zs; dst = nd + TM; }
          else if (k == 2) { src = P.w; dst = nd + 2 * TM; }
          else if (P.bw && k == 3) { src = P.bw; dst = nd + 3 * TM; }
          else {
            const int j = k - 3 - (P.bw ? 1 : 0);
            src = P.f + (int64_t)j * P.n;
            dst = nd + (4 + j) * TM;
          }
          bulk_g2s(dst, src + node0, ndbytes, &mbar[b]);
        }
        cp_async_commit();   // (empty group: keeps the wait_group bookkeeping of the ragged path uniform)
        return;
      }
      if (tid == 0) mbar_expect_tx(&mbar[b], 0);
    }
#pragma unroll
    for (int a = 0; a < DIM; ++a) {
      const double *src = P.ops[a] + e0 * (int64_t)pp;
      double *dst = buf + (size_t)a * epb * ES;
      for (int t = tid; t < ne * pp; t += 256) {
        const int el = (int)fdiv((unsigned int)t, P.dpp), rem = t - el * pp;
        const int c = (int)fdiv((unsigned int)rem, P.dp), r = rem - c * p;
        cp_async8(dst + el * ES + c * p1 + r, src + t);
      }
    }
    double *nd = buf + (size_t)DIM * epb * ES;
    if (tid < T) {
      const int64_t i = node0 + tid;
      cp_async8(nd + tid, P.zu + i);
      cp_async8(nd + TM + tid, P.zs + i);
      cp_async8(nd + 2 * TM + tid, P.w + i);
      if (P.bw) cp_async8(nd + 3 * TM + tid, P.bw + i);
#pragma unroll
      for (int j = 0; j < NF; ++j) cp_async8(nd + (4 + j) * TM + tid, P.f + i + (int64_t)j * P.n);
    }
    cp_async_commit();
  };
  int b = 0;
  if ((int64_t)blockIdx.x < ntiles) issue(blockIdx.x, 0);
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t next = tile + gridDim.x;
    if (next < ntiles) {
      issue(next, b ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    if (P.bulk) {
      mbar_wait(&mbar[b], (mphase >> b) & 1u);
      mphase ^= 1u << b;
    }
    __syncthreads();
    const double *ops_s = esm + (size_t)b * bufsz;
    const double *us = ops_s + (size_t)DIM * epb * ES;
    const double *ss = us + TM, *ws = us + 2 * TM, *bws = us + 3 * TM, *fs = us + 4 * TM;
    const int64_t e0 = tile * epb;
    const int ne = (int)min((int64_t)epb, P.N - e0);
    const int T = ne * p;
    const int64_t node0 = e0 * p;
    const int el = (int)fdiv((unsigned int)tid, P.dp), qn = tid - el * p;
    const bool on = tid < T;
    const int64_t i = node0 + tid;
    double G0 = 0.0, Gs = 0.0;
    if (on) {
      double q[DIM];
      const double *ue = us + el * p;
#pragma unroll
      for (int a = 0; a < DIM; ++a) {
        const double *blk = ops_s + (size_t)a * epb * ES + el * ES + qn;
        double acc = 0.0;
        for (int c = 0; c < p; ++c) acc += blk[c * p1] * ue[c];
        q[a] = acc;
      }
      const double uu = ue[qn];
      const double s = ss[tid];
      const double bwi = P.bw ? bws[tid] : 1.0;
      const bool active = !(P.bw && bwi == 0.0);
      const double sc = P.bw ? bwi : P.inv_n;
      const double wi = ws[tid];
      double qsq = 0.0;
#pragma unroll
      for (int a = 0; a < DIM; ++a) qsq += q[a] * q[a];
      const double ls = Log(s);
      const double sa = exp(al * ls);
      const double r = sa - qsq;
      const bool in = s > 0.0;
      const double inv_r = 1.0 / r;
      const double sam1 = in ? sa / s : safe_pow(s, al - 1.0);
      if (MODE == NODE_F01) {
        const double F0 = active ? (-Log(r) - P.mu * ls) : 0.0;
        const double c0 = P.t * fs[tid];
        const double cs = P.t * fs[(DIM + 1) * TM + tid];
        double lin = c0 * uu + cs * s;
        G0 = wi * c0;
        const double gs = -al * sam1 * inv_r - P.mu / s;
        Gs = (active ? sc * gs : 0.0) + wi * cs;
#pragma unroll
        for (int a = 0; a < DIM; ++a) {
          const double ca = P.t * fs[(a + 1) * TM + tid];
          lin += ca * q[a];
          ex[a * TM + tid] = (active ? sc * 2.0 * inv_r * q[a] : 0.0) + wi * ca;
        }
        red[0] += active ? (P.bw ? bwi * F0 : F0) : 0.0;
        red[1] += wi * lin;
        if (!isfinite(F0)) red[2] += 1.0;
      } else {
        if (active) {
          const double inv_r2 = inv_r * inv_r;
          const double coef = -2.0 * al * sam1 * inv_r2;
          const double sam2 = in ? sam1 / s : safe_pow(s, al - 2.0);
          const double s2am2 = in ? sam1 * sam1 : safe_pow(s, 2.0 * al - 2.0);
          // H_ss = A + B with A = (al s^(al-1) / r)^2 (the square of the coupling) and B the rest.  The node-local Schur
          // complement of the slack is  H_qq - H_qs H_sq / H_ss = (2/r) I + (4/r^2) (B / (A + B)) q q':  formed this way, not by
          // subtracting two terms of size 4 q q'/r^2 ~ t^2 whose difference is O(t) across q and O(1) along q -- at t ~ 1e8 the
          // subtraction leaves NO correct digit along q (absolute error eps t^2 ~ 1) and the reduced matrix turns indefinite.
          const double hA = al * al * s2am2 * inv_r2, hB = -al * (al - 1.0) * sam2 * inv_r + P.mu / (s * s);
          const double hss = sc * (hA + hB);
          const double ihs = COND ? 1.0 / hss : 0.0;
          const double schur = hB / (hA + hB);
          double hqs[DIM];
#pragma unroll
          for (int a = 0; a < DIM; ++a) hqs[a] = sc * coef * q[a];
          if (COND) {
            P.hEEinv[i] = ihs;
            P.hKE[i] = 0.0;
#pragma unroll
            for (int a = 0; a < DIM; ++a) P.hKE[i + (int64_t)(a + 1) * P.n] = hqs[a];
          } else {
#pragma unroll
            for (int a = 0; a < DIM; ++a) ex[(NH + a) * TM + tid] = hqs[a];
            ex[(NH + DIM) * TM + tid] = hss;
          }
          int k = 0;
#pragma unroll
          for (int a = 0; a < DIM; ++a)
#pragma unroll
            for (int bb = a; bb < DIM; ++bb, ++k) {
              const double qq4 = 4.0 * q[a] * q[bb] * inv_r2, dg = (a == bb ? 2.0 * inv_r : 0.0);
              ex[k * TM + tid] = COND ? sc * (qq4 * schur + dg) : sc * (qq4 + dg);
            }
        } else {
          if (COND) {
            P.hEEinv[i] = 0.0;
#pragma unroll
            for (int a = 0; a <= DIM; ++a) P.hKE[i + (int64_t)a * P.n] = 0.0;
          }
#pragma unroll
          for (int k = 0; k < (COND ? NH : NH + DIM + 1); ++k) ex[k * TM + tid] = 0.0;
        }
      }
    }
    __syncthreads();
    if (MODE == NODE_F01) {
      if (on) {
        double acc = G0;
#pragma unroll
        for (int a = 0; a < DIM; ++a) {
          const double *blk = ops_s + (size_t)a * epb * ES + el * ES + qn * p1;
          const double *g = ex + a * TM + el * p;
          for (int k = 0; k < p; ++k) acc += blk[k] * g[k];
        }
        P.gbu[i] = acc;
        P.gbs[i] = Gs;
      }
    } else {
      double *out = P.Hblk + e0 * (int64_t)pp;
      for (int t = tid; t < ne * pp; t += 256) {
        const int e2 = (int)fdiv((unsigned int)t, P.dpp), rem = t - e2 * pp;
        const int r = (int)fdiv((unsigned int)rem, P.dp), c = rem - r * p;
        const double *h = ex + e2 * p;
        const double *base = ops_s + e2 * ES;
        double acc = 0.0;
        for (int k = 0; k < p; ++k) {
          double dr[DIM], dc[DIM];
#pragma unroll
          for (int a = 0; a < DIM; ++a) {
            dr[a] = base[(size_t)a * epb * ES + r * p1 + k];
            dc[a] = base[(size_t)a * epb * ES + c * p1 + k];
          }
          int kk = 0;
#pragma unroll
          for (int a = 0; a < DIM; ++a)
#pragma unroll
            for (int bb = a; bb < DIM; ++bb, ++kk) {
              const double hv = h[kk * TM + k];
              acc += (a == bb) ? dr[a] * hv * dc[a] : hv * (dr[a] * dc[bb] + dr[bb] * dc[a]);
            }
        }
        out[t] = acc;
        if (!COND) {
          // (u,s): sum_a D_a[c][r] h_as[c];  (s,u): its transpose;  (s,s): diag(h_ss)
          double us_ = 0.0, su_ = 0.0;
#pragma unroll
          for (int a = 0; a < DIM; ++a) {
            us_ += base[(size_t)a * epb * ES + r * p1 + c] * h[(NH + a) * TM + c];
            su_ += h[(NH + a) * TM + r] * base[(size_t)a * epb * ES + c * p1 + r];
          }
          const int64_t pstride = P.N * (int64_t)pp;
          out[pstride + t] = us_;
          out[2 * pstride + t] = su_;
          out[3 * pstride + t] = (r == c) ? h[(NH + DIM) * TM + r] : 0.0;
        }
      }
    }
    __syncthreads();   // the exchange rows and (two tiles later) this input buffer are reused
    b ^= 1;
  }
  if (MODE == NODE_F01) grid_reduce<4>(red, op4, P.partials, P.ticket, P.red_out);
}

// Element-local slack (elem_schur.cuh), after the element kernel has written the node-local Schur complements into Hblk and
// 1/a, q into hEEinv, hKE: adds Y'Y to the element blocks of the kept pairs and stores the factor R of W.  One thread per
// element; the kept variables that own D rows are the distinct first members of the pairs (at most two).
__global__ void __launch_bounds__(128) k_elem_local_schur(ElemParams E, PairList PL, ElemLocal EL, const double *__restrict__ hEEinv,
                                                          const double *__restrict__ hKE, double *Hblk) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E.N) return;
  const int p = E.p, pp = p * p, nc = EL.nc;
  int vars[2], nv = 0;
  for (int pr = 0; pr < PL.npairs; ++pr)
    if (nv == 0 || (PL.va[pr] != vars[0] && nv < 2)) vars[nv++] = PL.va[pr];
  const int m = nv * p;
  double X[kElemMaxP * kElemMaxCols], hinv[kElemMaxP], Pe[kElemMaxP * kElemMaxNc];
  const int64_t node0 = e * p;
  for (int i = 0; i < p; ++i) {
    hinv[i] = hEEinv[node0 + i];
    for (int k = 0; k < nc; ++k) Pe[i * nc + k] = EL.P[(node0 + i) * nc + k];
    for (int c = 0; c < m; ++c) X[i * m + c] = 0.0;
  }
  for (int a = 0; a < E.nK; ++a) {   // X[i][(v, c)] = sum_{rows j of v} q_{j,i} D_j[i][c]
    const int j = E.Krow[a], o = E.D_op[j];
    const int col0 = (E.D_var[j] == vars[0]) ? 0 : p;
    for (int i = 0; i < p; ++i) {
      const double q = hKE[node0 + i + (int64_t)a * E.n];
      if (q == 0.0) continue;
      if (o < 0) X[i * m + col0 + i] += q;
      else {
        const double *blk = E.ops[o] + e * (int64_t)pp + i;
        for (int c = 0; c < p; ++c) X[i * m + col0 + c] += q * blk[(int64_t)c * p];
      }
    }
  }
  elem_condense(p, nc, Pe, hinv, X, m, EL.R + e * elem_rsize(nc));
  for (int pr = 0; pr < PL.npairs; ++pr) {
    const int ca = (PL.va[pr] == vars[0]) ? 0 : p, cb = (PL.vb[pr] == vars[0]) ? 0 : p;
    double *out = Hblk + ((int64_t)pr * E.N + e) * pp;
    for (int r = 0; r < p; ++r)
      for (int c = 0; c < p; ++c) {
        double s = 0.0;
        for (int i = 0; i < p; ++i) s += X[i * m + ca + r] * X[i * m + cb + c];
        out[r * p + c] += s;
      }
  }
}

__global__ void __launch_bounds__(256) k_sell_gather(SellPlan P, const double *__restrict__ in, double *__restrict__ out) {
  const int64_t nz = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (nz >= P.nout) return;
  const int64_t off = P.sptr[nz >> 5] + (nz & 31);
  const int c = P.cnt[nz];
  double acc = 0.0;
  if (P.w) {
    for (int k = 0; k < c; ++k) acc += P.w[off + 32 * (int64_t)k] * in[P.src[off + 32 * (int64_t)k]];
  } else {
    for (int k = 0; k < c; ++k) acc += in[P.src[off + 32 * (int64_t)k]];
  }
  out[nz] = acc;
}

}  // namespace mgbx
