// newton.cu -- damped Newton at one level, the level recursion of mgb_step, and the matched barrier parameter.
//   newton.jl:227-287          newton          -> Engine::newton
//   newton.jl:35-50,139-154    backtracking    -> Engine::newton (inlined trial loop)
//   newton.jl:187,222-225      stopping rules  -> stop_test
//   mgb.jl:10-82               divide_and_conquer / mgb_step -> Engine::step
//   mgb.jl:307-330             _matched_t      -> Engine::matched_t
// Host logic only: every launch goes through an Engine method of evaluate.cu or linear_solve.cu.
#include "engine.hpp"

namespace mgbx {
namespace {

bool stop_test(int kind, double lambda_tol, double theta, double ymin, double ynext, double gmin, double gnext, double ndec) {
  const bool ex = (ynext >= ymin) && (gnext >= theta * gmin);
  if (kind == 0) return ex;
  return (ndec < lambda_tol) || ex;
}

}  // namespace

Engine::NewtonOut Engine::newton(Amg &A, int J, double t, int maxit, int stop_kind, double lambda_tol, double theta,
                                 const mgbx_step_opts &o) {
  NewtonOut out{false, 0, MGBX_OK, 0.0, 0.0, 0.0};
  const int64_t m = A.m[J];
  System &S = system_for(A, J);
  if (dist() && J == A.L - 1)
    for (int v : S.kept)
      if (A.var_local[v]) throw std::runtime_error("multi-GPU: a node-local state variable could not be condensed out of the Newton system");
  // the finalize pass stops on floating-point stagnation (stopping_exact): give it directions converged to the
  // attainable accuracy so that it stagnates where a direct solve would
  const double rt = (stop_kind == 0) ? std::min(h->cfg.pcg_rtol, h->cfg.pcg_rtol_final) : h->cfg.pcg_rtol;
  const SolveTol tol{rt * rt, (stop_kind == 0) ? 6 : std::max(1, h->cfg.pcg_stall_window)};   // finalize: iterate to the attainable accuracy, detected quickly
  h->last_tol = tol;
  zero(A.x, m);
  EvalOut e0 = eval_f01(A, J, t, A.z, A.x, A.g);
  if (!e0.finite) {
    if (h->cfg.verbose > 0)
      fprintf(stderr, "[mgbx] newton J=%d: starting point outside the domain (y=%g, non-finite nodes=%g, |g|=%g)\n", J, e0.y, e0.nonfinite_nodes, e0.gnorm);
    out.status = MGBX_NON_FINITE;
    out.y = e0.y;
    return out;
  }
  double y = e0.y, gnorm = e0.gnorm;
  double ymin = y, gmin = gnorm, incmin = INFINITY;
  bool converged = false;
  int k = 0;
  const double eps = 2.220446049250313e-16;
  while (k < maxit && !converged) {
    ++k;
    assemble(A, S, J, t, A.z, A.x);
    const SolveResult sr = solve(A, S, J, A.g, A.dir, tol);
    const int pit = sr.iters;
    const double inc = sr.dg.ab;
    const bool dir_finite = (sr.dg.nonfinite == 0.0) && std::isfinite(sr.dg.aa) && std::isfinite(inc);
    out.inc = inc;
    if (h->cfg.verbose > 1)
      fprintf(stderr, "[mgbx] newton J=%d m=%lld k=%d y=%.17g |g|=%.6g lam2=%.6g pcg=%d status=%d rel=%.3g erel=%.3g t=%g\n", J, (long long)m, k, y, gnorm, inc, pit,
              sr.status, sr.rel, sr.erel, t);
    // An iterative solve that broke down or stopped far from the requested residual is a FAILED solve, as a failed
    // factorisation is for the reference's direct `H \\ g` (src/utils.jl:142-145): for a CG iterate g.x_k <= g.H^-1 g, so an
    // under-converged direction under-estimates the Newton decrement and could end the iteration early with a wrong z.
    // The Newton run is reported as not converged; mgb_core then shrinks kappa (or phase I grows the box).
    bool solve_inexact = false;
    if (sr.status < 0) {   // breakdown (indefinite or non-finite): no direction at all
      if (h->cfg.verbose > 0)
        fprintf(stderr, "[mgbx] newton J=%d m=%lld k=%d: linear solve broke down after %d PCG iterations\n", J, (long long)m, k, pit < 0 ? -pit : pit);
      if (h->res) h->res->solve_failures++;
      break;
    }
    if (sr.rel > 0.5 && sr.erel > h->cfg.pcg_fail_etol) {   // no better than the zero vector: a failed solve
      if (h->cfg.verbose > 0)
        fprintf(stderr, "[mgbx] newton J=%d m=%lld k=%d: linear solve failed (status %d, |r|/|b| = %.3g after %d PCG iterations)\n", J, (long long)m, k,
                sr.status, sr.rel, pit < 0 ? -pit : pit);
      if (h->res) h->res->solve_failures++;
      break;
    }
    if (sr.rel > h->cfg.pcg_fail_rtol && sr.erel > h->cfg.pcg_fail_etol) {
      // under-converged: the direction is still a descent direction and is used (inexact Newton, guarded by the line search),
      // but its decrement is not trusted to end the iteration
      solve_inexact = true;
      if (h->res) h->res->solve_failures++;
      if (h->cfg.verbose > 0)
        fprintf(stderr, "[mgbx] newton J=%d m=%lld k=%d: inexact linear solve (status %d, |r|/|b| = %.3g, energy gained in the last 4 iterations %.3g, after %d PCG iterations)\n",
                J, (long long)m, k, sr.status, sr.rel, sr.erel, pit < 0 ? -pit : pit);
    }
    if (!dir_finite) {
      if (h->cfg.verbose > 0)
        fprintf(stderr, "[mgbx] newton J=%d m=%lld k=%d: non-finite direction (g.d=%g |d|^2=%g non-finite entries=%g, pcg=%d, |r|/|b|=%g)\n", J,
                (long long)m, k, inc, sr.dg.aa, sr.dg.nonfinite, pit, sr.rel);
      out.status = MGBX_NON_FINITE;
      break;
    }
    if (inc <= 0.0) {
      converged = std::fabs(inc) <= eps * std::max(std::fabs(y), 1.0);
      break;
    }
    double sstep = 1.0;
    double yn = y, gnn = gnorm;
    bool have_trial = false;   // xbest/gbest hold the last finite trial
    // exact line search by Illinois root finding on phi(sigma) = F1(x - sigma n).n  (newton.jl:4-27,84-103)
    while (o.line_search == 1 && sstep > 0.0) {
      bool ok = true;
      auto phi = [&](double sigma) -> double {
        const TrialOut e = eval_trial(A, J, t, sigma);
        if (!std::isfinite(e.y)) {   // "line search: non-finite barrier value"
          ok = false;
          return NAN;
        }
        const double fc = dot2(A, J, A.gn, A.dir).ab;
        if (!std::isfinite(fc)) ok = false;   // @assert isfinite(fc)
        return fc;
      };
      double a = 0.0, b = sstep, fa = inc, fb = phi(b), sstar = b;
      if (ok) {
        if (fa == 0.0) sstar = a;
        else if (fa * fb >= 0.0) sstar = b;
        else {
          bool found = false;
          for (int kk = 0; kk < 10000 && ok; ++kk) {
            const double c = (a * fb - b * fa) / (fb - fa);
            const double fc = phi(c);
            if (!ok) break;
            if (c <= std::min(a, b) || c >= std::max(a, b) || fc * fa == 0.0 || fc * fb == 0.0) {
              sstar = c;
              found = true;
              break;
            }
            if (fb * fc < 0.0) {
              a = b;
              fa = fb;
            } else {
              fa /= 2.0;
            }
            b = c;
            fb = fc;
          }
          if (!found) ok = false;   // trial rejected (or "Illinois solver failed to converge")
        }
      }
      if (ok) {
        const TrialOut et = eval_trial(A, J, t, sstar);
        if (et.finite) {
          std::swap(A.xn, A.xbest);
          std::swap(A.gn, A.gbest);
          have_trial = true;
          yn = et.y;
          gnn = et.gnorm;
          break;
        }
      }
      sstep *= o.ls_beta;
    }
    // backtracking line search (newton.jl:139-154 with the trial loop of :35-50)
    while (o.line_search == 0 && sstep > 0.0) {
      const TrialOut et = eval_trial(A, J, t, sstep);
      const bool stalled = (et.step2 == 0.0);
      if (et.finite) {
        std::swap(A.xn, A.xbest);
        std::swap(A.gn, A.gbest);
        have_trial = true;
        yn = et.y;
        gnn = et.gnorm;
        if (stalled || yn <= y - o.ls_c1 * inc * sstep) break;
      }
      sstep *= o.ls_beta;
    }
    // an under-converged solve under-estimates the decrement (g.x_k <= g.H^-1 g): only the stagnation rule may stop then
    if (stop_test(solve_inexact ? 0 : stop_kind, lambda_tol, theta, ymin, yn, gmin, gnn, std::sqrt(inc))) converged = true;
    if (have_trial) {
      std::swap(A.x, A.xbest);
      std::swap(A.g, A.gbest);
    }
    y = yn;
    gnorm = gnn;
    gmin = std::min(gmin, gnorm);
    ymin = std::min(ymin, y);
    incmin = std::min(inc, incmin);
  }
  out.converged = converged;
  out.k = k;
  out.y = y;
  out.gnorm = gnorm;
  return out;
}

int Engine::step(int which, double t, const mgbx_step_opts &o, mgbx_step_result *r) {
  Amg &A = h->amg[which];
  memset(r, 0, sizeof(*r));
  h->res = r;
  const int L = A.L;
  copy(A.zsave, A.z, (int64_t)A.nu * A.n);
  int status = MGBX_OK;
  // eta(j, J): Newton in range(R_fine[J]) around the current z (levels 1-based as in the reference)
  auto eta = [&](int j, int J, int stop_kind, double ltol, double theta, int mxit) -> bool {
    (void)j;
    if (status != MGBX_OK) return false;
    NewtonOut n = newton(A, J - 1, t, mxit, stop_kind, ltol, theta, o);
    r->its[J - 1] += n.k;
    r->y = n.y;
    r->gnorm = n.gnorm;
    r->inc = n.inc;
    if (n.status != MGBX_OK) {
      status = n.status;
      return false;
    }
    if (n.converged) {
      prolong_to_fine(A, J - 1, A.x, A.z, A.zf);
      std::swap(A.z, A.zf);
    }
    return n.converged;
  };
  std::function<bool(int, int)> dac = [&](int j, int J) -> bool {
    const int mn = (o.initial_step && J - j == 1) ? o.maxit : o.max_newton;
    if (eta(j, J, o.stop_kind, o.stop_lambda_tol, o.stop_theta, mn)) return true;
    const int jmid = (j + J) / 2;
    if (jmid == j || jmid == J) return false;
    return dac(j, jmid) && dac(jmid, J);
  };
  bool converged = dac(0, L);
  copy(A.zunfin, A.z, (int64_t)A.nu * A.n);   // SOL.z_unfinalized (mgb.jl:76-80)
  if (o.finalize && status == MGBX_OK) {
    const int before = r->its[L - 1];
    const bool foo = eta(L - 1, L, 0, 0.0, o.finalize_theta, o.maxit);
    r->its_finalize = r->its[L - 1] - before;   // bookkeeping: the reference adds the finalize pass into its[L]
    converged = converged && foo;
  }
  r->converged = converged ? 1 : 0;
  if (status != MGBX_OK || !converged) copy(A.z, A.zsave, (int64_t)A.nu * A.n);   // the caller discards a failed step (mgb.jl:147-163)
  sync();
  h->res = nullptr;
  if (status != MGBX_OK || !converged) return status != MGBX_OK ? status : MGBX_NOT_CONVERGED;
  return MGBX_OK;
}

int Engine::matched_t(double t_default, double *t_out, double *tstar_out) {
  Amg &A = h->amg[MGBX_MAIN];
  const int J = A.L - 1;
  const int64_t m = A.m[J];
  System &S = system_for(A, J);
  zero(A.x, m);
  EvalOut e0 = eval_f01(A, J, 0.0, A.z, A.x, A.g);        // g = grad of the barrier term
  EvalOut e1 = eval_f01(A, J, 1.0, A.z, A.x, A.gn);       // gn = gphi + gc
  (void)e0;
  (void)e1;
  axpby(m, 1.0, A.gn, -1.0, A.g, A.gn);   // gn = gc
  assemble(A, S, J, 1.0, A.z, A.x);
  solve(A, S, J, A.g, A.dir, h->last_tol);                       // nphi
  const double d = solve(A, S, J, A.gn, A.xn, h->last_tol).dg.ab;   // gc . nc
  const double b1 = dot2(A, J, A.xn, A.g).ab;
  const double b = b1 + dot2(A, J, A.dir, A.gn).ab;
  *tstar_out = NAN;
  *t_out = t_default;
  if (!(d > 0.0)) return MGBX_OK;
  const double tstar = -b / (2.0 * d);
  *tstar_out = tstar;
  if (!(std::isfinite(tstar) && tstar > 0.0)) return MGBX_OK;
  *t_out = std::min(std::max(tstar, std::sqrt(2.220446049250313e-16)), t_default);
  return MGBX_OK;
}

}  // namespace mgbx
