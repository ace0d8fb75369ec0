// ORACLE CONTINUATION -- TEST INFRASTRUCTURE ONLY.
//
// The oracle's AL-iLQR solve (oracle/orc_ilqr.hpp, alilqr_solve) with the solver state of DESIGN.md section 4, K3
// (rules CS1-CS3) taken in and given out, so that "solve to M1, continue to M2" can be checked against "solve to M2"
// on the CPU and the GPU continuation against an independent one.  The outer loop below is alilqr_solve's, statement
// for statement; only the start (fresh or imported) and the export at the end are new.  With no state in it computes
// what alilqr_solve computes (tests/test_alilqr_state.py checks that bit for bit).
#pragma once
#include <cassert>

#include "../../oracle/orc_ilqr.hpp"

namespace orc {

struct AlState {   // = ts_al_state
  double mu, lam_goal[8], J, c_max;
  int32_t status, outer_iters, inner_iters, ls_rollouts;
};
static_assert(sizeof(AlState) == 104, "ts_al_state layout");

// X, U: outputs; with sin set also the imported trajectory (X columns 0..6, U) of a continuing trial.  lam: ragged
// N x 6 (last row unused).  A trial that does not continue (CS2) passes through: X, U, K untouched, the outcome
// rebuilt from the state, the state and lam copied.
inline void alilqr_solve_state(const IlqrProblem& p, const IlqrOpts& o, const double* U0, double* Xout, double* Uout, double* Kout,
                               IlqrOutcome* out, const AlState* sin, const double* lam_in, AlState* sout, double* lam_out) {
  using namespace detail;
  const int64_t N = p.N;
  if (sin && !(sin->status == ST_MAX_OUTER && sin->outer_iters < o.max_outer)) {   // CS2: pass through
    *out = IlqrOutcome{sin->status, sin->outer_iters, sin->inner_iters, sin->ls_rollouts, N, sin->J, sin->c_max, 0, 0, 0};
    if (sout) *sout = *sin;
    if (lam_out)
      for (int64_t i = 0; i < N * nb; ++i) lam_out[i] = lam_in[i];
    return;
  }
  Work w(p.N);
  int status = ST_MAX_OUTER, outer = 0, inner_total = 0, ls_total = 0;
  double J = 0, c_max = 0, c_max_prev = INFINITY;
  int first = 1;
  if (sin) {
    // CS3: the imported trajectory (not rolled out again; the clock column recomputed as the rollout computes it),
    // multipliers, and the penalty -- the oracle keeps one per constraint, A6 moves them all together
    for (int64_t i = 0; i < (N - 1) * m; ++i) w.U[i] = Uout[i];
    for (int64_t k = 0; k < N; ++k)
      for (int i = 0; i < 7; ++i) w.X[k * n + i] = Xout[k * n + i];
    w.X[7] = p.x0[7];
    for (int64_t k = 0; k < N - 1; ++k) {
      double xn[n];
      step(p, &w.X[k * n], &w.U[k * m], xn);
      w.X[(k + 1) * n + 7] = xn[7];
    }
    for (int64_t i = 0; i < (N - 1) * nb; ++i) {
      w.lam_b[i] = lam_in[i];
      w.mu_b[i] = sin->mu;
    }
    for (int i = 0; i < n; ++i) {
      w.lam_g[i] = sin->lam_goal[i];
      w.mu_g[i] = sin->mu;
    }
    outer = sin->outer_iters;
    inner_total = sin->inner_iters;
    ls_total = sin->ls_rollouts;
    J = sin->J;
    c_max = sin->c_max;
    c_max_prev = sin->c_max;
    first = sin->outer_iters + 1;
  } else {
    for (int64_t i = 0; i < (N - 1) * m; ++i) w.U[i] = U0 ? U0[i] : 0.0;
    for (int64_t i = 0; i < (N - 1) * nb; ++i) {
      w.lam_b[i] = 0;
      w.mu_b[i] = o.penalty_initial;
    }
    for (int i = 0; i < n; ++i) {
      w.lam_g[i] = 0;
      w.mu_g[i] = o.penalty_initial;
    }
    // initial rollout (open loop)
    for (int i = 0; i < n; ++i) w.X[i] = p.x0[i];
    for (int64_t k = 0; k < N - 1; ++k) step(p, &w.X[k * n], &w.U[k * m], &w.X[(k + 1) * n]);
  }
  for (int oi = first; oi <= o.max_outer; ++oi) {
    outer = oi;
    const bool last = (oi == o.max_outer) || o.a4_no_intermediate;
    const double ctol = last ? o.cost_tol : o.cost_tol_intermediate;
    const double gtol = last ? o.grad_tol : o.grad_tol_intermediate;
    Reg reg;
    double J_prev = al_cost(p, o, w, w.X.data(), w.U.data(), nullptr);
    if (o.a7_carry_cost && oi > 1) J_prev = J;  // A7 alternative: the cost carried over from the previous inner solve
    J = J_prev;
    int dJ_zero = 0;
    bool abort_trial = false;
    for (int it = 1; it <= o.max_inner; ++it) {
      ++inner_total;
      jacobians(p, w);
      double dV[2];
      if (!backward_pass(p, o, w, reg, dV)) {
        status = ST_REG_MAX;
        abort_trial = true;
        break;
      }
      double alpha = 1.0, z = -1.0, expected = 0.0, Jn = INFINITY;
      int iter = 0;
      bool accepted = true;
      while ((z <= o.ls_lower || z > o.ls_upper) && (Jn >= J_prev)) {
        if (iter > o.max_linesearch) {
          accepted = false;
          Jn = al_cost(p, o, w, w.X.data(), w.U.data(), nullptr);
          z = 0;
          alpha = 0;
          expected = 0;
          reg_increase(o, reg);
          reg.rho += o.bp_reg_fp;
          break;
        }
        ++ls_total;
        const bool ok = rollout(p, o, w, alpha);
        if (!ok) {
          ++iter;
          alpha /= 2.0;
          continue;
        }
        Jn = al_cost(p, o, w, w.Xb.data(), w.Ub.data(), nullptr);
        expected = -alpha * (dV[0] + alpha * dV[1]);
        z = (expected > 0) ? (J_prev - Jn) / expected : -1.0;
        ++iter;
        alpha /= 2.0;
      }
      if (accepted) {
        w.X = w.Xb;
        w.U = w.Ub;
      }
      if (!(Jn == Jn)) {
        status = ST_NAN;
        abort_trial = true;
        break;
      }
      if (Jn > o.max_cost_value) {
        J = Jn;
        status = ST_COST_BLOWUP;
        abort_trial = true;
        break;
      }
      const double dJ = std::fabs(Jn - J_prev);
      J_prev = Jn;
      J = Jn;
      if (dJ == 0) ++dJ_zero; else dJ_zero = 0;
      double g = 0;
      for (int64_t k = 0; k < N - 1; ++k) {
        double mxv = 0;
        for (int i = 0; i < m; ++i) mxv = std::max(mxv, std::fabs(w.d[k * m + i]) / (std::fabs(w.U[k * m + i]) + 1.0));
        g += mxv;
      }
      g /= (double)(o.a3_grad_over_N ? N : N - 1);
      if ((0.0 < dJ && dJ < ctol) || g < gtol || dJ_zero > o.dJ_counter_limit) break;
    }
    J = al_cost(p, o, w, w.X.data(), w.U.data(), &c_max);
    if (abort_trial) break;
    const bool grow = !o.a6_penalty_conditional || (c_max > o.constraint_decrease_ratio * c_max_prev);
    c_max_prev = c_max;
    for (int64_t k = 0; k < N - 1; ++k) {
      double c[nb];
      bound_c(o, &w.U[k * m], c);
      for (int i = 0; i < nb; ++i) {
        const double l0 = w.lam_b[k * nb + i];
        const bool act = (o.a2_active_ge ? (c[i] >= 0.0) : (c[i] > 0.0)) || (l0 > 0.0);
        double l = l0 + w.mu_b[k * nb + i] * c[i];
        l = std::min(std::max(l, -o.dual_max), o.dual_max);
        if (o.a5_dual_active_only && !act) l = l0;
        w.lam_b[k * nb + i] = std::max(0.0, l);
        if (grow) w.mu_b[k * nb + i] = std::min(w.mu_b[k * nb + i] * o.penalty_scaling, o.penalty_max);
      }
    }
    for (int i = 0; i < n; ++i) {
      if (!(o.goal_mask & (1 << i))) continue;
      const double e = w.X[(N - 1) * n + i] - p.xf[i];
      double l = w.lam_g[i] + w.mu_g[i] * e;
      w.lam_g[i] = std::min(std::max(l, -o.dual_max), o.dual_max);
      if (grow) w.mu_g[i] = std::min(w.mu_g[i] * o.penalty_scaling, o.penalty_max);
    }
    if (c_max < o.constraint_tol) {
      status = ST_CONVERGED;
      break;
    }
  }
  for (int64_t i = 0; i < N * n; ++i) Xout[i] = w.X[i];
  for (int64_t i = 0; i < (N - 1) * m; ++i) Uout[i] = w.U[i];
  if (Kout)
    for (int64_t i = 0; i < (N - 1) * m * n; ++i) Kout[i] = w.K[i];
  *out = IlqrOutcome{status, outer, inner_total, ls_total, N, J, c_max, 0, 0, 0};
  // CS1 export.  Under A6 every penalty moves together: the state holds the one value
  const double mu = (N > 1) ? w.mu_b[0] : o.penalty_initial;
  for (int64_t i = 0; i < (N - 1) * nb; ++i) assert(w.mu_b[i] == mu);
  for (int i = 0; i < n; ++i) assert(!(o.goal_mask & (1 << i)) || w.mu_g[i] == mu);
  if (sout) {
    sout->mu = mu;
    for (int i = 0; i < n; ++i) sout->lam_goal[i] = w.lam_g[i];
    sout->J = J;
    sout->c_max = c_max;
    sout->status = status;
    sout->outer_iters = outer;
    sout->inner_iters = inner_total;
    sout->ls_rollouts = ls_total;
  }
  if (lam_out) {
    for (int64_t i = 0; i < (N - 1) * nb; ++i) lam_out[i] = w.lam_b[i];
    for (int i = 0; i < nb; ++i) lam_out[(N - 1) * nb + i] = 0.0;
  }
}

}  // namespace orc
