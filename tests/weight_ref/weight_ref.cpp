// ORACLE TRUTH-MODEL REPLAY WITH A TORQUER LIMIT -- TEST INFRASTRUCTURE ONLY.
// The CPU reference of the weight-sweep ensemble (ts_mc_weight_ensemble, WE2 and WE4 of DESIGN.md section 4, K4): the
// dispersion ensemble's truth-model replay (tests/dispersion_ref/dispersion_ref.cpp, included unchanged for its truth
// model simulator_truth), with the gains of the weighting in the options passed in, and every component of the
// commanded dipole saturated at +-u_limit (u_limit > 0) before it drives the rk4 step.  Written from the rules, not from
// the kernel source.  Built by tests/weight_ref.py.
#include <algorithm>

#include "../dispersion_ref/dispersion_ref.cpp"

extern "C" {

// As dre_attitude_simulation_truth (prm, noise, outputs), with the limit u_limit (0: none).  Returns N_sim.
int64_t wre_attitude_simulation_truth_limited(const dre_dyn* d, const dre_tvlqr_opts* o, int64_t N, const double* X_lqr,
                                              const double* U_lqr, const double* x0, const double* noise, const double* prm,
                                              double* X_sim, double* K, double u_limit) {
  DynCtx c;
  c.B_eci = d->B_eci;
  c.B_rows = d->B_rows;
  c.index_scale = d->index_scale;
  c.clock_rate = d->clock_rate;
  for (int i = 0; i < 9; ++i) c.J[i] = d->J[i];
  inv3(c.J, c.Jinv);
  TvlqrOpts t;
  t.dt = o->dt; t.t0 = o->t0; t.tf = o->tf; t.dt_squared = o->dt_squared;
  for (int i = 0; i < 6; ++i) { t.Qd[i] = o->Qd[i]; t.Qfd[i] = o->Qfd[i]; }
  for (int i = 0; i < 3; ++i) t.Rd[i] = o->Rd[i];
  // the gains of the nominal model under the weighting of o (attitude_simulation's own; its closed loop is discarded)
  std::vector<double> Xn((size_t)N * 8), Un((size_t)N * 3), dXn((size_t)N * 6);
  const int64_t N_sim = attitude_simulation(c, t, N, X_lqr, U_lqr, x0, noise, Xn.data(), Un.data(), dXn.data(), K);
  // the truth model of prm
  Truth tr;
  tr.c = c;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) tr.c.J[i * 3 + j] = prm[i] * c.J[i * 3 + j] * prm[j];
  inv3(tr.c.J, tr.c.Jinv);
  for (int i = 0; i < 3; ++i) tr.g[i] = prm[3 + i];
  tr.sB = prm[6];
  const double th = std::sqrt(prm[7] * prm[7] + prm[8] * prm[8] + prm[9] * prm[9]);
  tr.rot = th > 1e-300;
  tr.p[0] = std::cos(th / 2);
  for (int i = 0; i < 3; ++i) tr.p[1 + i] = tr.rot ? prm[7 + i] / th * std::sin(th / 2) : 0.0;
  // the closed loop with the command limit
  constexpr int n = 8, m = 3;
  std::vector<double> U_sim((size_t)N_sim * m, 0.0);
  for (int64_t i = 0; i < N_sim * n; ++i) X_sim[i] = 0;
  for (int i = 0; i < n; ++i) X_sim[i] = x0[i];
  for (int64_t k = 0; k < N_sim - 1; ++k) {
    double dx[6];
    for (int i = 0; i < 3; ++i) dx[i] = X_sim[k * n + i] - X_lqr[k * n + i];
    double qi[4], qe[4];
    q_inv(X_lqr + k * n + 3, qi);
    qmult(qi, X_sim + k * n + 3, qe);
    for (int i = 0; i < 3; ++i) dx[3 + i] = qe[1 + i];
    for (int i = 0; i < m; ++i) {
      double s = 0;
      for (int j = 0; j < 6; ++j) s += K[k * 18 + i * 6 + j] * dx[j];
      U_sim[k * m + i] = U_lqr[k * m + i] - s;
      if (u_limit > 0) U_sim[k * m + i] = std::min(std::max(U_sim[k * m + i], -u_limit), u_limit);
    }
    const double* nz = noise ? noise + k * 36 : nullptr;
    rk4_step<double>([&](int stage, const double* xx, const double* uu, double* dxx) { simulator_truth(tr, xx, uu, nz ? nz + stage * 9 : nullptr, dxx); },
                     X_sim + k * n, &U_sim[k * m], o->dt, X_sim + (k + 1) * n);
  }
  return N_sim;
}

}  // extern "C"
