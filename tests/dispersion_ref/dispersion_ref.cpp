// ORACLE TRUTH-MODEL REPLAY -- TEST INFRASTRUCTURE ONLY.
// attitude_simulation (oracle/orc_tvlqr.hpp) with a truth model that differs from the planning model, the CPU reference
// of the dispersion ensemble (ts_mc_dispersion_ensemble, DE2 of DESIGN.md section 4, K4): the gains come from the
// nominal DynCtx exactly as in attitude_simulation, and the closed loop integrates simulator() (reference
// src/simulator.jl:1-42) with the truth inertia J_true[i][j] = (d_i J[i][j]) d_j and its inverse, the torque
// ((u / 100) * g_i) x B_B, and the stage field s_B * qrot(p, B_row) + B_noise (the model error on the table row first,
// then the noise).  Written from the rules, not from the kernel source.  Built by tests/dispersion_ref.py.
#include <cmath>
#include <cstdint>
#include <vector>

#include "../../oracle/orc_tvlqr.hpp"

using namespace orc;

namespace {

struct Truth {
  DynCtx c;        // truth inertia, nominal field table and clock
  double g[3];     // torquer gains
  double sB;       // field scale
  double p[4];     // field rotation
  bool rot;
};

void simulator_truth(const Truth& t, const double x[8], const double u[3], const double* noise, double dx[8]) {
  const DynCtx& c = t.c;
  double om[3] = {x[0], x[1], x[2]};
  const double nq = std::sqrt(x[3] * x[3] + x[4] * x[4] + x[5] * x[5] + x[6] * x[6]);
  double q[4] = {x[3] / nq, x[4] / nq, x[5] / nq, x[6] / nq};
  const double* Bn = field_row(c, x[7]);
  double Bm[3] = {Bn[0], Bn[1], Bn[2]};
  if (t.rot) qrot(t.p, Bn, Bm);
  for (int i = 0; i < 3; ++i) Bm[i] = t.sB * Bm[i];
  double Bf[3] = {Bm[0], Bm[1], Bm[2]};
  if (noise) {
    for (int i = 0; i < 3; ++i) om[i] = x[i] + noise[i];
    const double th = std::sqrt(noise[3] * noise[3] + noise[4] * noise[4] + noise[5] * noise[5]);
    const double qn[4] = {std::cos(th / 2), noise[3] / th * std::sin(th / 2), noise[4] / th * std::sin(th / 2),
                          noise[5] / th * std::sin(th / 2)};
    double q2[4];
    qmult(q, qn, q2);
    for (int i = 0; i < 4; ++i) q[i] = q2[i];
    for (int i = 0; i < 3; ++i) Bf[i] = Bm[i] + noise[6 + i];
  }
  const double w4[4] = {0.0, om[0], om[1], om[2]};
  double qd[4];
  qmult(q, w4, qd);
  double BB[3];
  qrot(q, Bf, BB);
  const double us[3] = {u[0] / 100 * t.g[0], u[1] / 100 * t.g[1], u[2] / 100 * t.g[2]};
  double tau[3];
  cross3(us, BB, tau);
  double Jw[3];
  for (int i = 0; i < 3; ++i) Jw[i] = c.J[i * 3 + 0] * om[0] + c.J[i * 3 + 1] * om[1] + c.J[i * 3 + 2] * om[2];
  double wJw[3];
  cross3(om, Jw, wJw);
  const double rhs[3] = {tau[0] - wJw[0], tau[1] - wJw[1], tau[2] - wJw[2]};
  for (int i = 0; i < 3; ++i) dx[i] = c.Jinv[i * 3 + 0] * rhs[0] + c.Jinv[i * 3 + 1] * rhs[1] + c.Jinv[i * 3 + 2] * rhs[2];
  for (int i = 0; i < 4; ++i) dx[3 + i] = 0.5 * qd[i];
  dx[7] = c.clock_rate;
}

}  // namespace

extern "C" {

// The layouts of oracle.cpp's orc_dyn and orc_tvlqr_opts (oracle.py's Dyn and TvlqrOpts).
struct dre_dyn {
  const double* B_eci;
  int64_t B_rows;
  double index_scale, clock_rate;
  double J[9];
};
struct dre_tvlqr_opts {
  double dt, t0, tf;
  double Qd[6], Qfd[6], Rd[3];
  int32_t dt_squared, noise_mode;
  uint64_t seed;
};

// prm: d0 d1 d2 g0 g1 g2 s_B phi0 phi1 phi2.  noise: (N x 4 x 9) explicit stage draws, nullable.  Outputs X_sim (N_sim x 8)
// and K ((N-1) x 18, the nominal gains); returns N_sim.
int64_t dre_attitude_simulation_truth(const dre_dyn* d, const dre_tvlqr_opts* o, int64_t N, const double* X_lqr, const double* U_lqr,
                                      const double* x0, const double* noise, const double* prm, double* X_sim, double* K) {
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
  // the gains of the nominal model (attitude_simulation's own; its nominal closed loop is discarded)
  std::vector<double> Xn((size_t)N * 8), Un((size_t)N * 3), dXn((size_t)N * 6);
  const int64_t N_sim = attitude_simulation(c, t, N, X_lqr, U_lqr, x0, noise, Xn.data(), Un.data(), dXn.data(), K);
  // the truth model
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
  // the closed loop of attitude_simulation with simulator_truth
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
    }
    const double* nz = noise ? noise + k * 36 : nullptr;
    rk4_step<double>([&](int stage, const double* xx, const double* uu, double* dxx) { simulator_truth(tr, xx, uu, nz ? nz + stage * 9 : nullptr, dxx); },
                     X_sim + k * n, &U_sim[k * m], o->dt, X_sim + (k + 1) * n);
  }
  return N_sim;
}

}  // extern "C"
