// TVLQR closed-loop replay of ONE optimised slew (one thread per trial) and the
// Monte-Carlo slew-time post-processing.  Replaces
//   attitude_simulation(f!,f_gains!,:rk4,X,U,dt,x0,t0,tf,Q,R,Qf)   reference src/attitude_controller.jl:1-48
//   attitude_lqr (ForwardDiff Jacobians of rk4(f_augmented(gain_simulator)))  :95-119
//   attitude_lqr (G(q) projection to 6x6/6x3 + backward Riccati)            :50-93
//   rk4 of simulator with fresh noise in every stage                        :122-132, src/simulator.jl:1-42
//   slew-time / fail detection of the Monte-Carlo script                    src/monte_carlo.jl:237-262
// Quirks kept: the linearisation step is dt^2 (attitude_controller.jl:111,137, Q6);
// u/100 in the simulators (Q8); noise redrawn in each RK stage (Q7).
#pragma once
#include <stdint.h>

#include "ilqr_math.cuh"
#include "philox.cuh"

struct ts_tvlqr_opts_dev {
  double dt, t0, tf;
  double Qd[6], Qfd[6], Rd[3];
  int32_t dt_squared;   // 1 = reference behaviour (Q6)
  int32_t noise_mode;   // 0 none, 1 explicit array, 2 Philox(seed, trial, step, stage)
  uint64_t seed;
  // slew-time detection (monte_carlo.jl:69-71,237-262)
  double w_limit, ang_limit;
  int32_t literal_postproc;  // 1 = keep the `[1:3,i]` column bug (Q12)
  int32_t pad_;
};

namespace ts {

// length(a:s:b) for Float64 ranges (t_sim / t_total)
TS_HD long long range_len(double a, double s, double b) {
  if (b < a) return 0;
  return (long long)floor((b - a) / s + 1e-9) + 1;
}

TS_HD void inv3_general(const double A[9], double out[9]) {
  // Gauss-Jordan with partial pivoting (== inv() of a dense 3x3)
  double M[3][6];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      M[i][j] = A[i * 3 + j];
      M[i][3 + j] = (i == j) ? 1.0 : 0.0;
    }
  for (int c = 0; c < 3; ++c) {
    int p = c;
    for (int r = c + 1; r < 3; ++r)
      if (fabs(M[r][c]) > fabs(M[p][c])) p = r;
    if (p != c)
      for (int j = 0; j < 6; ++j) {
        const double t = M[c][j];
        M[c][j] = M[p][j];
        M[p][j] = t;
      }
    const double piv = M[c][c];
    for (int j = 0; j < 6; ++j) M[c][j] /= piv;
    for (int r = 0; r < 3; ++r) {
      if (r == c) continue;
      const double f = M[r][c];
      if (f == 0.0) continue;
      for (int j = 0; j < 6; ++j) M[r][j] -= f * M[c][j];
    }
  }
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) out[i * 3 + j] = M[i][3 + j];
}

#ifdef __CUDA_ARCH__
#define TS_UNROLL _Pragma("unroll")
#else
#define TS_UNROLL
#endif

// inverse of a well-conditioned 3x3 (R + B'SB, symmetric positive definite and dominated by R) by the adjugate: no
// pivot search, hence no dynamically indexed scratch in the sequential Riccati sweep
TS_HD void inv3_adj(const double A[9], double out[9]) {
  const double c00 = A[4] * A[8] - A[5] * A[7], c01 = A[5] * A[6] - A[3] * A[8], c02 = A[3] * A[7] - A[4] * A[6];
  const double det = A[0] * c00 + A[1] * c01 + A[2] * c02;
  const double id = 1.0 / det;
  out[0] = c00 * id;
  out[1] = (A[2] * A[7] - A[1] * A[8]) * id;
  out[2] = (A[1] * A[5] - A[2] * A[4]) * id;
  out[3] = c01 * id;
  out[4] = (A[0] * A[8] - A[2] * A[6]) * id;
  out[5] = (A[2] * A[3] - A[0] * A[5]) * id;
  out[6] = c02 * id;
  out[7] = (A[1] * A[6] - A[0] * A[7]) * id;
  out[8] = (A[0] * A[4] - A[1] * A[3]) * id;
}

// The truth-model errors of one realisation of a dispersion ensemble (K4d, DE2 of DESIGN.md section 4, K4) that act in
// the stage dynamics: torquer gains, and the field transform s_B * qrot(p, row).  A group at its nominal value is
// skipped (torq / scale / rot false), so a realisation without errors runs K4e's arithmetic exactly (DE3, DE4).
struct TvlqrDisp {
  double g[3], sB, p[4];
  bool torq, scale, rot;
};

struct TvlqrIn {
  int N;                 // knots of the optimised trajectory
  const double* X_lqr;   // N x 8
  const double* U_lqr;   // (N-1) x 3
  double x0[8];
  Inertia I;
  const double* Bt;
  long long B_rows;
  double index_scale, clock_rate;
  const double* noise;   // (N_sim-1) x 4 x 9 or null
  uint32_t trial;        // Philox stream id
  uint32_t real = 0;     // realisation of a disturbance ensemble (counter blocks 4 real + {0,1,2}); 0 = the single replay
  double q_final[4];
  double t_final, time_step;
  long long trial_index_1based;
  TvlqrDisp disp;        // read by the dispersed instantiations (DISP = true) only
};

// A dispersed realisation's truth model from its ten parameters (dispersion_params): J_true[i][j] = (d_i J[i][j]) d_j in
// place of J (positive definite for any draw; the caller inverts it as for the nominal J), the torquer gains, and the
// field rotation p = [cos(|phi|/2); phi/|phi| sin(|phi|/2)] (the identity for |phi| <= 1e-300, tvlqr_stage_record's guard).
TS_HD void tvlqr_disp_setup(const double prm[10], double J[9], TvlqrDisp& d) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) J[i * 3 + j] = (prm[i] * J[i * 3 + j]) * prm[j];
  for (int i = 0; i < 3; ++i) d.g[i] = prm[3 + i];
  d.torq = prm[3] != 1.0 || prm[4] != 1.0 || prm[5] != 1.0;
  d.sB = prm[6];
  d.scale = prm[6] != 1.0;
  const double th = sqrt(prm[7] * prm[7] + prm[8] * prm[8] + prm[9] * prm[9]);
  d.rot = th > 1e-300;
  d.p[0] = 1.0;
  d.p[1] = d.p[2] = d.p[3] = 0.0;
  if (d.rot) {
    const double sh = sin(th / 2);
    d.p[0] = cos(th / 2);
    for (int i = 0; i < 3; ++i) d.p[1 + i] = prm[7 + i] / th * sh;
  }
}

// The truth field row of a dispersed stage: s_B * qrot(p, row); tvlqr_stage_record then adds the stage's field noise.
TS_HD void tvlqr_disp_field(const TvlqrDisp& d, const double* Bn, double out[3]) {
  if (d.rot) {
    qrot(d.p, Bn, out);
  } else {
    for (int i = 0; i < 3; ++i) out[i] = Bn[i];
  }
  if (d.scale)
    for (int i = 0; i < 3; ++i) out[i] = mul_rn(d.sB, out[i]);
}

// stage clocks of rk4 on the decoupled clock state: c = rate*h; x8, x8+c/2, x8+c/2, x8+c; next = x8 + (c+2c+2c+c)/6
TS_HD void clock_rk4(double x8, double rate, double h, double t[4], double& next) {
#ifdef __CUDA_ARCH__
  const double c = __dmul_rn(rate, h);
  t[0] = x8;
  t[1] = __dadd_rn(x8, __ddiv_rn(c, 2.0));
  t[2] = t[1];
  t[3] = __dadd_rn(x8, c);
  const double s = __dadd_rn(__dadd_rn(__dadd_rn(c, __dmul_rn(2.0, c)), __dmul_rn(2.0, c)), c);
  next = __dadd_rn(x8, __ddiv_rn(s, 6.0));
#else
  const volatile double c = rate * h;
  volatile double hc = c / 2.0;
  t[0] = x8;
  t[1] = x8 + hc;
  t[2] = t[1];
  t[3] = x8 + c;
  volatile double c2 = 2.0 * c;
  volatile double s = c + c2;
  s = s + c2;
  s = s + c;
  volatile double inc = s / 6.0;
  next = x8 + inc;
#endif
}

// ---- stage records -----------------------------------------------------------------------------------------------------
// Everything of one simulator() call (simulator.jl:1-42) that does not depend on the state, 10 doubles per rk4 stage:
//   [0:3) omega_noise   (randn(3)*(.38pi/180)^2, :5)
//   [3:7) the perturbation quaternion [cos(th/2); r sin(th/2)] of q_noise = randn(3)*(pi/180)^2 (:10-13); identity if none
//   [7:10) B_ECI[floor(t*N+1),:] + B_N_noise (:22) -- the field row of the stage's clock value, already perturbed
// The GPU path produces the records of all (trial, step, stage) in one fully parallel launch (K4n: Philox + Box-Muller +
// sincos + field lookup), so the sequential replay only multiplies and adds; the host emulator builds them on the fly
// with the same function, so both run the same arithmetic.
constexpr int TV_REC = 10;
TS_HD void tvlqr_stage_record(const double* nz9, const double* Bn, double rec[TV_REC]) {
  rec[0] = rec[1] = rec[2] = 0.0;
  rec[3] = 1.0;
  rec[4] = rec[5] = rec[6] = 0.0;
  for (int i = 0; i < 3; ++i) rec[7 + i] = Bn[i];
  if (nz9) {
    for (int i = 0; i < 3; ++i) rec[i] = nz9[i];
    const double th = sqrt(nz9[3] * nz9[3] + nz9[4] * nz9[4] + nz9[5] * nz9[5]);
    if (th > 1e-300) {  // a zero attitude perturbation is the identity (the reference's q_noise/0 would be NaN)
      const double sh = sin(th / 2);
      rec[3] = cos(th / 2);
      rec[4] = nz9[3] / th * sh;
      rec[5] = nz9[4] / th * sh;
      rec[6] = nz9[5] / th * sh;
    }
    for (int i = 0; i < 3; ++i) rec[7 + i] = Bn[i] + nz9[6 + i];
  }
}

// simulator(dx,x,u) (simulator.jl:1-42) for the 7 dynamic states, from a stage record.  q/|q| is x * rsqrt(q.q) (one
// rounding apart from the reference's four divisions, like the solver kernels; inside the 1e-10 rollout bar).
// DISP: a dispersed realisation's torque ((u_i * 0.01) * g_i) x B_B (I is then its truth inertia).
template <bool DISP = false>
TS_HD void simulator7_rec(const Inertia& I, const double x[7], const double u[3], const double* rec, double dx[7],
                          const TvlqrDisp* disp = nullptr) {
  const double om[3] = {x[0] + rec[0], x[1] + rec[1], x[2] + rec[2]};
  const double inq = rnorm(x[3] * x[3] + x[4] * x[4] + x[5] * x[5] + x[6] * x[6]);
  const double q0[4] = {x[3] * inq, x[4] * inq, x[5] * inq, x[6] * inq};
  double q[4];
  qmult(q0, rec + 3, q);
  const double w4[4] = {0.0, om[0], om[1], om[2]};
  double qd[4], BB[3], tau[3], Jw[3], wJw[3];
  qmult(q, w4, qd);
  qrot(q, rec + 7, BB);
  double us[3] = {u[0] * 0.01, u[1] * 0.01, u[2] * 0.01};
  if constexpr (DISP) {
    if (disp->torq)
      for (int i = 0; i < 3; ++i) us[i] = mul_rn(us[i], disp->g[i]);
  }
  cross3(us, BB, tau);
  for (int i = 0; i < 3; ++i) Jw[i] = I.J[i * 3 + 0] * om[0] + I.J[i * 3 + 1] * om[1] + I.J[i * 3 + 2] * om[2];
  cross3(om, Jw, wJw);
  const double r0 = tau[0] - wJw[0], r1 = tau[1] - wJw[1], r2 = tau[2] - wJw[2];
  for (int i = 0; i < 3; ++i) dx[i] = I.Jinv[i * 3 + 0] * r0 + I.Jinv[i * 3 + 1] * r1 + I.Jinv[i * 3 + 2] * r2;
  for (int i = 0; i < 4; ++i) dx[3 + i] = 0.5 * qd[i];
}

// ---- attitude_lqr, first method (attitude_controller.jl:95-119) + the G(q) projection of the second (:59-81), for ONE
// knot: the reduced discrete linearisation A (6x6), B (6x3) -> AB54 = [A row-major 36 | B row-major 18].
// The reference takes the full 12x12 ForwardDiff Jacobian of rk4(f_augmented(gain_simulator)) with step dt^2 (Q6) and then
// forms A = perm_Gn * Aq * perm_Gk, B = perm_Gn * Bq.  Here the 9 needed directional derivatives are taken directly:
// the three rate directions, the three columns of G(q_k) in the quaternion block (Aq * perm_Gk without ever forming Aq's
// four quaternion columns) and the three control directions -- the same numbers up to summation order (1e-16 relative).
TS_HD void tvlqr_linearise_knot(const Inertia& I, const double* xk, const double* xn_, const double* uk, const double* Bt, long long B_rows,
                                double index_scale, double clock_rate, double h, double* AB54) {
  double tcl[4], nxt;
  clock_rk4(xk[7], clock_rate, h, tcl, nxt);
  const double* Br[4];
  for (int s = 0; s < 4; ++s) Br[s] = Bt + (long long)field_row(tcl[s], index_scale, B_rows) * 3;
  // G(q) = [-v'; s I + hat(v)]   (attitude_controller.jl:59-71), row-major 4x3
  double Gn[12];
  {
    const double s = xn_[3], v0 = xn_[4], v1 = xn_[5], v2 = xn_[6];
    const double g[12] = {-v0, -v1, -v2, s, -v2, v1, v2, s, -v0, -v1, v0, s};
    for (int i = 0; i < 12; ++i) Gn[i] = g[i];
  }
  double dirs[90];
  for (int i = 0; i < 90; ++i) dirs[i] = 0.0;
  {
    const double s = xk[3], v0 = xk[4], v1 = xk[5], v2 = xk[6];
    const double Gk[12] = {-v0, -v1, -v2, s, -v2, v1, v2, s, -v0, -v1, v0, s};
    for (int d = 0; d < 3; ++d) {
      dirs[d * 10 + d] = 1.0;                                         // rate directions
      for (int l = 0; l < 4; ++l) dirs[(3 + d) * 10 + 3 + l] = Gk[l * 3 + d];   // column d of G(q_k)
      dirs[(6 + d) * 10 + 7 + d] = 1.0;                               // control directions
    }
  }
  double cols[63];
  rk4_jvp7(I, xk, uk, Br[0], Br[1], Br[2], Br[3], h, 9, dirs, cols);
  // perm_Gn * column: rows 0..2 copy, rows 3..5 = Gn' * (quaternion rows)
  for (int d = 0; d < 9; ++d) {
    const double* c = cols + d * 7;
    double r[6];
    for (int i = 0; i < 3; ++i) r[i] = c[i];
    for (int i = 0; i < 3; ++i) {
      double s = 0.0;
      for (int l = 0; l < 4; ++l) s += Gn[l * 3 + i] * c[3 + l];
      r[3 + i] = s;
    }
    if (d < 6)
      for (int i = 0; i < 6; ++i) AB54[i * 6 + d] = r[i];
    else
      for (int i = 0; i < 6; ++i) AB54[36 + i * 3 + (d - 6)] = r[i];
  }
}

// ---- attitude_lqr, second method (attitude_controller.jl:84-91): one backward Riccati step.
// K = inv(R + B'SB) (B'SA) ; S <- Q + K'RK + (A-BK)'S(A-BK).  Kout: 3x6 row-major.
TS_HD void tvlqr_riccati_step(const ts_tvlqr_opts_dev& o, const double* AB54, double S[36], double* Kout) {
  const double* A = AB54;
  const double* B = AB54 + 36;
  double SB[18], SA[36], BSB[9], BSA[18], Minv[9], Kk[18], Acl[36], SAcl[36];
  TS_UNROLL
  for (int i = 0; i < 6; ++i) {
    TS_UNROLL
    for (int j = 0; j < 3; ++j) {
      double s = 0.0;
      TS_UNROLL
      for (int l = 0; l < 6; ++l) s += S[i * 6 + l] * B[l * 3 + j];
      SB[i * 3 + j] = s;
    }
    TS_UNROLL
    for (int j = 0; j < 6; ++j) {
      double s = 0.0;
      TS_UNROLL
      for (int l = 0; l < 6; ++l) s += S[i * 6 + l] * A[l * 6 + j];
      SA[i * 6 + j] = s;
    }
  }
  TS_UNROLL
  for (int i = 0; i < 3; ++i) {
    TS_UNROLL
    for (int j = 0; j < 3; ++j) {
      double s = 0.0;
      TS_UNROLL
      for (int l = 0; l < 6; ++l) s += B[l * 3 + i] * SB[l * 3 + j];
      BSB[i * 3 + j] = s + ((i == j) ? o.Rd[i] : 0.0);
    }
    TS_UNROLL
    for (int j = 0; j < 6; ++j) {
      double s = 0.0;
      TS_UNROLL
      for (int l = 0; l < 6; ++l) s += B[l * 3 + i] * SA[l * 6 + j];
      BSA[i * 6 + j] = s;
    }
  }
  inv3_adj(BSB, Minv);
  TS_UNROLL
  for (int i = 0; i < 3; ++i)
    TS_UNROLL
    for (int j = 0; j < 6; ++j) {
      double s = 0.0;
      TS_UNROLL
      for (int l = 0; l < 3; ++l) s += Minv[i * 3 + l] * BSA[l * 6 + j];
      Kk[i * 6 + j] = s;
      Kout[i * 6 + j] = s;
    }
  TS_UNROLL
  for (int i = 0; i < 6; ++i)
    TS_UNROLL
    for (int j = 0; j < 6; ++j) {
      double s = 0.0;
      TS_UNROLL
      for (int l = 0; l < 3; ++l) s += B[i * 3 + l] * Kk[l * 6 + j];
      Acl[i * 6 + j] = A[i * 6 + j] - s;
    }
  TS_UNROLL
  for (int i = 0; i < 6; ++i)
    TS_UNROLL
    for (int j = 0; j < 6; ++j) {
      double s = 0.0;
      TS_UNROLL
      for (int l = 0; l < 6; ++l) s += S[i * 6 + l] * Acl[l * 6 + j];
      SAcl[i * 6 + j] = s;
    }
  double Sn[36];
  TS_UNROLL
  for (int i = 0; i < 6; ++i)
    TS_UNROLL
    for (int j = 0; j < 6; ++j) {
      double s = (i == j) ? o.Qd[i] : 0.0;
      double kr = 0.0;
      TS_UNROLL
      for (int l = 0; l < 3; ++l) kr += Kk[l * 6 + i] * o.Rd[l] * Kk[l * 6 + j];
      s += kr;
      double t = 0.0;
      TS_UNROLL
      for (int l = 0; l < 6; ++l) t += Acl[l * 6 + i] * SAcl[l * 6 + j];
      Sn[i * 6 + j] = s + t;
    }
  TS_UNROLL
  for (int i = 0; i < 36; ++i) S[i] = Sn[i];
}

// Gains K ((N-1) x 18, row-major 3x6 per knot) -- attitude_lqr, both methods, for one trial in one thread (host
// lane-emulator and small batches; the GPU path runs the linearisation as its own fully parallel kernel, K4a).
// ABp: optional precomputed linearisations ((N-1) x 54); null -> computed on the fly.
TS_HD void tvlqr_gains(const TvlqrIn& in, const ts_tvlqr_opts_dev& o, double* K, const double* ABp = nullptr) {
  const int N = in.N;
  const double h = o.dt_squared ? o.dt * o.dt : o.dt;
  double S[36];
  for (int i = 0; i < 36; ++i) S[i] = 0.0;
  for (int i = 0; i < 6; ++i) S[i * 6 + i] = o.Qfd[i];
  for (int k = N - 2; k >= 0; --k) {
    double AB[54];
    const double* ab = AB;
    if (ABp) {
      ab = ABp + (long long)k * 54;
    } else {
      tvlqr_linearise_knot(in.I, in.X_lqr + (long long)k * 8, in.X_lqr + (long long)(k + 1) * 8, in.U_lqr + (long long)k * 3, in.Bt, in.B_rows,
                           in.index_scale, in.clock_rate, h, AB);
    }
    tvlqr_riccati_step(o, ab, S, K + (long long)k * 18);
  }
}

// Stage record s of step k when it is not pre-generated (tcl_s: the stage's clock value): field row -> noise -> record.
// DISP: the row goes through the realisation's field transform (tvlqr_disp_field) before the noise is added.
template <bool DISP = false>
TS_HD void tvlqr_stage_record_at(const TvlqrIn& in, const ts_tvlqr_opts_dev& o, long long k, int s, double tcl_s, double rec[TV_REC]) {
  const double* Bn = in.Bt + (long long)field_row(tcl_s, in.index_scale, in.B_rows) * 3;
  double Bd[3];
  if constexpr (DISP) {
    tvlqr_disp_field(in.disp, Bn, Bd);
    Bn = Bd;
  }
  if (o.noise_mode == 2) {   // (its own call: the draws stay in registers, no pointer may alias them)
    double nzb[9];
    tvlqr_noise(o.seed, in.trial, (uint32_t)k, (uint32_t)s, nzb, in.real);
    tvlqr_stage_record(nzb, Bn, rec);
  } else {
    tvlqr_stage_record(o.noise_mode == 1 ? in.noise + (k * 4 + s) * 9 : nullptr, Bn, rec);
  }
}

// The replay's initial state (TortoiseSat.jl:227-234): omega from x0, attitude x0's perturbed by the rotation of q_noise
// (qn, nullable; a zero row = no perturbation: the reference's r_noise = q_noise/0 would be NaN), clock 0.  Built so by
// ts_monte_carlo_run from q_noise0 and by the disturbance ensemble (K4e) from its initial draw.
TS_HD void tvlqr_x0_lqr(const double* x0, const double* qn, double xl[8]) {
  for (int i = 0; i < 3; ++i) xl[i] = x0[i];
  const double* q0 = x0 + 3;
  bool rotated = false;
  if (qn) {
    const double th = sqrt(qn[0] * qn[0] + qn[1] * qn[1] + qn[2] * qn[2]);
    if (th > 1e-300) {
      const double sh = sin(th / 2);
      const double qp[4] = {cos(th / 2), qn[0] / th * sh, qn[1] / th * sh, qn[2] / th * sh};
      qmult(q0, qp, xl + 3);
      rotated = true;
    }
  }
  if (!rotated)
    for (int i = 0; i < 4; ++i) xl[3 + i] = q0[i];
  xl[7] = 0.0;
}

// Closed-loop replay + slew-time detection.  Outputs nullable.  Returns N_sim; *slew_time_out as
// monte_carlo.jl:237-262 (== t_final when the trial "fails").  recs: pre-generated stage records (40 doubles per step,
// K4n) or null -> built on the fly.  The slew-time rule is evaluated without sqrt / acos: |w| < w_limit is w.w < w_limit^2
// and 2 acos(min(q_e1,1)) < ang_limit is q_e1 > cos(ang_limit/2) (acos is decreasing; identical decisions except within one
// rounding of the thresholds).
// Where the replay reads the per-step inputs from (reference state 8, gain 18, reference control 3, stage records 40 if
// pre-generated):
// straight from the arrays (host twin, unit entries), or from a per-thread staging ring filled ahead of the sequential
// loop by asynchronous copies (K4c, k4_tvlqr.cuh), or from a per-warp ring when the 32 lanes replay the same slew under
// 32 noise draws (K4e).  x_last (nullable): the state at the last simulated step, X_sim row N_sim - 1.
struct TvlqrDirectSrc {
  const double *X, *U, *K, *recs;
  TS_HD void fetch(long long k, const double*& xr, const double*& Kk, const double*& ul, const double*& rk) const {
    xr = X + k * 8;
    Kk = K + k * 18;
    ul = U + k * 3;
    rk = recs ? recs + k * (4 * TV_REC) : nullptr;
  }
  TS_HD void done(long long) const {}
};
// DISP: a dispersed realisation (in.disp; in.I holds its truth inertia): transformed field rows when the records are
// built here, and the scaled torque in every stage.  CLAMP: the torquer limit of a weight-sweep ensemble (WE4 of DESIGN.md
// section 4, K4): each component of u = U_lqr - K dx is clamped to [-u_lim, u_lim] before it drives the step (a NaN
// stays NaN); the gains are unchanged.
template <bool PRE, class Src, bool DISP = false, bool CLAMP = false>
TS_HD long long tvlqr_replay_src(const TvlqrIn& in, const ts_tvlqr_opts_dev& o, Src& src, double* X_sim, double* U_sim,
                                 double* dX, double* slew_time_out, double* x_last = nullptr, double u_lim = 0.0) {
  const int N = in.N;
  long long N_sim = range_len(o.t0, o.dt, o.tf);
  if (N_sim > N) N_sim = range_len(o.t0, o.dt, o.tf - o.dt);
  if (N_sim > N) N_sim = N;
  double x[8];
  for (int i = 0; i < 8; ++i) x[i] = in.x0[i];
  double slew = in.t_final;
  const double qi[4] = {in.q_final[0], -in.q_final[1], -in.q_final[2], -in.q_final[3]};
  const double w2_limit = o.w_limit * o.w_limit;
  const double cos_limit = cos(o.ang_limit / 2);
  // literal post-processing reads omega of column = trial index (quirk Q12): that column is only
  // known once the replay has reached it, so the literal mode evaluates the rule in a second pass.
  for (long long k = 0; k < N_sim; ++k) {
    if (X_sim)
      for (int i = 0; i < 8; ++i) X_sim[k * 8 + i] = x[i];
    if (!o.literal_postproc) {
      const long long j = k + 1;
      const double w2 = x[0] * x[0] + x[1] * x[1] + x[2] * x[2];
      const double qe0 = qi[0] * x[3] - (qi[1] * x[4] + qi[2] * x[5] + qi[3] * x[6]);   // scalar part of qmult(q_inv(q_final), q)
      if (j > 10 && w2 < w2_limit && qe0 > cos_limit && slew == in.t_final) slew = in.time_step * (double)j;
    }
    if (k == N_sim - 1) {
      if (x_last)
        for (int i = 0; i < 8; ++i) x_last[i] = x[i];
      if (U_sim) U_sim[k * 3 + 0] = U_sim[k * 3 + 1] = U_sim[k * 3 + 2] = 0.0;
      if (dX)
        for (int i = 0; i < 6; ++i) dX[k * 6 + i] = 0.0;
      break;
    }
    const double *xr, *Kk, *ul, *rk_src;
    src.fetch(k, xr, Kk, ul, rk_src);
    double d6[6], u[3];
    for (int i = 0; i < 3; ++i) d6[i] = x[i] - xr[i];
    {
      const double qri[4] = {xr[3], -xr[4], -xr[5], -xr[6]};
      double qe[4];
      qmult(qri, x + 3, qe);
      d6[3] = qe[1];
      d6[4] = qe[2];
      d6[5] = qe[3];
    }
    for (int i = 0; i < 3; ++i) {
      double s = 0.0;
      for (int j = 0; j < 6; ++j) s += Kk[i * 6 + j] * d6[j];
      u[i] = ul[i] - s;
    }
    if constexpr (CLAMP)
      for (int i = 0; i < 3; ++i) u[i] = u[i] < -u_lim ? -u_lim : (u[i] > u_lim ? u_lim : u[i]);
    if (U_sim)
      for (int i = 0; i < 3; ++i) U_sim[k * 3 + i] = u[i];
    if (dX)
      for (int i = 0; i < 6; ++i) dX[k * 6 + i] = d6[i];
    // rk4(simulator) with per-stage records
    double tcl[4], nxt;
    clock_rk4(x[7], in.clock_rate, o.dt, tcl, nxt);
    // stage record s: pre-generated, or built right before its stage (10 live doubles rather than a step's 40)
    double rbuf[TV_REC];
    auto rec = [&](int s) -> const double* {
      if constexpr (PRE) {
        return rk_src + s * TV_REC;
      } else {
        tvlqr_stage_record_at<DISP>(in, o, k, s, tcl[s], rbuf);
        return rbuf;
      }
    };
    double k1[7], k2[7], k3[7], k4[7], xs[7];
    simulator7_rec<DISP>(in.I, x, u, rec(0), k1, &in.disp);
    for (int i = 0; i < 7; ++i) k1[i] = k1[i] * o.dt;
    for (int i = 0; i < 7; ++i) xs[i] = x[i] + k1[i] / 2.0;
    simulator7_rec<DISP>(in.I, xs, u, rec(1), k2, &in.disp);
    for (int i = 0; i < 7; ++i) k2[i] = k2[i] * o.dt;
    for (int i = 0; i < 7; ++i) xs[i] = x[i] + k2[i] / 2.0;
    simulator7_rec<DISP>(in.I, xs, u, rec(2), k3, &in.disp);
    for (int i = 0; i < 7; ++i) k3[i] = k3[i] * o.dt;
    for (int i = 0; i < 7; ++i) xs[i] = x[i] + k3[i];
    simulator7_rec<DISP>(in.I, xs, u, rec(3), k4, &in.disp);
    for (int i = 0; i < 7; ++i) k4[i] = k4[i] * o.dt;
    for (int i = 0; i < 7; ++i) x[i] = x[i] + (k1[i] + 2.0 * k2[i] + 2.0 * k3[i] + k4[i]) * TS_SIXTH;
    x[7] = nxt;
    src.done(k);
  }
  if (o.literal_postproc && X_sim) {
    for (long long j = 1; j <= N_sim; ++j) {
      long long col = in.trial_index_1based;
      if (col > N_sim) col = N_sim;
      const double* w = X_sim + (col - 1) * 8;
      const double wn = sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
      double qe[4];
      qmult(qi, X_sim + (j - 1) * 8 + 3, qe);
      const double ang = 2 * acos(fmin(qe[0], 1.0));
      if (j > 10 && wn < o.w_limit && ang < o.ang_limit && slew == in.t_final) slew = in.time_step * (double)j;
    }
  }
  if (slew_time_out) *slew_time_out = slew;
  return N_sim;
}
template <bool PRE>
TS_HD long long tvlqr_replay_t(const TvlqrIn& in, const ts_tvlqr_opts_dev& o, const double* K, double* X_sim, double* U_sim,
                               double* dX, double* slew_time_out, const double* recs) {
  TvlqrDirectSrc src = {in.X_lqr, in.U_lqr, K, recs};
  return tvlqr_replay_src<PRE>(in, o, src, X_sim, U_sim, dX, slew_time_out);
}
TS_HD long long tvlqr_replay(const TvlqrIn& in, const ts_tvlqr_opts_dev& o, const double* K, double* X_sim, double* U_sim,
                             double* dX, double* slew_time_out) {
  return tvlqr_replay_t<false>(in, o, K, X_sim, U_sim, dX, slew_time_out, nullptr);
}

}  // namespace ts
