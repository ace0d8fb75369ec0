// FLOP counter (TEST / MEASUREMENT INFRASTRUCTURE -- never linked into the product).
//
// SURVEY.md section 8(d) asks for the algorithmic FLOP figures of the roofline to be COUNTED, not estimated: this tool
// re-compiles (a) the CPU oracle's AL-iLQR (oracle/orc_ilqr.hpp: the literal reference algorithm -- dense 8-state model,
// forward-mode dual numbers with 11 seeds like ForwardDiff, dense Riccati) and (b) the lane-local math of the CUDA
// kernels (csrc/ilqr_math.cuh, ilqr_solver.cuh: 7-state model, analytic JVP linearisation) with `double` replaced by a
// counting scalar, runs each per-knot unit once on a real slew, and prints the counts (add/sub/mul = 1, FMA = 2 because
// it is counted as its mul and its add; div, sqrt counted separately and also at 1 FLOP each in the totals).
//
//   g++ -O1 -std=c++17 -I oracle -I tortoisesat.jl_b200/csrc -o /tmp/flopcount tools/flopcount.cpp && /tmp/flopcount
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <math.h>
#include <vector>

struct Counters {
  long long add = 0, mul = 0, div = 0, sqrt_ = 0, cmp = 0;
  long long flops() const { return add + mul + div + sqrt_; }
};
static Counters g_cnt;

struct CD {
  double v;
  CD() : v(0.0) {}
  CD(double x) : v(x) {}
  CD(int x) : v((double)x) {}
  CD(long x) : v((double)x) {}
  CD(long long x) : v((double)x) {}
  CD(unsigned x) : v((double)x) {}
  explicit operator long long() const { return (long long)v; }
  explicit operator long() const { return (long)v; }
  explicit operator int() const { return (int)v; }
  explicit operator bool() const { return v != 0.0; }
  CD& operator+=(const CD& o) { ++g_cnt.add; v += o.v; return *this; }
  CD& operator-=(const CD& o) { ++g_cnt.add; v -= o.v; return *this; }
  CD& operator*=(const CD& o) { ++g_cnt.mul; v *= o.v; return *this; }
  CD& operator/=(const CD& o) { ++g_cnt.div; v /= o.v; return *this; }
};
inline CD operator+(const CD& a, const CD& b) { ++g_cnt.add; return CD(a.v + b.v); }
inline CD operator-(const CD& a, const CD& b) { ++g_cnt.add; return CD(a.v - b.v); }
inline CD operator*(const CD& a, const CD& b) { ++g_cnt.mul; return CD(a.v * b.v); }
inline CD operator/(const CD& a, const CD& b) { ++g_cnt.div; return CD(a.v / b.v); }
inline CD operator-(const CD& a) { return CD(-a.v); }
inline CD operator+(const CD& a) { return a; }
#define CD_CMP(op) inline bool operator op(const CD& a, const CD& b) { ++g_cnt.cmp; return a.v op b.v; }
CD_CMP(<) CD_CMP(>) CD_CMP(<=) CD_CMP(>=) CD_CMP(==) CD_CMP(!=)
// (templates: the non-template std:: overloads below win where a `using std::sqrt` makes both visible)
#include <type_traits>
#define CD_ONLY template <class T, class = std::enable_if_t<std::is_same<T, CD>::value>>
CD_ONLY inline CD sqrt(const T& a) { ++g_cnt.sqrt_; return CD(::sqrt(a.v)); }
CD_ONLY inline CD fabs(const T& a) { return CD(::fabs(a.v)); }
CD_ONLY inline CD floor(const T& a) { return CD(::floor(a.v)); }
CD_ONLY inline CD sin(const T& a) { return CD(::sin(a.v)); }
CD_ONLY inline CD cos(const T& a) { return CD(::cos(a.v)); }
CD_ONLY inline CD acos(const T& a) { return CD(::acos(a.v)); }
CD_ONLY inline CD log(const T& a) { return CD(::log(a.v)); }
inline CD fmax(const CD& a, const CD& b) { ++g_cnt.cmp; return CD(::fmax(a.v, b.v)); }
inline CD fmin(const CD& a, const CD& b) { ++g_cnt.cmp; return CD(::fmin(a.v, b.v)); }
namespace std {
inline CD sqrt(const CD& a) { ++g_cnt.sqrt_; return CD(::sqrt(a.v)); }
inline CD fabs(const CD& a) { return CD(::fabs(a.v)); }
inline CD floor(const CD& a) { return CD(::floor(a.v)); }
inline CD sin(const CD& a) { return CD(::sin(a.v)); }
inline CD cos(const CD& a) { return CD(::cos(a.v)); }
inline CD log(const CD& a) { return CD(::log(a.v)); }
inline CD max(const CD& a, const CD& b) { ++g_cnt.cmp; return a.v < b.v ? b : a; }
inline CD min(const CD& a, const CD& b) { ++g_cnt.cmp; return b.v < a.v ? b : a; }
}  // namespace std

// ---- everything below sees `double` as the counting scalar
#define double CD
#define volatile
#include "orc_ilqr.hpp"          // (a) the oracle: literal reference algorithm
#include "ilqr_solver.cuh"       // (b) the kernels' lane-local math (host build)
#include "tvlqr_solver.cuh"      // (c) the TVLQR replay step with its inline draws (the disturbance ensemble, K4e)
#undef volatile
#undef double

static Counters diff(const Counters& a, const Counters& b) {
  Counters d;
  d.add = a.add - b.add; d.mul = a.mul - b.mul; d.div = a.div - b.div; d.sqrt_ = a.sqrt_ - b.sqrt_; d.cmp = a.cmp - b.cmp;
  return d;
}
static void show(const char* what, const Counters& c, double per) {
  printf("  %-58s add %8.1f  mul %8.1f  div %6.1f  sqrt %5.1f  => %9.1f FLOP\n", what, c.add / per, c.mul / per, c.div / per, c.sqrt_ / per,
         c.flops() / per);
}

int main() {
  using namespace orc;
  // a real problem shape: N knots on a synthetic field table, inertia 1U, saturating controls so that bounds are active
  const int N = 65;
  std::vector<CD> Bt(3 * 4 * N);
  for (size_t i = 0; i < Bt.size(); ++i) Bt[i] = CD(2e-5 * std::sin(0.37 * (double)i) + 1e-5);
  IlqrProblem p;
  p.N = N; p.dt = CD(0.2);
  const double x0[8] = {0.01, -0.02, 0.005, 0.8, 0.1, -0.5, 0.3, 0.0}, xf[8] = {0, 0, 0, 0.7071, 0.7071, 0, 0, 1};
  for (int i = 0; i < 8; ++i) { p.x0[i] = CD(x0[i]); p.xf[i] = CD(xf[i]); p.Qd[i] = CD(i < 3 ? 3e3 : (i < 7 ? 100.0 : 0.0)); p.Qfd[i] = p.Qd[i] * CD(10.0); }
  for (int i = 0; i < 3; ++i) p.Rd[i] = CD(2.0);
  p.dyn.B_eci = Bt.data(); p.dyn.B_rows = 4 * N; p.dyn.index_scale = CD((double)N); p.dyn.clock_rate = CD(1.0 / 2400.0);
  for (int i = 0; i < 9; ++i) p.dyn.J[i] = CD((i % 4 == 0) ? 0.00125 : 0.0);
  inv3(p.dyn.J, p.dyn.Jinv);
  IlqrOpts o;
  detail::Work w(N);
  for (auto& u : w.U) u = CD(1.3);
  for (auto& l : w.lam_b) l = CD(0.1);
  for (auto& m : w.mu_b) m = CD(10.0);
  for (int i = 0; i < 8; ++i) { w.lam_g[i] = CD(0.0); w.mu_g[i] = CD(10.0); p.x0[i] = CD(x0[i]); }
  for (int i = 0; i < 8; ++i) w.X[i] = p.x0[i];
  for (int k = 0; k < N - 1; ++k) detail::step(p, &w.X[k * 8], &w.U[k * 3], &w.X[(k + 1) * 8]);
  const double K = N - 1;
  printf("(a) oracle = literal reference algorithm (8-state, 11-seed forward-mode duals, dense Riccati), per knot:\n");
  Counters c0 = g_cnt;
  detail::jacobians(p, w);
  Counters c_jac = diff(g_cnt, c0); show("jacobians (ForwardDiff through rk3 o DerivFunction)", c_jac, K);
  c0 = g_cnt;
  detail::Reg reg; CD dV[2];
  detail::backward_pass(p, o, w, reg, dV);
  Counters c_bwd = diff(g_cnt, c0); show("backward_pass (cost expansion + Riccati step)", c_bwd, K);
  c0 = g_cnt;
  detail::rollout(p, o, w, CD(0.5));
  CD cm;
  (void)detail::al_cost(p, o, w, w.Xb.data(), w.Ub.data(), &cm);
  Counters c_roll = diff(g_cnt, c0); show("line-search rollout (feedback + rk3 + AL cost)", c_roll, K);
  const double orc_iter = (c_jac.flops() + c_bwd.flops()) / K, orc_roll = c_roll.flops() / K;

  printf("(b) kernel math (7-state, analytic JVP linearisation; what k3_* executes per knot, one lane's share where noted):\n");
  ts::TrialIn in;
  in.N = N; in.dt = CD(0.2);
  for (int i = 0; i < 7; ++i) in.x0[i] = CD(x0[i]);
  in.clk0 = CD(0.0);
  for (int i = 0; i < 8; ++i) { in.xf[i] = CD(xf[i]); in.Qd[i] = p.Qd[i]; in.Qfd[i] = p.Qfd[i]; }
  for (int i = 0; i < 3; ++i) in.Rd[i] = CD(2.0);
  for (int i = 0; i < 9; ++i) { in.I.J[i] = p.dyn.J[i]; in.I.Jinv[i] = p.dyn.Jinv[i]; }
  ts_ilqr_opts_dev ko;
  memset((void*)&ko, 0, sizeof(ko));
  ko.u_max = CD(1.0); ko.u_min = CD(-1.0); ko.max_state_value = ko.max_control_value = CD(1e8);
  CD x[7], u[3] = {CD(1.3), CD(-0.4), CD(0.9)}, bk[10], lam[6], rec[ts::REC];
  for (int i = 0; i < 7; ++i) x[i] = CD(x0[i]);
  for (int i = 0; i < 10; ++i) bk[i] = CD(2e-5 * (i + 1));
  for (int i = 0; i < 6; ++i) lam[i] = CD(0.1 * i);
  c0 = g_cnt;
  ts::rk3_jac7_jvp(in.I, x, u, bk, bk + 3, bk + 6, in.dt, rec);
  Counters k_lin = diff(g_cnt, c0); show("linearisation: rk3_jac7_jvp (10 JVPs through 3 stages)", k_lin, 1);
  c0 = g_cnt;
  {  // stage-cost / AL gradient part of linearise_knot
    CD c6[6]; ts::bound_c(ko, u, c6);
    for (int i = 0; i < 7; ++i) rec[70 + i] = CD(1.0) * in.Qd[i] * (x[i] - in.xf[i]);
    for (int i = 0; i < 3; ++i) { CD lu = CD(1.0) * in.Rd[i] * u[i]; lu += (lam[i] + CD(10.0) * c6[i]) - (lam[3 + i] + CD(10.0) * c6[3 + i]); rec[77 + i] = lu; }
  }
  Counters k_grad = diff(g_cnt, c0); show("cost / AL gradients of the knot", k_grad, 1);
  // Riccati knot step, 7-state dense, in the arithmetic of the narrow team (summed over its lanes; the 3x3 factorisation once)
  c0 = g_cnt;
  {
    CD S[49], s7[7], AB[70], M[70], Qxx[49], Qux[21], Quu[9], Qx[7], Qu[3];
    for (int i = 0; i < 49; ++i) S[i] = CD(0.01 * (i % 7 + 1));
    for (int i = 0; i < 7; ++i) s7[i] = CD(0.1);
    for (int i = 0; i < 70; ++i) AB[i] = rec[i];
    for (int c = 0; c < 10; ++c) for (int i = 0; i < 7; ++i) { CD t(0.0); for (int l = 0; l < 7; ++l) t += S[i * 7 + l] * AB[c * 7 + l]; M[c * 7 + i] = t; }
    for (int j = 0; j < 7; ++j) for (int i = 0; i < 7; ++i) { CD t(0.0); for (int l = 0; l < 7; ++l) t += AB[i * 7 + l] * M[j * 7 + l]; Qxx[j * 7 + i] = t + in.Qd[i]; }
    for (int j = 0; j < 7; ++j) for (int c = 0; c < 3; ++c) { CD t(0.0); for (int l = 0; l < 7; ++l) t += AB[(7 + c) * 7 + l] * M[j * 7 + l]; Qux[j * 3 + c] = t; }
    for (int j = 0; j < 3; ++j) for (int c = 0; c < 3; ++c) { CD t(0.0); for (int l = 0; l < 7; ++l) t += AB[(7 + c) * 7 + l] * M[(7 + j) * 7 + l]; Quu[c * 3 + j] = t + CD(2.0); }
    for (int j = 0; j < 7; ++j) { CD t(0.0); for (int l = 0; l < 7; ++l) t += AB[j * 7 + l] * s7[l]; Qx[j] = rec[70 + j] + t; }
    for (int j = 0; j < 3; ++j) { CD t(0.0); for (int l = 0; l < 7; ++l) t += AB[(7 + j) * 7 + l] * s7[l]; Qu[j] = rec[77 + j] + t; }
    CD Qr[9], L[9], d[3], Quud[3], nb[3] = {-Qu[0], -Qu[1], -Qu[2]};
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) Qr[i * 3 + j] = CD(0.5) * (Quu[i * 3 + j] + Quu[j * 3 + i]) + CD(i == j ? 1e-3 : 0.0);
    ts::quu_factor(Qr, L);
    ts::quu_solve(L, nb, d);
    for (int i = 0; i < 3; ++i) Quud[i] = Quu[i * 3] * d[0] + Quu[i * 3 + 1] * d[1] + Quu[i * 3 + 2] * d[2];
    CD Kc[21], QuuK[21], dV1(0.0), dV2(0.0);
    for (int j = 0; j < 7; ++j) {
      CD b3[3] = {-Qux[j * 3], -Qux[j * 3 + 1], -Qux[j * 3 + 2]};
      ts::quu_solve(L, b3, Kc + j * 3);
      for (int i = 0; i < 3; ++i) QuuK[j * 3 + i] = Quu[i * 3] * Kc[j * 3] + Quu[i * 3 + 1] * Kc[j * 3 + 1] + Quu[i * 3 + 2] * Kc[j * 3 + 2];
    }
    for (int l = 0; l < 3; ++l) { dV1 += d[l] * Qu[l]; dV2 += CD(0.5) * d[l] * Quud[l]; }
    for (int j = 0; j < 7; ++j) {
      for (int i = 0; i < 7; ++i) { CD t = Qxx[j * 7 + i]; for (int l = 0; l < 3; ++l) t += Kc[i * 3 + l] * QuuK[j * 3 + l]; for (int l = 0; l < 3; ++l) t += Kc[i * 3 + l] * Qux[j * 3 + l]; for (int l = 0; l < 3; ++l) t += Qux[i * 3 + l] * Kc[j * 3 + l]; S[j * 7 + i] = t; }
      CD t = Qx[j]; for (int l = 0; l < 3; ++l) t += Kc[j * 3 + l] * Quud[l]; for (int l = 0; l < 3; ++l) t += Kc[j * 3 + l] * Qu[l]; for (int l = 0; l < 3; ++l) t += Qux[j * 3 + l] * d[l]; s7[j] = t;
    }
    for (int i = 0; i < 7; ++i) for (int j = i; j < 7; ++j) S[i * 7 + j] = CD(0.5) * (S[i * 7 + j] + S[j * 7 + i]);
  }
  Counters k_ric = diff(g_cnt, c0); show("Riccati knot step (dense 7-state, 3x3 cofactor solve once)", k_ric, 1);
  c0 = g_cnt;
  {  // one line-search rollout knot: feedback, AL stage cost, rk3 step (the divergence check is comparisons only)
    CD xb[7], ub[3], kd[24], dx[7], Jc(0.0), cmax(0.0), xn[7];
    for (int i = 0; i < 7; ++i) xb[i] = x[i] + CD(1e-3);
    for (int i = 0; i < 24; ++i) kd[i] = CD(0.01 * i);
    for (int i = 0; i < 7; ++i) dx[i] = xb[i] - x[i];
    for (int i = 0; i < 3; ++i) { CD t = u[i]; for (int j = 0; j < 7; ++j) t += kd[j * 3 + i] * dx[j]; t += CD(0.25) * kd[21 + i]; ub[i] = t; }
    ts::add_stage_cost(in, ko, CD(1.0), CD(10.0), xb, CD(0.0), ub, lam, Jc, cmax);
    ts::rk3_step7<0>(in.I, xb, ub, bk, bk + 3, bk + 6, in.dt, xn);
  }
  Counters k_roll = diff(g_cnt, c0); show("line-search rollout knot (feedback + AL cost + rk3)", k_roll, 1);
  // the same two units in the diagonal-inertia instantiation (every preset of input_parameters.jl; what the benchmark runs)
  c0 = g_cnt;
  ts::rk3_jac7_jvp<true>(in.I, x, u, bk, bk + 3, bk + 6, in.dt, rec);
  Counters k_lin_d = diff(g_cnt, c0); show("linearisation, diagonal inertia", k_lin_d, 1);
  c0 = g_cnt;
  {
    CD xb[7], ub[3], kd[24], dx[7], Jc(0.0), cmax(0.0), xn[7];
    for (int i = 0; i < 7; ++i) xb[i] = x[i] + CD(1e-3);
    for (int i = 0; i < 24; ++i) kd[i] = CD(0.01 * i);
    for (int i = 0; i < 7; ++i) dx[i] = xb[i] - x[i];
    for (int i = 0; i < 3; ++i) { CD t = u[i]; for (int j = 0; j < 7; ++j) t += kd[j * 3 + i] * dx[j]; t += CD(0.25) * kd[21 + i]; ub[i] = t; }
    ts::add_stage_cost(in, ko, CD(1.0), CD(10.0), xb, CD(0.0), ub, lam, Jc, cmax);
    ts::rk3_step7<0, true>(in.I, xb, ub, bk, bk + 3, bk + 6, in.dt, xn);
  }
  Counters k_roll_d = diff(g_cnt, c0); show("line-search rollout knot, diagonal inertia", k_roll_d, 1);
  // gradient measure of the convergence test: once per knot of the accepted trajectory (3 divisions, 3 additions)
  const long long k_gradm = 6;
  const double k_iter = (double)(k_lin.flops() + k_grad.flops() + k_ric.flops() + k_gradm), k_rollf = (double)k_roll.flops();
  const double k_iter_d = (double)(k_lin_d.flops() + k_grad.flops() + k_ric.flops() + k_gradm), k_rollf_d = (double)k_roll_d.flops();
  printf("\nsummary per knot-iteration / per rollout knot:  oracle (literal) %.0f / %.0f    kernel math %.0f / %.0f    diagonal inertia %.0f / %.0f\n",
         orc_iter, orc_roll, k_iter, k_rollf, k_iter_d, k_rollf_d);
  printf("JSON {\"per_knot_iteration\": %.0f, \"per_rollout_knot\": %.0f, \"per_knot_iteration_diag\": %.0f, \"per_rollout_knot_diag\": %.0f, "
         "\"linearise\": %lld, \"linearise_diag\": %lld, \"cost_gradients\": %lld, \"riccati\": %lld, \"gradient_measure\": %lld, "
         "\"oracle_per_knot_iteration\": %.0f, \"oracle_per_rollout_knot\": %.0f, \"oracle_jacobians\": %.0f, \"oracle_backward\": %.0f}\n",
         k_iter, k_rollf, k_iter_d, k_rollf_d, k_lin.flops(), k_lin_d.flops(), k_grad.flops(), k_ric.flops(), k_gradm, orc_iter, orc_roll,
         c_jac.flops() / K, c_bwd.flops() / K);
  // (c) one step of the replay with inline draws, as K4e runs it per lane: feedback, four stage records (Philox +
  // Box-Muller draws, perturbation quaternion, field row) and the rk4 step of the simulator.  Counted as the difference
  // of two replays of 65 and 33 knots over the 32 extra steps; log / sin / cos calls are not FLOPs in this count.
  auto replay = [&](int n) {
    std::vector<CD> Xr(8 * n), Ur(3 * n), Kr(18 * n);
    for (int k = 0; k < n; ++k) for (int i = 0; i < 8; ++i) Xr[k * 8 + i] = CD(x0[i]);
    for (int i = 0; i < 18 * n; ++i) Kr[i] = CD(0.01);
    ts::TvlqrIn ti;
    ti.N = n; ti.X_lqr = Xr.data(); ti.U_lqr = Ur.data();
    for (int i = 0; i < 8; ++i) ti.x0[i] = CD(x0[i]);
    for (int i = 0; i < 9; ++i) { ti.I.J[i] = p.dyn.J[i]; ti.I.Jinv[i] = p.dyn.Jinv[i]; }
    ti.Bt = Bt.data(); ti.B_rows = 4 * N; ti.index_scale = CD((double)N); ti.clock_rate = CD(1.0 / 2400.0);
    ti.noise = nullptr; ti.trial = 3; ti.real = 5;
    for (int i = 0; i < 4; ++i) ti.q_final[i] = CD(xf[3 + i]);
    ti.t_final = CD(0.2 * (n - 1)); ti.time_step = CD(0.2); ti.trial_index_1based = 4;
    ts_tvlqr_opts_dev to = {};
    to.dt = CD(0.2); to.t0 = CD(0.0); to.tf = ti.t_final; to.noise_mode = 2; to.seed = 7; to.w_limit = CD(0.05); to.ang_limit = CD(0.08727);
    CD slew(0.0);
    const Counters a = g_cnt;
    ts::tvlqr_replay(ti, to, Kr.data(), nullptr, nullptr, nullptr, &slew);
    return diff(g_cnt, a);
  };
  const Counters r65 = replay(65), r33 = replay(33);
  const Counters c_step = diff(r65, r33);
  c0 = g_cnt;
  { CD nz[9]; ts::tvlqr_noise(7, 3, 1, 2, nz, 5); }
  const Counters c_draw = diff(g_cnt, c0);
  printf("\n(c) TVLQR replay with inline draws (disturbance ensemble, K4e), per replay step:\n");
  show("replay step (feedback + 4 stage records with draws + rk4)", c_step, 32);
  show("draws of one stage (tvlqr_noise: 3 Philox blocks, 3 Box-Muller pairs, scaling)", c_draw, 1);
  printf("JSON {\"ensemble_replay_step\": %.0f, \"stage_draws\": %lld}\n", c_step.flops() / 32.0, c_draw.flops());
  return 0;
}
