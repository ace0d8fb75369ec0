// HOST BUILD OF THE WEIGHT-SWEEP ENSEMBLE REPLAY -- TEST INFRASTRUCTURE ONLY.
// The K4 source (tvlqr_solver.cuh) compiled for the CPU with the entry point the weight-sweep tests need: one dispersed
// realisation's replay under the gains of a given tracking weighting and an optional torquer limit (WE2, WE4 of
// DESIGN.md section 4, K4) -- the code K4w runs per lane: the Riccati sweep with the set's Qd, Qfd, Rd, then
// tvlqr_replay_src<..., DISP = true, CLAMP> with the truth model of the given parameters.  Built into its own library
// by tests/weight_ref.py.
#include <cstdint>
#include <cstring>

#include "../../tortoisesat.jl_b200/csrc/ilqr_solver.cuh"
#include "../../tortoisesat.jl_b200/csrc/tvlqr_solver.cuh"

using namespace ts;

extern "C" {

// w15: Qd 6 | Qfd 6 | Rd 3 (ts_tvlqr_weights); u_limit 0 = the replay without the clamp switch.  Returns N_sim.
int64_t hsw_tvlqr_weight_real(int64_t N, const double* X_lqr, const double* U_lqr, const double* x0, const double* Jmat,
                              const double* B_eci, int64_t B_rows, double index_scale, double clock_rate, double t_final,
                              const double* q_final, uint32_t trial, uint32_t real, const double* prm, const ts_tvlqr_opts_dev* opts,
                              const double* w15, double u_limit, double* X_sim, double* K, double* x_last, double* slew_time) {
  TvlqrIn in;
  in.N = (int)N;
  in.X_lqr = X_lqr;
  in.U_lqr = U_lqr;
  for (int i = 0; i < 8; ++i) in.x0[i] = x0[i];
  memcpy(in.I.J, Jmat, 72);
  inv3_gj(in.I.J, in.I.Jinv);
  in.Bt = B_eci;
  in.B_rows = B_rows;
  in.index_scale = index_scale;
  in.clock_rate = clock_rate;
  in.noise = nullptr;
  in.trial = trial;
  in.real = real;
  for (int i = 0; i < 4; ++i) in.q_final[i] = q_final[i];
  in.t_final = t_final;
  in.time_step = opts->dt;
  in.trial_index_1based = (long long)trial + 1;
  ts_tvlqr_opts_dev o = *opts;
  o.tf = t_final;
  memcpy(o.Qd, w15, 48);
  memcpy(o.Qfd, w15 + 6, 48);
  memcpy(o.Rd, w15 + 12, 24);
  tvlqr_gains(in, o, K);   // the nominal model, weighting w15
  tvlqr_disp_setup(prm, in.I.J, in.disp);
  inv3_gj(in.I.J, in.I.Jinv);
  TvlqrDirectSrc src = {in.X_lqr, in.U_lqr, K, nullptr};
  if (u_limit > 0.0) return tvlqr_replay_src<false, TvlqrDirectSrc, true, true>(in, o, src, X_sim, nullptr, nullptr, slew_time, x_last, u_limit);
  return tvlqr_replay_src<false, TvlqrDirectSrc, true>(in, o, src, X_sim, nullptr, nullptr, slew_time, x_last);
}

}  // extern "C"
