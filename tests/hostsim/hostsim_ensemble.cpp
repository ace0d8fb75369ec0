// HOST BUILD OF THE DISTURBANCE-ENSEMBLE DRAWS -- TEST INFRASTRUCTURE ONLY.
// The K4 source (tvlqr_solver.cuh, philox.cuh) compiled for the CPU with the entry points the ensemble tests need: the
// stage draws of realisation r (tvlqr_noise), the initial attitude draw of realisation r >= 1 (tvlqr_initial_qnoise), the
// replay's initial state (tvlqr_x0_lqr) and one realisation's replay (gains + tvlqr_replay with TvlqrIn::real = r), the
// code K4e runs per lane (RE2, DESIGN.md section 4, K4).  Built into its own library by tests/test_replay_ensemble.py.
#include <cstdint>
#include <cstring>

#include "../../tortoisesat.jl_b200/csrc/ilqr_solver.cuh"
#include "../../tortoisesat.jl_b200/csrc/tvlqr_solver.cuh"

using namespace ts;

extern "C" {

void hse_tvlqr_noise(uint64_t seed, uint32_t trial, uint32_t step, uint32_t stage, uint32_t real, double* out9) {
  tvlqr_noise(seed, trial, step, stage, out9, real);
}
void hse_initial_qnoise(uint64_t seed, uint32_t trial, uint32_t real, double scale, double* qn3) {
  tvlqr_initial_qnoise(seed, trial, real, scale, qn3);
}
void hse_x0_lqr(const double* x0, const double* qn, double* xl) { tvlqr_x0_lqr(x0, qn, xl); }

// One realisation of one slew: gains + replay + slew-time rule, starting from x0 (the caller builds it for r >= 1).
int64_t hse_tvlqr_real(int64_t N, const double* X_lqr, const double* U_lqr, const double* x0, const double* Jmat, const double* B_eci,
                       int64_t B_rows, double index_scale, double clock_rate, double t_final, const double* q_final, uint32_t trial,
                       uint32_t real, const ts_tvlqr_opts_dev* opts, double* X_sim, double* K, double* x_last, double* slew_time) {
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
  tvlqr_gains(in, o, K);
  TvlqrDirectSrc src = {in.X_lqr, in.U_lqr, K, nullptr};
  return tvlqr_replay_src<false>(in, o, src, X_sim, nullptr, nullptr, slew_time, x_last);
}

}  // extern "C"
