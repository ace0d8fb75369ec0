// HOST BUILD OF THE DISPERSION-ENSEMBLE DRAWS AND REPLAY -- TEST INFRASTRUCTURE ONLY.
// The K4 source (tvlqr_solver.cuh, philox.cuh) compiled for the CPU with the entry points the dispersion tests need: the
// ten truth-model parameters of realisation r (dispersion_params, DE2) and one dispersed realisation's replay (nominal
// gains, then tvlqr_replay_src<..., DISP = true> with the truth inertia, torquer gains and field transform of the given
// parameters), the code K4d runs per lane.  Built into its own library by tests/dispersion_ref.py.
#include <cstdint>
#include <cstring>

#include "../../tortoisesat.jl_b200/csrc/ilqr_solver.cuh"
#include "../../tortoisesat.jl_b200/csrc/tvlqr_solver.cuh"

using namespace ts;

extern "C" {

void hsd_dispersion_params(uint64_t seed, uint32_t stream, uint32_t real, const double* sig4, double* out10) {
  dispersion_params(seed, stream, real, sig4, out10);
}

// One dispersed realisation of one slew from x0 (the caller builds it for r >= 1) under the parameters prm (10, in the
// order of dispersion_params): gains of the nominal Jmat, replay with the truth model and the stage draws of realisation
// `real`.  Returns N_sim.
int64_t hsd_tvlqr_disp_real(int64_t N, const double* X_lqr, const double* U_lqr, const double* x0, const double* Jmat, const double* B_eci,
                            int64_t B_rows, double index_scale, double clock_rate, double t_final, const double* q_final, uint32_t trial,
                            uint32_t real, const double* prm, const ts_tvlqr_opts_dev* opts, double* X_sim, double* K, double* x_last,
                            double* slew_time) {
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
  tvlqr_gains(in, o, K);   // the nominal model
  tvlqr_disp_setup(prm, in.I.J, in.disp);
  inv3_gj(in.I.J, in.I.Jinv);
  TvlqrDirectSrc src = {in.X_lqr, in.U_lqr, K, nullptr};
  return tvlqr_replay_src<false, TvlqrDirectSrc, true>(in, o, src, X_sim, nullptr, nullptr, slew_time, x_last);
}

}  // extern "C"
