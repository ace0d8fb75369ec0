// C exports of the oracle continuation (orc_alilqr_state.hpp): test infrastructure, built by tests/alilqr_state.py.
// The oracle's translation unit is included for its option-block conversion and problem set-up.
#include "../../oracle/oracle.cpp"
#include "orc_alilqr_state.hpp"

extern "C" {
// orc_alilqr_solve_batch's arguments in the same order, plus the state in and out (ts_alilqr_solve_state_batch)
void orc_alilqr_solve_state_batch(int64_t n_trials, const int64_t* N_i, const int64_t* offs, const double* x0, const double* xf,
                                  const double* Jmat, const double* Qd, const double* Qfd, const double* Rd, const double* B_eci,
                                  const int64_t* B_offs, const int64_t* B_rows, const double* index_scale, const double* clock_rate,
                                  double dt, const double* U0, const orc_ilqr_opts* opts, double* X, double* U, double* K,
                                  IlqrOutcome* out, int nthreads, const AlState* state_in, const double* lam_in, AlState* state_out,
                                  double* lam_out) {
  const IlqrOpts o = make_opts(opts);
  if (nthreads < 1) nthreads = 1;
#pragma omp parallel for num_threads(nthreads) schedule(dynamic, 1)
  for (int64_t t = 0; t < n_trials; ++t) {
    IlqrProblem p;
    p.N = N_i[t];
    p.dt = dt;
    for (int i = 0; i < 8; ++i) {
      p.x0[i] = x0[t * 8 + i];
      p.xf[i] = xf[t * 8 + i];
      p.Qd[i] = Qd[t * 8 + i];
      p.Qfd[i] = Qfd[t * 8 + i];
    }
    for (int i = 0; i < 3; ++i) p.Rd[i] = Rd[t * 3 + i];
    p.dyn.B_eci = B_eci + B_offs[t] * 3;
    p.dyn.B_rows = B_rows[t];
    p.dyn.index_scale = index_scale[t];
    p.dyn.clock_rate = clock_rate[t];
    for (int i = 0; i < 9; ++i) p.dyn.J[i] = Jmat[t * 9 + i];
    inv3(p.dyn.J, p.dyn.Jinv);
    alilqr_solve_state(p, o, U0 ? U0 + offs[t] * 3 : nullptr, X + offs[t] * 8, U + offs[t] * 3, K ? K + offs[t] * 24 : nullptr,
                       &out[t], state_in ? &state_in[t] : nullptr, lam_in ? lam_in + offs[t] * 6 : nullptr,
                       state_out ? &state_out[t] : nullptr, lam_out ? lam_out + offs[t] * 6 : nullptr);
  }
}
}
