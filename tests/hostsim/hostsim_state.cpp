// HOST LANE-EMULATOR, continuation pair -- TEST INFRASTRUCTURE ONLY.
// The emulator of hostsim.cpp plus an export / import pair around the team solver: a solve that returns the trial's
// state (solve_export, CS1) and bound multipliers, and a solve that starts from them (solve_import, CS3) -- the code
// the K3 kernels run to finish a trial and to resume one (k3_store_results, park_import_kernel).  Built into its own
// library by tests/alilqr_state.py.
#include "hostsim.cpp"

template <int W_, class TeamT = CpuTeamT<W_>>
static void solve_state_with_width(const TrialIn& in, const ts_ilqr_opts_dev* opts, int64_t N, double* X, double* U, double* K,
                                   ts_trial_outcome_dev* out, const ts_al_state_dev* sin, const double* lam_in,
                                   ts_al_state_dev* sout, double* lam_out) {
  const size_t per_slot = (size_t)9 * N * 10;
  std::vector<double> xu(4 * per_slot), kd((size_t)N * 24), lam((size_t)N * 6), clk((size_t)N), bk((size_t)N * 10);
  TrialWork w;
  w.xu = xu.data();
  w.xu_warp = xu.data();
  w.slot_stride = (long long)per_slot;
  w.kd = kd.data();
  w.lam = lam.data();
  w.clk = clk.data();
  w.bk = bk.data();
  w.Nmax = N;
  if (sin)   // the imported trajectory and multipliers, where park_import_kernel puts them (buffer 0, w.lam)
    for (int64_t k = 0; k < N; ++k) {
      for (int i = 0; i < 7; ++i) xu[k * 10 + i] = X[k * 8 + i];
      for (int i = 0; i < 3; ++i) xu[k * 10 + 7 + i] = (k < N - 1) ? U[k * 3 + i] : 0.0;
      for (int i = 0; i < 6; ++i) lam[k * 6 + i] = (k < N - 1) ? lam_in[k * 6 + i] : 0.0;
    }
  TeamSharedT<W_> sh;
  ts_trial_outcome_dev oc[W_];
  ts_al_state_dev so[W_];
  int cur[W_];
  std::vector<std::thread> th;
  for (int l = 0; l < W_; ++l)
    th.emplace_back([&, l]() {
      TeamT tm;
      tm.sh = &sh;
      tm.ln = l;
      TrialState st;
      if (sin)
        solve_import(tm, in, *opts, w, *sin, st);
      else
        solve_init(tm, in, *opts, w, st);
      while (st.phase != PH_DONE) {
        if (st.phase == PH_BACKWARD) solve_backward(tm, in, *opts, w, st);
        while (st.phase == PH_FORWARD) solve_forward(tm, in, *opts, w, st);
      }
      solve_finish(in, st, oc[l]);
      solve_export(st, so[l]);
      cur[l] = st.cur;
      tm.sync();
    });
  for (auto& t : th) t.join();
  *out = oc[0];
  *sout = so[0];
  const double* x = xu_buf<W_>(w, cur[0]);
  for (int64_t k = 0; k < N; ++k) {
    for (int i = 0; i < 7; ++i) X[k * 8 + i] = x[k * 10 + i];
    X[k * 8 + 7] = clk[k];
    for (int i = 0; i < 6; ++i) lam_out[k * 6 + i] = (k < N - 1) ? lam[k * 6 + i] : 0.0;
    if (k < N - 1) {
      for (int i = 0; i < 3; ++i) U[k * 3 + i] = x[k * 10 + 7 + i];
      if (K)
        for (int i = 0; i < 3; ++i) {
          for (int j = 0; j < 7; ++j) K[k * 24 + i * 8 + j] = kd[k * 24 + j * 3 + i];
          K[k * 24 + i * 8 + 7] = 0.0;
        }
    }
  }
}

extern "C" {
// hs_alilqr_solve_w with the state out (state_in == NULL: a fresh solve) or in and out.  A trial that does not
// continue (CS2) passes through: X, U, K untouched, outcome rebuilt from the state, state and lam copied.
void hs_alilqr_solve_state_w(int width, int64_t N, const double* x0, const double* xf, const double* Jmat, const double* Qd,
                             const double* Qfd, const double* Rd, const double* B_eci, int64_t B_rows, double index_scale,
                             double clock_rate, double dt, const double* U0, const ts_ilqr_opts_dev* opts, double* X, double* U,
                             double* K, ts_trial_outcome_dev* out, const ts_al_state_dev* state_in, const double* lam_in,
                             ts_al_state_dev* state_out, double* lam_out) {
  if (state_in && !(state_in->status == ST_MAX_OUTER && state_in->outer_iters < opts->max_outer)) {
    *out = ts_trial_outcome_dev{state_in->status, state_in->outer_iters, state_in->inner_iters, state_in->ls_rollouts, N,
                                state_in->J, state_in->c_max, 0.0, 0.0, 0.0};
    *state_out = *state_in;
    for (int64_t i = 0; i < N * 6; ++i) lam_out[i] = lam_in[i];
    return;
  }
  TrialIn in;
  in.N = (int)N;
  in.dt = dt;
  for (int i = 0; i < 7; ++i) in.x0[i] = x0[i];
  in.clk0 = x0[7];
  for (int i = 0; i < 8; ++i) {
    in.xf[i] = xf[i];
    in.Qd[i] = Qd[i];
    in.Qfd[i] = Qfd[i];
  }
  for (int i = 0; i < 3; ++i) in.Rd[i] = Rd[i];
  memcpy(in.I.J, Jmat, 72);
  inv3_gj(in.I.J, in.I.Jinv);
  in.Bt = B_eci;
  in.B_rows = B_rows;
  in.index_scale = index_scale;
  in.clock_rate = clock_rate;
  in.U0 = U0;
  if (opts->quat_error && width == 32)
    solve_state_with_width<32, CpuQuatTeamT<32>>(in, opts, N, X, U, K, out, state_in, lam_in, state_out, lam_out);
  else if (opts->quat_error)
    solve_state_with_width<8, CpuQuatTeamT<8>>(in, opts, N, X, U, K, out, state_in, lam_in, state_out, lam_out);
  else if (width == 32)
    solve_state_with_width<32>(in, opts, N, X, U, K, out, state_in, lam_in, state_out, lam_out);
  else
    solve_state_with_width<8>(in, opts, N, X, U, K, out, state_in, lam_in, state_out, lam_out);
}
}
