/* tortoise_b200.h -- C ABI of libtortoise_b200.so
 *
 * B200-native (sm_100a, FP64 CUDA cores) batched Monte-Carlo engine for the
 * data-parallel hot path of RoboticExplorationLab/TortoiseSat.jl: thousands of
 * independent magnetorquer slew trials.  The reference is a set of Julia
 * scripts with no FFI; every entry point below is what a Julia `ccall` (or the
 * Python ctypes host in tortoisesat.jl_b200/host.py) binds in place of the
 * reference function cited next to it.  See INTEGRATION.md for the bindings.
 *
 * Conventions
 *  - extern "C", plain pointers + sizes, all reals are FP64, all sizes int64_t.
 *  - return 0 = TS_OK, negative = error (message: ts_last_error()).  A failure of
 *    ONE trial is never a call failure: it is reported in
 *    ts_trial_outcome.status.
 *  - every data pointer is a HOST pointer unless the call has a
 *    `pointers_are_device` argument set to 1 (then all array arguments of that
 *    call are device pointers on the context's GPU; option structs stay host).
 *  - the caller owns its buffers for the duration of the (blocking) call; the
 *    library owns all device memory behind ts_ctx.  A ts_ctx is bound to one GPU
 *    and is not re-entrant.  There is NO CPU fallback: without a usable CUDA
 *    device ts_create() fails.
 *  - matrices are row-major "by sample / by knot": e.g. a field table is
 *    rows x 3, a state trajectory is N x 8 (Julia: declare them 3 x rows / 8 x N
 *    column-major and pass the array as is).
 */
#ifndef TORTOISE_B200_H
#define TORTOISE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TS_OK 0
#define TS_ERR_CUDA (-1)      /* CUDA runtime / launch failure */
#define TS_ERR_ARG (-2)       /* bad argument (null pointer, negative size, ...) */
#define TS_ERR_DATE (-3)      /* igrf12: date outside [1900, 2025]        (igrf.jl:80-81) */
#define TS_ERR_DOMAIN (-4)    /* igrf12: |lat| > pi/2 or |lon| > pi at >=1 point (igrf.jl:84-88);
                                 field map: a non-finite index at >=1 point;
                                 the offending outputs are NaN, the rest are valid */
#define TS_ERR_NOMEM (-5)

typedef struct ts_ctx ts_ctx;

/* ---- context -------------------------------------------------------------- */
int ts_create(ts_ctx** out, int device_id);
void ts_destroy(ts_ctx* ctx);
const char* ts_last_error(const ts_ctx* ctx); /* valid until the next call on ctx */
int ts_version(void);
/* multiprocessor count and name of the bound device */
int ts_device_info(ts_ctx* ctx, int* sm_count, char* name, int name_len);
/* number of kernels this context has launched since creation (bench bookkeeping) */
int64_t ts_launch_count(const ts_ctx* ctx);
/* wait for all work queued by this context */
int ts_synchronize(ts_ctx* ctx);
/* device time (ms, CUDA events on the context's stream) of the kernels launched by the
 * most recent call on ctx, excluding host<->device copies */
double ts_last_kernel_ms(const ts_ctx* ctx);
/* diagnostics of the most recent AL-iLQR solve on ctx (K3): device time of the persistent 4-trials-per-warp
 * kernel, of the straggler kernel (one warp per trial), and how many trials were handed from one to the other */
int ts_k3_last_split(ts_ctx* ctx, double* persistent_ms, double* straggler_ms, int64_t* n_parked);
/* per-trial SM-cycle counters of the most recent AL-iLQR solve on ctx (profiling aid; trial order of that call, or the
 * order of the trials that reached the solver in ts_monte_carlo_run): cycles3 = n_trials x 3 HOST doubles
 * [backward pass, forward pass (line search), linearisation share of the backward pass].                        */
int ts_k3_last_cycles(ts_ctx* ctx, int64_t n_trials, double* cycles3);
/* the trials the most recent AL-iLQR solve on ctx handed from the first to the second launch (profiling aid for the
 * hand-over order): for each, its index in that call's trial order and the outer / total inner iteration counters
 * it had when it was parked.  HOST arrays of `cap` entries; *n_out = entries written.                           */
int ts_k3_last_parked(ts_ctx* ctx, int64_t cap, int64_t* trial, int32_t* outer_at_park, int32_t* inner_at_park, int64_t* n_out);

/* Measures the FP64 FMA peak of the bound GPU with a register-resident DFMA
 * micro-benchmark (the roofline denominator; MEASURED_PEAKS.json has no FP64 row). */
int ts_fp64_peak_probe(ts_ctx* ctx, double* tflops_out);
/* Latency micro-benchmark of the bound GPU (one warp): cycles4 = SM cycles per DEPENDENT operation for
 * [DFMA, DADD/DMUL, rsqrt + DADD, shared-memory store -> __syncwarp -> load round trip] -- the quantities that bound
 * the strictly sequential Riccati / rollout chains of K3 (profiles/README.md).                                  */
int ts_fp64_latency_probe(ts_ctx* ctx, double* cycles4);

/* ---- K1: batched IGRF-12 --------------------------------------------------- *
 * Replaces igrf12(date, r, lat, lon) [src/igrf.jl:67-274] (+ legendre.jl:254-292,
 * dlegendre.jl:221-309) evaluated at n points -- e.g. the 10^6-point map of
 * igrf_data() [src/magnetic_toolbox.jl:108-121].  Geocentric: r in metres,
 * lat in [-pi/2, pi/2], lon in [-pi, pi] (rad).  Output north/east/down in nT.   */
int ts_igrf12_batch(ts_ctx* ctx, double date, int64_t n, const double* r_m, const double* lat, const double* lon,
                    double* Bn, double* Be, double* Bd, int pointers_are_device);

/* ---- K2: orbit + ECI field table + gramian cutoff --------------------------- *
 * One entry of ts_field_opts per trial (the reference keeps these in the `params`
 * struct / globals: p.GM, p.MJD, the hard-coded igrf date 2019 and the constant
 * field radius (alt+R_E)*1000 of src/magnetic_toolbox.jl:44,81).                   */
typedef struct ts_field_opts {
  double GM;             /* km^3/s^2                        (input_parameters.jl:26) */
  double mjd;            /* modified Julian day of t = 0    (input_parameters.jl:63) */
  double igrf_date;      /* year A.D. passed to igrf12      (magnetic_toolbox.jl:81: 2019) */
  double field_radius_m; /* radius passed to igrf12 [m]     (magnetic_toolbox.jl:81: (alt+R_E)*1000) */
  double t0, tf;         /* s; the orbit is propagated over [t0, 2 tf] with dt = (tf-t0)/N */
  int64_t N;             /* knot count; the table has 2N rows, pos/vel 2N+1 rows */
} ts_field_opts;

/* magnetic_simulation(p,t0,tf,N,mag_field) [src/magnetic_toolbox.jl:33-106] (which calls
 * kep_ECI [src/kep_ECI.jl:1-49] and Euler-integrates OrbitPlotter [src/OrbitPlotter.jl:1-52])
 * for n_trials trials.  kep6: n_trials x 6 = [e, a km, i deg, RAAN deg, argp deg, nu deg]
 * (NOT mutated, unlike kep_ECI.jl:7-8).  Ragged layout: trial t owns rows
 * [B_offs[t], B_offs[t]+2N_t) of B_eci (rows x 3, Tesla; last row 0 like the reference) and
 * rows [B_offs[t]+t, B_offs[t]+t+2N_t+1) of pos / vel (km, km/s; nullable).  B_offs has
 * n_trials+1 entries (host pointer).  rows_limit (host, nullable): if rows_limit[t] > 0 only
 * the first rows_limit[t] table rows are computed (the rest are 0) -- the solver only ever
 * reads rows <= floor(x8*N+1) (DerivFunction.jl:28, quirk Q1).                            */
int ts_magnetic_simulation_batch(ts_ctx* ctx, int64_t n_trials, const double* kep6, const ts_field_opts* opts,
                                 const int64_t* B_offs, const int64_t* rows_limit, double* B_eci, double* pos, double* vel,
                                 int pointers_are_device);

/* magnetic_gramian(B_N, dt) [src/magnetic_toolbox.jl:1-12]: G (rows x 9 per trial, row-major 3x3,
 * same row offsets as B_eci).  rows/dt: host arrays of n_trials.                           */
int ts_magnetic_gramian_batch(ts_ctx* ctx, int64_t n_trials, const double* B_eci, const int64_t* B_offs, const int64_t* rows,
                              const double* dt, double* G, int pointers_are_device);

/* condition_based_time(B_gram, cutoff) [src/magnetic_toolbox.jl:14-31]: first 1-based sample
 * whose gramian has cond_2 < cutoff, else 0.  tf_index: host array of n_trials.             */
int ts_condition_based_time_batch(ts_ctx* ctx, int64_t n_trials, const double* G, const int64_t* offs, const int64_t* rows,
                                  const double* cutoff, int64_t* tf_index, int pointers_are_device);

/* Fused magnetic_gramian + condition_based_time (no rows x 9 intermediate).               */
int ts_condition_cutoff_batch(ts_ctx* ctx, int64_t n_trials, const double* B_eci, const int64_t* B_offs, const int64_t* rows,
                              const double* dt, const double* cutoff, int64_t* tf_index, int pointers_are_device);

/* ---- K3: batched Augmented-Lagrangian iLQR ---------------------------------- *
 * Option block = the AugmentedLagrangianSolverOptions / iLQRSolverOptions fields of
 * TrajectoryOptimization.jl v0.1.2 that the reference sets or relies on
 * (src/TortoiseSat.jl:194-196: opts_uncon.iterations = 50, iterations = 20); semantics
 * frozen in SURVEY.md Appendix C (assumptions A1..A10).                             */
typedef struct ts_ilqr_opts {
  int32_t max_outer;        /* 20  opts_al.iterations                                  */
  int32_t max_inner;        /* 50  opts_al.opts_uncon.iterations                       */
  int32_t max_linesearch;   /* 20  iterations_linesearch                               */
  int32_t dJ_counter_limit; /* 10                                                      */
  int32_t stage_cost_dt;    /* 0   A1: 1 = stage cost and its expansion scaled by dt   */
  int32_t goal_mask;        /* 0x7F Q2: bit i = terminal equality on state i; 0xFF = literal
                                   goal_constraint(xf) incl. the infeasible clock state */
  double cost_tol, cost_tol_intermediate;   /* 1e-4, 1e-3 */
  double grad_tol, grad_tol_intermediate;   /* 1e-5, 1e-5 */
  double constraint_tol;                    /* 1e-3       */
  double penalty_initial, penalty_scaling, penalty_max, dual_max; /* 1, 10, 1e8, 1e8 */
  double ls_lower, ls_upper;                /* 1e-8, 10   */
  double bp_reg_increase, bp_reg_max, bp_reg_min, bp_reg_fp; /* 1.6, 1e8, 1e-8, 10 */
  double max_cost_value, max_state_value, max_control_value; /* 1e8 each */
  double u_max, u_min;      /* BoundConstraint(n,m,u_max=1,u_min=-1)  (TortoiseSat.jl:178) */
  /* Assumption registry (SURVEY.md App. C): TrajectoryOptimization.jl v0.1.2 is not in the reference tree, so every
   * choice its call sites do not pin is a named switch; 0 = the frozen default, 1 = the alternative reading.
   * tests/test_assumption_flips.py flips each one (oracle and kernel agree under every setting).            */
  int32_t a2_active_ge;           /* A2: inequality active when c >= 0 (default c > 0) or lambda > 0          */
  int32_t a3_grad_over_N;         /* A3: Todorov gradient averaged over N knots (default N-1 controls)         */
  int32_t a4_no_intermediate;     /* A4: final tolerances on every outer iteration (default: intermediate ones
                                         on all but the last)                                                 */
  int32_t a5_dual_active_only;    /* A5: dual update on active inequalities only (default: all, then max(0,.)) */
  int32_t a6_penalty_conditional; /* A6: penalty x scaling only if c_max > constraint_decrease_ratio x previous
                                         c_max (default: every outer iteration, every constraint)             */
  int32_t a7_carry_cost;          /* A7: J_prev of an inner solve = last cost under the OLD multipliers
                                         (default: re-evaluated with the new lambda, mu)                      */
  double constraint_decrease_ratio; /* 0.25 (only read when a6_penalty_conditional = 1)                       */
  /* K3 launch scheme (no effect on results): a trial is handed from the 4-trials-per-warp kernel to the
   * one-warp-per-trial kernel once it has used k3_suspend_after inner iterations of a mean-horizon trial and the
   * queue is empty (0 = never), or k3_early_factor x that while fresh trials are still queued (0 = never early);
   * k3_tail_share: finished teams lend their lanes to their warp's unfinished trials.                         */
  int32_t k3_suspend_after;       /* 150 */
  int32_t k3_tail_share;          /* 1   */
  double k3_early_factor;         /* 2.0 */
  int32_t k3_pair;                /* 2; 1: the one-warp-per-trial launch runs as k3_pair_kernel: 4 solver warps per SM, each
                                        with a producer warp (same SM sub-partition) that linearises the next 32-knot chunk
                                        while the solver runs the Riccati steps; 0: never; 2: when the ensemble's horizons
                                        are ragged (longest >= 2 x mean).  Same algorithm (last-bit differences from FMA
                                        contraction, like between the two default kernels).  Measured: slower on an
                                        equal-horizon ensemble (half the solver warps: 6.32 s vs 5.72 s), faster on the
                                        sweep, whose second launch is the chain of a few very long slews (13.4 s vs 16.2 s) */
  int32_t k3_wide_occ;            /* 0: as many one-warp blocks per SM as fit (8); n > 0: at most n.  Measured on the
                                        4096-trial ensemble: 8 -> 5.72 s, 6 -> 5.98 s, 4 -> 6.64 s, 2 -> 10.5 s            */
  int32_t quat_error;             /* 0; 1: the quaternion-aware variant the reference's Monte-Carlo script requests from its forked
                                        solver (monte_carlo.jl:158 Model(..., quaternion_error, quaternion_expansion), :192
                                        sat_att = true; hooks in quaternion_toolbox.jl:15-75): the feedback law uses
                                        dx = [w - wbar; MRP(conj(qbar) (x) q)], the backward pass runs on the 6-dim error
                                        state with A_e = E(x_k+1)' A E(x_k), B_e = E(x_k+1)' B, E = blkdiag(I3, G(q)).  Gains
                                        come back in error coordinates (3 x 8 rows, entries 6 and 7 zero).  Needs equal
                                        weights / goal mask on the four quaternion components.                           */
  int32_t k3_generic_inertia;     /* 0: when every trial's inertia matrix is diagonal (every preset of input_parameters.jl is) the
                                        solve runs the diagonal-inertia kernel instantiations (products with the exact zeros
                                        of J and J^-1 left out: the same values, 14 % fewer instructions per rollout knot);
                                        1: always the general kernels (A/B runs and the test that both give the same result) */
} ts_ilqr_opts;
void ts_ilqr_default_opts(ts_ilqr_opts* o);

/* per-trial status codes */
#define TS_ST_CONVERGED 0   /* c_max < constraint_tol                              */
#define TS_ST_MAX_OUTER 1   /* all outer iterations used                           */
#define TS_ST_COST_BLOWUP 2 /* J > max_cost_value (TrajOpt would error())          */
#define TS_ST_REG_MAX 3     /* backward-pass regularisation exceeded bp_reg_max    */
#define TS_ST_NAN 4
#define TS_ST_NO_CUTOFF 5   /* condition_based_time returned 0 (magnetic_toolbox.jl:23) */

/* 64-byte per-trial record (what the multi-GPU driver gathers) */
typedef struct ts_trial_outcome {
  int32_t status, outer_iters, inner_iters, ls_rollouts;
  int64_t N;
  double J, c_max, t_final, slew_time, flops;
} ts_trial_outcome;

/* solve!(Problem(rk3(Model(DerivFunction,8,3)), LQRObjective(Q,R,Qf,xf,N), constraints, x0, N, dt),
 *        AugmentedLagrangianSolver)  [src/TortoiseSat.jl:145-146,169,178-199] for n_trials trials.
 * HOST arrays, one entry (or row) per trial: N_i knots; offs[t] = first knot of trial t in the
 * ragged X/U/K arrays; x0, xf (8: omega, q scalar-first, clock); Jmat (3x3 row-major); Qd, Qfd
 * (8 diagonal weights), Rd (3); B_offs/B_rows = first row / row count of the trial's field
 * table inside B_eci; index_scale = the N of floor(Int,t*N+1) and clock_rate = 1/(tf-t0)
 * (DerivFunction.jl:28,44, quirk Q1).  dt is the knot spacing.
 * Arrays that follow pointers_are_device: B_eci (rows x 3), U0 (nullable -> zeros; ragged
 * (N-1) x 3 at offs*3), X (ragged N x 8 at offs*8), U (ragged (N-1) x 3 at offs*3), K (nullable;
 * ragged (N-1) x 3 x 8 at offs*24).  out: HOST array of n_trials records.                       */
int ts_alilqr_solve_batch(ts_ctx* ctx, int64_t n_trials, const int64_t* N_i, const int64_t* offs, const double* x0,
                          const double* xf, const double* Jmat, const double* Qd, const double* Qfd, const double* Rd,
                          const double* B_eci, const int64_t* B_offs, const int64_t* B_rows, const double* index_scale,
                          const double* clock_rate, double dt, const double* U0, const ts_ilqr_opts* opts, double* X,
                          double* U, double* K, ts_trial_outcome* out, int pointers_are_device);

/* ---- K3 continuation: export the solver state and continue max-outer trials from it ----------------------- *
 * The state of one finished trial (104 bytes).  The per-knot bound multipliers go alongside it in a ragged `lam`
 * array of (sum N) x 6 doubles at offs[t]*6 (the layout of U; the last row of each trial is unused and zero).  Rules
 * (DESIGN.md section 4, K3):
 *  CS1 export: the state is what the solver holds after its final outer update.  At a TS_ST_MAX_OUTER end the dual,
 *      goal-multiplier and penalty updates have been applied, so mu, lam_goal and lam are the values the next outer
 *      iteration would use.
 *  CS2 a trial continues when status == TS_ST_MAX_OUTER and outer_iters < opts->max_outer of the continuing call.
 *      Every other trial passes through: its X, U and K rows are not written, its outcome is rebuilt from the state
 *      (N from N_i, the rest of the record zero), its state and lam rows are copied to the outputs.
 *  CS3 a continuing trial resumes with the next outer iteration: outer_iters + 1, a fresh inner solve, J_prev = the
 *      cost of (X, U) under the imported multipliers (A7: the carried J), previous c_max = c_max.  The trajectory is
 *      imported from X (columns 0-6; the clock column is recomputed) and U, not rolled out again.  Counters and costs
 *      accumulate: a continued outcome reports totals over both calls.
 *  CS4 "solve to M1, then continue to M2" equals "solve to M2" exactly when cost_tol_intermediate == cost_tol and
 *      grad_tol_intermediate == grad_tol, or a4_no_intermediate = 1.  Otherwise outer iteration M1 ran with the final
 *      tolerances in the first call and would have run with the intermediate ones in a direct solve to M2: a slightly
 *      different, documented schedule (the defaults differ in cost_tol).
 * The continuing call's opts apply to the continuation (raise max_outer, change penalty_max, ...).  The call does not
 * check that X, U and lam come from the same solve as the state: that is the caller's contract.               */
typedef struct ts_al_state {
  double mu;           /* penalty after the last outer (dual + penalty) update                     */
  double lam_goal[8];  /* goal-constraint multipliers after that update                            */
  double J;            /* = ts_trial_outcome.J: cost at the last inner iteration (the A7 carry)    */
  double c_max;        /* = ts_trial_outcome.c_max: violation at the last outer update              */
  int32_t status, outer_iters, inner_iters, ls_rollouts;   /* as in ts_trial_outcome               */
} ts_al_state;

/* ts_alilqr_solve_batch with the state in and out.  state_in == NULL: a fresh solve, bit-identical to
 * ts_alilqr_solve_batch (which is this call with four NULLs).  state_in set: X and U are inputs for the continuing
 * trials (CS2) and outputs for all trials, and lam_in (required) holds the bound multipliers.  state_out (nullable)
 * receives every trial's state and lam_out (nullable) its multipliers.  lam_in, lam_out, X, U and K follow
 * pointers_are_device; state_in and state_out are HOST arrays of n_trials, like out.  A status outside 0-5 or
 * outer_iters < 1 in state_in, or state_in without lam_in, is TS_ERR_ARG and nothing is written.  The continuing
 * trials run on the one-warp-per-trial straggler kernels; TS_ERR_NOMEM (nothing written) if their parked records do not
 * fit in device memory.  ts_k3_last_split reports 0 ms for the persistent kernel and every continuing trial as handed over.   */
int ts_alilqr_solve_state_batch(ts_ctx* ctx, int64_t n_trials, const int64_t* N_i, const int64_t* offs, const double* x0,
                                const double* xf, const double* Jmat, const double* Qd, const double* Qfd, const double* Rd,
                                const double* B_eci, const int64_t* B_offs, const int64_t* B_rows, const double* index_scale,
                                const double* clock_rate, double dt, const double* U0, const ts_ilqr_opts* opts, double* X,
                                double* U, double* K, ts_trial_outcome* out, int pointers_are_device,
                                const ts_al_state* state_in, const double* lam_in, ts_al_state* state_out, double* lam_out);

/* ---- slew preparation: eigen-axis guess + Bryson weights ---------------------- *
 * eigen_axis_slew(x0,xf,t) [src/eigen_axis_slew.jl:1-38] over t = t0:dt:t_final[t], followed by
 * Bryson's rule [src/TortoiseSat.jl:157-168; alpha = 10 there, 0.1 in src/monte_carlo.jl:169;
 * beta = 1e3].  eigen_axis_fix = 0 reproduces eigen_axis_slew.jl:16 literally: `qmult([q2;-q2[2:4]],q1)` hands qmult
 * a 7-vector of which it reads entries 1 and 2:4, i.e. the error quaternion is qmult(q_f, q_0) WITHOUT the conjugate;
 * eigen_axis_fix = 1 uses conj(q_f) (x) q_0 (the evident intent; same theta_f whenever either attitude is the identity).
 * HOST arrays: x0, xf (8 per trial), Jmat (9), t_final (1) -> Qd, Qfd (8), Rd (3).
 * Optional guess outputs (nullable): w_guess (ragged nt x 3) / q_guess (ragged nt x 4) at row
 * offsets goffs[t] (host, n_trials entries), nt = length(t0:dt:t_final[t]).                   */
int ts_slew_weights_batch(ts_ctx* ctx, int64_t n_trials, const double* x0, const double* xf, const double* Jmat,
                          const double* t_final, double t0, double dt, double alpha, double beta, int eigen_axis_fix,
                          double* Qd, double* Qfd, double* Rd, const int64_t* goffs, double* w_guess, double* q_guess);

/* ---- K4: batched TVLQR closed-loop replay -------------------------------------- */
typedef struct ts_tvlqr_opts {
  double dt;                 /* dt_lqr (0.2)                                                  */
  double t0, tf;             /* t0; tf is taken per trial from t_final[]                       */
  double Qd[6], Qfd[6], Rd[3]; /* Q_lqr = diag(10,10,10,10,10,10), Qf = 100 Q, R = 7.5e3 I
                                 (TortoiseSat.jl:251-260)                                     */
  int32_t dt_squared;        /* 1: linearise with dt^2 (attitude_controller.jl:111,137, Q6)   */
  int32_t noise_mode;        /* 0 none, 1 explicit `noise` array, 2 Philox4x32-10(seed,trial,step,stage) */
  uint64_t seed;
  double w_limit, ang_limit; /* slew limits .05 rad/s, .08727 rad (monte_carlo.jl:69-71)       */
  int32_t literal_postproc;  /* 1: keep the `[1:3,i]` column bug of monte_carlo.jl:247 (Q12)   */
  int32_t pad_;
} ts_tvlqr_opts;
void ts_tvlqr_default_opts(ts_tvlqr_opts* o);

/* attitude_simulation(simulator, gain_simulator, :rk4, X, U, dt, x0, t0, tf, Q, R, Qf)
 * [src/attitude_controller.jl:1-48, with attitude_lqr :50-119, rk4 :122-145, simulator.jl,
 * gain_simulator.jl] for n_trials optimised slews, plus the slew-time rule of
 * src/monte_carlo.jl:237-262.  HOST per-trial arrays: N_i, offs, x0_lqr (8), Jmat (9), B_offs,
 * B_rows, index_scale, clock_rate, t_final, q_final (4), stream_id (nullable; Philox stream of
 * the trial, default = t).  Arrays following pointers_are_device: X_lqr (ragged N x 8), U_lqr
 * (ragged (N-1) x 3 at offs*3), B_eci, noise (nullable; ragged N x 4 x 9 at offs*36), outputs
 * (all nullable) X_sim (ragged N x 8), U_sim (N x 3), dX (N x 6), K (N x 3 x 6).  HOST outputs
 * (nullable): N_sim, slew_time (== t_final[t] when the trial "fails").                          */
int ts_tvlqr_sim_batch(ts_ctx* ctx, int64_t n_trials, const int64_t* N_i, const int64_t* offs, const double* X_lqr,
                       const double* U_lqr, const double* x0_lqr, const double* Jmat, const double* B_eci,
                       const int64_t* B_offs, const int64_t* B_rows, const double* index_scale, const double* clock_rate,
                       const double* t_final, const double* q_final, const uint32_t* stream_id, const ts_tvlqr_opts* opts,
                       const double* noise, double* X_sim, double* U_sim, double* dX, double* K, int64_t* N_sim,
                       double* slew_time, int pointers_are_device);

/* ---- fused Monte-Carlo run: the metric path -------------------------------------- *
 * For each trial: scoping field pass -> gramian cutoff -> fine field table -> eigen-axis /
 * Bryson weights -> AL-iLQR -> (optional) TVLQR replay + slew-time rule, i.e. the loop body of
 * src/monte_carlo.jl:118-262 with the solver block of src/TortoiseSat.jl:178-199.  Everything
 * between the per-trial inputs and the 64-byte outcome records stays in HBM.                  */
typedef struct ts_mc_config {
  int64_t n_trials;
  int32_t shared_orbit;  /* 1: all trials use kep6[0..5] / fopts[0] (fixed-orbit ensemble, configs[2]) */
  int32_t run_tvlqr;     /* 1: K4 replay + slew-time post-processing                                  */
  double t0, tf;         /* scoping window (0, 2400 in monte_carlo.jl:74-75; 0, 5400 in TortoiseSat.jl) */
  int64_t N_scope;       /* 5000                                                                      */
  double cutoff;         /* condition-number cutoff (30 / 50 / 100)                                   */
  double dt;             /* 0.2                                                                       */
  double alpha, beta;    /* Bryson weights                                                            */
  int32_t eigen_axis_fix;    /* see ts_slew_weights_batch; 0 = literal reference                          */
  int32_t keep_trajectories; /* 1: X, U, X_sim, U_sim and the fine field tables of this run stay resident in HBM
                                    for ts_mc_fetch_trajectories (the `states`, `control_inputs`, `sim_states`,
                                    `sim_control_inputs`, `B_ECI_total` arrays of monte_carlo.jl:52-66)
                                2: as 1, and the solver states, multipliers and per-trial inputs are kept too, for
                                    ts_mc_fetch_state and ts_mc_continue (same results as 1)                 */
  ts_ilqr_opts ilqr;
  ts_tvlqr_opts tvlqr;
} ts_mc_config;
typedef struct ts_mc_stats {
  int64_t n_trials, n_converged, n_no_cutoff, n_fail_slew;
  double sum_slew_time, sum_slew_time_sq, sum_t_final, sum_inner_iters, sum_ls_rollouts, sum_knots, flops;
  double ms_field, ms_prep, ms_solve, ms_tvlqr; /* device time of each stage (CUDA events) */
  int64_t n_status[6];                          /* trials per TS_ST_* code                  */
} ts_mc_stats;
/* HOST inputs: kep6 (n x 6, or 1 x 6 if shared_orbit), fopts (n, or 1; only GM, mjd, igrf_date,
 * field_radius_m are read), x0, xf (n x 8), Jmat (n x 9), q_noise0 (n x 3, nullable: initial
 * attitude perturbation of the replay, TortoiseSat.jl:231-234), stream_id (nullable).
 * HOST outputs: out (n records), stats (nullable).                                            */
int ts_monte_carlo_run(ts_ctx* ctx, const ts_mc_config* cfg, const double* kep6, const ts_field_opts* fopts, const double* x0,
                       const double* xf, const double* Jmat, const double* q_noise0, const uint32_t* stream_id,
                       ts_trial_outcome* out, ts_mc_stats* stats);

/* Trajectories of the most recent ts_monte_carlo_run on ctx that had cfg->keep_trajectories = 1 (they stay in HBM until
 * the next Monte-Carlo run on ctx).  Layout call: knot_offs (n_trials+1, HOST) -- trial t owns knots
 * [knot_offs[t], knot_offs[t+1]) (none if its status is TS_ST_NO_CUTOFF); row_offs (n_trials+1, HOST) -- trial t's
 * fine field table starts at row row_offs[t] and has 2*N_t rows (a shared-orbit run has ONE table: every row_offs[t]
 * is 0 and row_offs[n_trials] = 2N).  Fetch call: any of the HOST outputs may be null; X, X_sim: knots x 8 (states of
 * monte_carlo.jl:200, sim_states :232; rows >= N_sim of a trial's X_sim are 0), U, U_sim: knots x 3 (last row of each
 * trial unused = 0), B_eci: rows x 3 Tesla (B_ECI_total, monte_carlo.jl:149; rows the solver cannot index are 0).   */
int ts_mc_trajectory_layout(ts_ctx* ctx, int64_t n_trials, int64_t* knot_offs, int64_t* row_offs);
int ts_mc_fetch_trajectories(ts_ctx* ctx, double* X, double* U, double* X_sim, double* U_sim, double* B_eci);

/* ---- Monte-Carlo continuation: more outer iterations for the max-outer trials of a kept run ---------------- *
 * A ts_monte_carlo_run with cfg->keep_trajectories = 2 keeps, besides the trajectories, every active trial's solver
 * state (ts_al_state, CS1) and bound multipliers, its per-trial solver and replay inputs, the run's config and the final
 * outcome records.  They stay valid until the next ts_monte_carlo_run on ctx, whatever other entries run in between.
 * ts_mc_fetch_state copies the kept state to HOST arrays (either may be null): state gets n_trials records (a
 * TS_ST_NO_CUTOFF trial gets a zero record with status 5), lam (sum N) x 6 doubles in the layout of
 * ts_mc_trajectory_layout's knot_offs.  With ts_mc_fetch_trajectories that is what ts_alilqr_solve_state_batch needs
 * to continue a trial on its own.
 * ts_mc_continue continues the kept run in place (DESIGN.md section 4, K3):
 *  MC1 which trials: CS2 under the continuing call's opts, status == TS_ST_MAX_OUTER && outer_iters < opts->max_outer.
 *      Every other trial passes through unchanged, NO_CUTOFF trials included: its outcome record (byte for byte), its
 *      rows of X, U, X_sim and U_sim, its state and its lam.
 *  MC2 solve: the continuation path of ts_alilqr_solve_state_batch on the kept block (import, then the one-warp-per-
 *      trial kernels), the producer-warp kernel chosen by opts->k3_pair over the run's active trials.  X, U, the states
 *      and lam are updated in place.
 *  MC3 replay and records: with run_tvlqr, the continuing trials alone are replayed with the run's TVLQR options (after
 *      the fused path's overrides), stream ids and initial states; their X_sim / U_sim rows are cleared first.  A
 *      continued record has counters, J and c_max from the solver as totals over both calls (CS3), N and t_final
 *      unchanged, slew_time from the new replay (0 without run_tvlqr) and flops by ts_monte_carlo_run's formula over
 *      the totals.  `out` (HOST, n_trials records) returns the whole ensemble in caller order, and the kept block holds
 *      it: the fetch calls return the continued run and a second ts_mc_continue chains.
 *  MC4 equivalence: the continuing trials' solver results (X, U, counters, J, c_max, state, lam) equal bit for bit
 *      those of ts_alilqr_solve_state_batch continuing over the run's active trials from ts_mc_fetch_state and
 *      ts_mc_fetch_trajectories with the run's inputs.  Against a direct run to the larger max_outer, CS4 applies.
 * stats (nullable): counts and sums describe the whole ensemble after the call, as ts_monte_carlo_run reports them;
 * ms_solve, ms_tvlqr and flops this call's work (the added iterations and the replay); ms_field = ms_prep = 0.
 * ts_last_kernel_ms, ts_k3_last_split and ts_k3_last_parked report the continuation.  TS_ERR_ARG, with out and stats
 * untouched, when no run on ctx had keep_trajectories = 2 (the last run decides), n_trials differs from the kept run,
 * opts or out is null, or opts fails the checks of ts_alilqr_solve_state_batch; TS_ERR_NOMEM, nothing kept written and
 * the run still continuable, when the parked records of the continuing trials do not fit in device memory.          */
int ts_mc_fetch_state(ts_ctx* ctx, ts_al_state* state, double* lam);
int ts_mc_continue(ts_ctx* ctx, int64_t n_trials, const ts_ilqr_opts* opts, ts_trial_outcome* out, ts_mc_stats* stats);

/* ---- disturbance ensembles: the kept run's slews under many independent noise draws ------------------------- *
 * ts_mc_replay_ensemble replays every selected trial of the kept run n_real times, each time under an independent draw
 * of the simulator.jl disturbances, with the trial's kept optimised trajectory and its TVLQR gains (computed once per
 * call), and returns the slew time and final state of every (trial, realisation) pair (DESIGN.md section 4, K4):
 *  RE1 the kept run: the most recent ts_monte_carlo_run on ctx with keep_trajectories >= 1, continued by
 *      ts_mc_continue or not (after a continuation the continued trajectories are replayed).
 *  RE2 the draws of realisation r (0 <= r < 2^30), key = the run's tvlqr.seed, stream = the trial's stream id: the stage
 *      disturbances of step k, stage s are tvlqr_noise's with counter (stream, k, s, block + 4r), block 0..2 (r = 0 is
 *      the run's own stream); realisation r >= 1 starts from the trial's unperturbed x0 perturbed, as ts_monte_carlo_run
 *      applies q_noise0, by q_noise = q_noise_scale * (z0, z1, z2), (z0, z1) = box_muller(o0, o1), z2 = the first of
 *      box_muller(o2, o3), o = Philox4x32-10 of counter (stream, 0xFFFFFFFF, 0, 4r) (q_noise_scale = 0: x0 itself);
 *      realisation 0 starts from the run's x0_lqr.  Realisations always draw (noise mode 2), whatever the run's
 *      noise_mode; the run's TVLQR options apply with the fused path's overrides (dt, t0, literal_postproc = 0).
 *  RE3 realisation 0 is the run: when the run drew noise (noise_mode 1 or 2), realisation 0 of a trial has the kept
 *      record's slew_time and the kept X_sim row N_sim - 1 as x_final, bit for bit.
 *  RE4 row (trial t, realisation r) depends on the kept run, t, r and q_noise_scale alone, bit for bit: not on r_first
 *      or n_real (chunking), the other selected trials or their order, or the number of devices.
 *  RE5 isolation: nothing a later call reads is written; the kept run (records, trajectories, states) is unchanged.
 * trials (HOST, caller indices, repeats allowed; null = all n_trials, then n_sel == n_trials).  HOST outputs: slew_time
 * (n_sel x n_real, == t_final when the realisation "fails", monte_carlo.jl:257-261), x_final (n_sel x n_real x 8,
 * nullable): the state at the last simulated step.  A TS_ST_NO_CUTOFF trial gets NaN rows.  ts_last_kernel_ms is the
 * device time of the call (gains + ensemble replay); ts_mc_replay_ensemble_last_split gives the two parts.
 * TS_ERR_ARG, outputs untouched: no kept run, n_trials differs from the kept run's, n_real < 1, r_first < 0,
 * r_first + n_real > 2^30, a trial index out of range, opts or slew_time null.  TS_ERR_NOMEM, outputs untouched, when
 * the device outputs do not fit: chunk the realisations with r_first (RE4 makes that exact).                          */
typedef struct ts_replay_ensemble_opts {
  int64_t n_real;        /* realisations per selected trial, >= 1                     */
  int64_t r_first;       /* first realisation index; r_first + n_real <= 2^30         */
  double  q_noise_scale; /* initial attitude perturbation of realisations r >= 1 (RE2) */
} ts_replay_ensemble_opts;
int ts_mc_replay_ensemble(ts_ctx* ctx, int64_t n_trials, const ts_replay_ensemble_opts* opts, int64_t n_sel,
                          const int64_t* trials, double* slew_time, double* x_final);
int ts_mc_replay_ensemble_last_split(ts_ctx* ctx, double* gains_ms, double* replay_ms);

/* ---- dispersion ensembles: the kept run's slews under drawn truth-model errors ----------------------------------- *
 * ts_mc_dispersion_ensemble replays the kept run's slews as ts_mc_replay_ensemble does, with the TVLQR gains of the
 * nominal model, but each realisation's "truth" dynamics carry drawn errors of the inertia, the torquer gains and the
 * field model (DESIGN.md section 4, K4):
 *  DE1 the kept run: as RE1, with the argument checks of ts_mc_replay_ensemble.
 *  DE2 the draws of realisation r: the stage noise and (r >= 1) the initial attitude of RE2, and ten standard normals
 *      z0..z9 with key = the run's tvlqr.seed, counters (stream, 0xFFFFFFFE, 0, 4r + b), b = 0, 1, 2: (z0, z1) and
 *      (z2, z3) = box_muller of block 0's (o0, o1) and (o2, o3), (z4 .. z7) the same of block 1, (z8, z9) = box_muller
 *      of block 2's (o0, o1).  Parameters: d_i = exp(sigma_inertia z_i / 2) (i = 0..2), truth inertia
 *      J_true[i][j] = (d_i J[i][j]) d_j; g_i = exp(sigma_torquer z_{3+i}), truth torque ((u_i * 0.01) g_i) x B_B;
 *      s_B = exp(sigma_field_scale z6) and phi = sigma_field_angle (z7, z8, z9) rad, p = [cos(|phi|/2);
 *      phi/|phi| sin(|phi|/2)] (identity for |phi| <= 1e-300): truth field of a stage = s_B qrot(p, B_row) + B_noise.
 *      A group with sigma 0 keeps its nominal value exactly (1, 1, 1 / no rotation); each group reads fixed normals,
 *      so one sigma leaves the other groups' parameters and the stage noise unchanged (paired one-factor studies).
 *  DE3 realisation 0 carries no dispersion whatever the sigmas: its row is RE3's, bit for bit.
 *  DE4 with all four sigmas 0 every row equals ts_mc_replay_ensemble's row for the same (trial, r, q_noise_scale).
 *  DE5 a row depends on the kept run, t, r, q_noise_scale and the sigmas alone (as RE4).
 *  DE6 isolation, as RE5: later calls behave as if this call never ran.
 * Outputs as ts_mc_replay_ensemble, plus params (HOST, nullable): n_sel x n_real x 10, in the order d0 d1 d2 g0 g1 g2
 * s_B phi0 phi1 phi2.  A TS_ST_NO_CUTOFF trial gets NaN rows in every output.  ts_last_kernel_ms and
 * ts_mc_replay_ensemble_last_split report this call.  TS_ERR_ARG, outputs untouched: every case of
 * ts_mc_replay_ensemble, a null disp, a sigma negative or not finite, sigma_inertia, sigma_torquer or sigma_field_scale
 * above 1, sigma_field_angle above pi.  TS_ERR_NOMEM as ts_mc_replay_ensemble.                                       */
typedef struct ts_dispersion_opts {
  double sigma_inertia;     /* log-standard deviation of each principal inertia scale (J_true = D J D, D = diag(d)) */
  double sigma_torquer;     /* log-standard deviation of each torquer gain                                          */
  double sigma_field_scale; /* log-standard deviation of the field magnitude                                        */
  double sigma_field_angle; /* standard deviation of each field rotation-vector component, rad                      */
} ts_dispersion_opts;
int ts_mc_dispersion_ensemble(ts_ctx* ctx, int64_t n_trials, const ts_replay_ensemble_opts* opts, const ts_dispersion_opts* disp,
                              int64_t n_sel, const int64_t* trials, double* slew_time, double* x_final, double* params);

/* ---- weight-sweep ensembles: the kept run's slews under the TVLQR gains of many tracking weightings ---------------- *
 * ts_mc_weight_ensemble replays the kept run's slews as ts_mc_dispersion_ensemble does, once per weighting of sets:
 * the gains of set w come from the kept trajectory, linearised once, and a Riccati sweep with set w's diagonals of Q,
 * Qf and R (DESIGN.md section 4, K4):
 *  WE1 the kept run: as RE1, with the argument checks of ts_mc_replay_ensemble.
 *  WE2 paired draws: row (t, w, r) uses DE2's draws for (t, r) -- stage noise, initial attitude (r >= 1) and the ten
 *      truth-model normals; a null disp means all four sigmas 0.  The draws do not depend on w.  Every TVLQR option
 *      other than the weights is the run's, with the fused path's overrides.
 *  WE3 a set equal to the run's cfg.tvlqr weights, with u_limit 0, gives ts_mc_dispersion_ensemble's rows bit for bit
 *      (ts_mc_replay_ensemble's with a null disp); its realisation 0 is the kept record.
 *  WE4 torquer limit: u_limit 0 = none (simulator.jl); u_limit > 0 clamps each component of u = U_lqr - K dx to
 *      [-u_limit, u_limit] before it drives the step's four rk4 stages (a NaN stays NaN).  It acts in the truth model
 *      only; the gains are unchanged.  The planner's bound cfg.ilqr.u_max is the physical choice.
 *  WE5 a row depends on the kept run, t, r, q_noise_scale, the sigmas, set w's weights and u_limit alone: not on the
 *      other sets, their number or order, chunking, the other selected trials, their order or the number of devices.
 *  WE6 isolation, as RE5: later calls behave as if this call never ran.
 *  WE7 TS_ERR_ARG, outputs untouched: every case of ts_mc_dispersion_ensemble (the sigma checks when disp is
 *      non-null), n_sets < 1, a null sets, a Qd or Qfd entry negative or not finite, an Rd entry <= 0 or not finite, a
 *      u_limit negative or not finite.  TS_ERR_NOMEM, outputs untouched, when the gains of all sets (144 bytes per kept
 *      knot and set) or the device outputs do not fit: chunk the sets or the realisations (exact by WE5).
 * Outputs (HOST): slew_time n_sel x n_sets x n_real, x_final (nullable) n_sel x n_sets x n_real x 8.  A TS_ST_NO_CUTOFF
 * trial gets NaN rows in every set.  ts_last_kernel_ms and ts_mc_replay_ensemble_last_split report this call (gains:
 * the linearisation and every set's Riccati sweep; replay: the ensemble replay).                                        */
typedef struct ts_tvlqr_weights {   /* one tracking weighting: the diagonals of ts_tvlqr_opts' Q, Qf, R (120 bytes)   */
  double Qd[6], Qfd[6], Rd[3];
} ts_tvlqr_weights;
int ts_mc_weight_ensemble(ts_ctx* ctx, int64_t n_trials, const ts_replay_ensemble_opts* opts, const ts_dispersion_opts* disp,
                          int64_t n_sets, const ts_tvlqr_weights* sets, double u_limit, int64_t n_sel, const int64_t* trials,
                          double* slew_time, double* x_final);

/* ---- igrf12syn: the Fortran-style twin of igrf12 -------------------------------------------- *
 * igrf12syn(isv, date, itype, alt, colat, elong) [src/igrf.jl:335-534] at n points.  isv 0 = main field, 1 = secular
 * variation; itype 1 = geodetic (alt = height above the WGS-84 ellipsoid, km), 2 = geocentric (alt = radius, km);
 * colat in [0,180] deg, elong in [0,360] deg.  Outputs x (north), y (east), z (down), f (total) in nT (nT/yr for isv 1).
 * Returns TS_ERR_DATE for dates outside [1900, 2025] (igrf.jl:343-345).                                              */
int ts_igrf12syn_batch(ts_ctx* ctx, int isv, double date, int itype, int64_t n, const double* alt_km, const double* colat_deg,
                       const double* elong_deg, double* x, double* y, double* z, double* f, int pointers_are_device);

/* ---- K8: cubic B-spline interpolant of the igrf_data field map -------------------------------- *
 * extrapolate(interpolate(A, BSpline(Cubic(Reflect(OnCell())))), Periodic()) [src/magnetic_toolbox.jl:124-125] of an
 * n0 x n1 x 3 map A (e.g. the lat/long map of igrf_data, :108-121), under rules FM1..FM4 of DESIGN.md section 4 (K8).
 * 2 <= n0, n1 <= 2^20.  ts_field_map_prefilter (FM1): grid (n0 x n1 x 3) -> coefs ((n0+2) x (n1+2) x 3), each component
 * on its own.  ts_field_map_eval_batch (FM2, FM3): x0, x1 (n each, 1-based fractional indices along axis 0 / 1, any real
 * value: both axes wrap with period n0 / n1) -> out (n x 3: all three components; FM4, the integer component index with
 * period 3, is the caller's choice of column).  A non-finite index gives a NaN row and TS_ERR_DOMAIN; the other rows
 * are valid.                                                                                                         */
int ts_field_map_prefilter(ts_ctx* ctx, int64_t n0, int64_t n1, const double* grid, double* coefs, int pointers_are_device);
int ts_field_map_eval_batch(ts_ctx* ctx, int64_t n0, int64_t n1, const double* coefs, int64_t n, const double* x0,
                            const double* x1, double* out, int pointers_are_device);

/* ---- several GPUs of one node behind one handle ---------------------------------------------- *
 * ts_create_multi owns one ts_ctx per device, one host thread per device while a call runs, and (for n_devices > 1)
 * one NCCL communicator per device (libnccl.so.2 is loaded on first use; the single-GPU entry points never need it).
 * ts_multi_monte_carlo_run shards the trials round-robin (trial t -> device t mod n_devices: horizons are ragged),
 * runs ts_monte_carlo_run on every shard concurrently, gathers the 64-byte outcome records with ncclAllGather and
 * sums the statistics with ncclAllReduce; `out` comes back in the caller's trial order.  Same arguments as
 * ts_monte_carlo_run (a shared orbit is replicated on every device).  stats->ms_* = max over devices.               */
typedef struct ts_multi ts_multi;
int ts_create_multi(ts_multi** out, const int* device_ids, int n_devices);
void ts_destroy_multi(ts_multi* m);
const char* ts_multi_last_error(const ts_multi* m);
int ts_multi_device_count(const ts_multi* m);
ts_ctx* ts_multi_ctx(ts_multi* m, int i); /* the i-th device's context (borrowed) */
int ts_multi_monte_carlo_run(ts_multi* m, const ts_mc_config* cfg, const double* kep6, const ts_field_opts* fopts,
                             const double* x0, const double* xf, const double* Jmat, const double* q_noise0,
                             const uint32_t* stream_id, ts_trial_outcome* out, ts_mc_stats* stats);
/* ts_mc_continue on every device's kept shard of a ts_multi_monte_carlo_run with keep_trajectories = 2, then the
 * records gathered and the statistics reduced as after the run.  (Per-process multi-GPU needs no library call: each
 * rank continues its own context and gathers as after its run.)                                                     */
int ts_multi_mc_continue(ts_multi* m, int64_t n_trials, const ts_ilqr_opts* opts, ts_trial_outcome* out, ts_mc_stats* stats);
/* ts_mc_replay_ensemble over a ts_multi_monte_carlo_run kept with keep_trajectories >= 1: each selected trial is replayed
 * on the device that holds it (t mod n_devices), all devices at once, and the rows come back in the caller's order,
 * equal bit for bit to the single-device rows (RE4).  No collective is needed; per-process multi-GPU needs no library
 * call (each rank replays the trials of its own context).  ts_last_kernel_ms of device i's context is its own part.    */
int ts_multi_mc_replay_ensemble(ts_multi* m, int64_t n_trials, const ts_replay_ensemble_opts* opts, int64_t n_sel,
                                const int64_t* trials, double* slew_time, double* x_final);
/* ts_mc_dispersion_ensemble over a ts_multi_monte_carlo_run kept with keep_trajectories >= 1, dispatched as
 * ts_multi_mc_replay_ensemble; the rows equal the single-device rows bit for bit (DE5).                              */
int ts_multi_mc_dispersion_ensemble(ts_multi* m, int64_t n_trials, const ts_replay_ensemble_opts* opts, const ts_dispersion_opts* disp,
                                    int64_t n_sel, const int64_t* trials, double* slew_time, double* x_final, double* params);
/* ts_mc_weight_ensemble over a ts_multi_monte_carlo_run kept with keep_trajectories >= 1, dispatched as
 * ts_multi_mc_replay_ensemble; the rows equal the single-device rows bit for bit (WE5).                                  */
int ts_multi_mc_weight_ensemble(ts_multi* m, int64_t n_trials, const ts_replay_ensemble_opts* opts, const ts_dispersion_opts* disp,
                                int64_t n_sets, const ts_tvlqr_weights* sets, double u_limit, int64_t n_sel, const int64_t* trials,
                                double* slew_time, double* x_final);

/* ---- element-wise batch versions of the reference's building blocks (all HOST pointers) --- *
 * Correctness / drop-in paths for callers that use the small functions on their own; the fused
 * kernels above inline the same device code.                                                    */
/* kep_ECI(kep,t0,GM) [src/kep_ECI.jl:1-49]: kep6 n x 6, t0 n (nullable -> 0) -> rv6 n x 6 = [r km; v km/s]
 * (the input is NOT mutated, unlike kep_ECI.jl:7-8).                                            */
int ts_kep_eci_batch(ts_ctx* ctx, int64_t n, const double* kep6, const double* t0, double GM, double* rv6);
/* OrbitPlotter(x,p,t) [src/OrbitPlotter.jl:1-52]: x6 n x 6 -> dx6 n x 6.                       */
int ts_orbit_rhs_batch(ts_ctx* ctx, int64_t n, const double* x6, double* dx6);
/* legendre(Val{:schmidt},phi,n_max,false) [src/legendre.jl:254-292] and dlegendre(Val{:schmidt},phi,P,false)
 * [src/dlegendre.jl:221-309]: theta n -> P, dP (nullable) n x (n_max+1)^2 row-major, 1 <= n_max <= 13. */
int ts_legendre_schmidt_batch(ts_ctx* ctx, int64_t n, const double* theta, int n_max, double* P, double* dP);
/* mode 0 DerivFunction(dx,x,u) [src/DerivFunction.jl:1-48], 1 gain_simulator [src/gain_simulator.jl:1-53]:
 *   x n x 8, u n x 3, B = field table (B_rows x 3, the global B_ECI), index_scale = global N, clock_rate = 1/(tf-t0);
 * mode 2 attitude_dynamics(x,u,B_B,J) [src/attitude_dynamics.jl:2-24]: x n x 7, B = n x 3 body-frame field
 *   (B_rows, index_scale, clock_rate ignored).  Jmat: one 3x3 row-major inertia.  dx: n x 8 (modes 0,1) / n x 7. */
int ts_dynamics_batch(ts_ctx* ctx, int mode, int64_t n, const double* x, const double* u, const double* B, int64_t B_rows,
                      double index_scale, double clock_rate, const double* Jmat, double* dx);
/* rk3 ZOH step of Model(DerivFunction,8,3) [TrajOpt rk3 = src/attitude_controller.jl:178-187]: x n x 8 -> xn n x 8. */
int ts_rk3_step_batch(ts_ctx* ctx, int64_t n, const double* x, const double* u, const double* B, int64_t B_rows,
                      double index_scale, double clock_rate, const double* Jmat, double dt, double* xn);

/* ---- comparison controller (SURVEY 8f row 4) -------------------------------------------------- *
 * The Psiaki-style PD magnetic controller closed loop of src/comparison/psiaki2005.jl:116-164 for n_trials trials:
 * x[:,1] = x0; one explicit Euler step with zero moment (:124-125); then for i = 2:N-1
 *   B_meas = qrot(q_inv(q_i), B_ECI[:,i]); w_bar = w_guess[:,i] - w_i; q_bar = qmult(q_i, q_guess[:,i]);
 *   m = psiaki_controller(C_1, C_2, J, q_bar, w_bar, B_meas)      [src/comparison/psiaki_dynamics.jl:1-26]
 *   x_{i+1} = rk4_psiaki(attitude_dynamics, x_i, dt, m, B_meas, J)  [:63-73; src/attitude_dynamics.jl:2-24], q normalised.
 * HOST arrays: N_i, offs (knot offsets), x0 (n x 7), w_guess / q_guess (ragged N x 3 / N x 4: the eigen-axis reference of
 * eigen_axis_slew), B_eci (ragged N x 3: the field at every step), Jmat (n x 9).  Outputs: X (ragged N x 7), M (ragged N x 3
 * moments, nullable), q_err (ragged N x 4 error quaternions, nullable).                                              */
int ts_psiaki_pd_batch(ts_ctx* ctx, int64_t n_trials, const int64_t* N_i, const int64_t* offs, const double* x0,
                       const double* w_guess, const double* q_guess, const double* B_eci, const double* Jmat, double dt,
                       double C_1, double C_2, double* X, double* M, double* q_err);
/* attitude_dynamics_linear(x,u,x_linear,B_B,J) [src/attitude_dynamics.jl:26-48]: x, x_linear n x 7, u n x 3, B_B n x 3,
 * Jmat one 3x3 -> dx n x 7 (all HOST).                                                                              */
int ts_attitude_dynamics_linear_batch(ts_ctx* ctx, int64_t n, const double* x, const double* u, const double* x_linear,
                                      const double* B_B, const double* Jmat, double* dx);

#ifdef __cplusplus
}
#endif
#endif /* TORTOISE_B200_H */
