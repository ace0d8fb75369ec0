// Augmented-Lagrangian iLQR for ONE trial, executed cooperatively by a TEAM of 8
// lanes (four teams per warp).  Replaces the solve the reference gets from
// TrajectoryOptimization.jl v0.1.2 at src/TortoiseSat.jl:145-146,169,178-199
// (Model+rk3, LQRObjective, BoundConstraint u in [-1,1], goal_constraint(xf),
// AugmentedLagrangianSolver, solve!) -- algorithm = SURVEY.md Appendix C, the
// same frozen specification the CPU oracle implements independently.
//
// Lane roles inside one iLQR iteration
//   Jacobian phase  lane l linearises knot (chunk*8 + l): analytic rk3 Jacobians
//                   [A|B] (7x10) + stage-cost/AL gradients -> team shared memory
//   Riccati phase   lane j<7 owns column j of A (state column), lanes 0..2 also a
//                   column of B: M = S*col, G(:,j) = [A B]'*M.  The 3x3 Quu system
//                   is factorised redundantly by every lane (no exchange), lane j
//                   solves its own gain column K(:,j); S is re-replicated into
//                   registers (28 unique entries) through shared memory.
//   Line search     lane a rolls out step alpha = 2^-a: 8 candidate trajectories
//                   are evaluated speculatively in parallel, the first one the
//                   sequential rule of Appendix C would accept is taken.
// The `Team` parameter abstracts warp intrinsics so that the identical source
// runs under the host lane-emulator of the CPU tests (tests/hostsim).
#pragma once
#include <stdint.h>

#include "ilqr_math.cuh"

#ifdef __CUDACC__
#define TS_FN __device__ __forceinline__
#define TS_FN_NOINLINE __device__ __forceinline__  /* single call sites: inlining keeps TrialIn/opts out of local memory */
#define TS_NO_UNROLL _Pragma("unroll 1")
#else
#define TS_FN inline
#define TS_FN_NOINLINE inline
#define TS_NO_UNROLL
#endif

// Option block of the AL-iLQR solve (C ABI: ts_ilqr_opts has the same layout).
struct ts_ilqr_opts_dev {
  int32_t max_outer, max_inner, max_linesearch, dJ_counter_limit, stage_cost_dt, goal_mask;
  double cost_tol, cost_tol_intermediate, grad_tol, grad_tol_intermediate, constraint_tol;
  double penalty_initial, penalty_scaling, penalty_max, dual_max;
  double ls_lower, ls_upper, bp_reg_increase, bp_reg_max, bp_reg_min, bp_reg_fp;
  double max_cost_value, max_state_value, max_control_value, u_max, u_min;
  // assumption registry of SURVEY.md App. C (0 = frozen default, 1 = named alternative)
  int32_t a2_active_ge, a3_grad_over_N, a4_no_intermediate, a5_dual_active_only, a6_penalty_conditional, a7_carry_cost;
  double constraint_decrease_ratio;
  // K3 launch scheme (host side only)
  int32_t k3_suspend_after, k3_tail_share;
  double k3_early_factor;
  int32_t k3_pair, k3_wide_occ;
  int32_t quat_error, k3_generic_inertia;
};
// 64-byte per-trial record (C ABI: ts_trial_outcome).
struct ts_trial_outcome_dev {
  int32_t status, outer_iters, inner_iters, ls_rollouts;
  int64_t N;
  double J, c_max, t_final, slew_time, flops;
};
// 104-byte solver state of a finished trial (C ABI: ts_al_state; rules CS1-CS4 in DESIGN.md section 4, K3)
struct ts_al_state_dev {
  double mu, lam_goal[8], J, c_max;
  int32_t status, outer_iters, inner_iters, ls_rollouts;
};

namespace ts {

// cycle counter for the per-phase diagnostics returned in the outcome record of the low-level solve
TS_HD long long ts_clock() {
#ifdef __CUDA_ARCH__
  return clock64();
#else
  return 0;
#endif
}

enum { ST_CONVERGED = 0, ST_MAX_OUTER = 1, ST_COST_BLOWUP = 2, ST_REG_MAX = 3, ST_NAN = 4, ST_NO_CUTOFF = 5 };

constexpr int TEAM = 8;                       // lanes of a (narrow) team
// Shared-memory strides (compile-time, overridable for A/B builds; the round-1 layout is TS_SMEM_SKEW=0).  Measured on the
// 4096-trial benchmark ensemble, K3 time with the cofactor Quu solve: round-1 layout (84 / 8 / regions 128-byte
// multiples apart) 7.35 s -> 85 / 9 / skewed 7.04 s -> 84 / 10 / skewed 6.95 s -> 86 / 9 / skewed 6.92 s.
#ifndef TS_SMEM_SKEW
#define TS_SMEM_SKEW 1
#endif
#ifndef TS_REC
#define TS_REC (TS_SMEM_SKEW ? 86 : 84)
#endif
#ifndef TS_SS
#define TS_SS (TS_SMEM_SKEW ? 9 : 8)
#endif
// doubles per knot record in shared memory (84 used).  The lanes of a chunk write their records side by side: with a
// stride of 84 doubles (672 B = 32 mod 128) 32 lanes share four 8-byte bank slots, with 86 (48 mod 128) eight, and the
// records stay 16-byte aligned for the vectorised reads of the Riccati step (85 would be conflict-free but costs them).
constexpr int REC = TS_REC;
constexpr int FWD_REC = 50;                   // [x7 u3 | K 21 d 3 | lam 6 | B 9 +pad] doubles per staged knot
// Shared-memory layout of a team of W lanes (W = 8: one of four teams of a warp; W = 32: the whole warp
// working on ONE trial -- "wide" mode, used for the straggler of a warp once its three siblings are done).
template <int W>
struct SmL {
  static constexpr int REC0 = 0;                   // [W][REC]   Jacobians + cost gradients of the chunk
  // row stride of S and of M = S*[A|B]: the whole-warp step reads them by row AND by column from 28-30 lanes at once,
  // and a narrow team's lanes store one column each; with a stride of 8 doubles 7-10 rows fall on two 8-byte bank
  // slots (4- and 5-way conflicts), with 9 every row starts on its own slot (whole-warp step: 141 -> 78 shared-memory
  // wavefronts in stages A + B of a knot)
  static constexpr int SS = TS_SS;
  static constexpr int SCOL = REC0 + W * REC;      // [7][SS]    new S columns
  static constexpr int SVEC = SCOL + 7 * SS;       // [7]        new s
  static constexpr int KQ = SVEC + ((TS_SS & 1) ? 7 : 8);   // [7][6]     K(:,j), Qux(:,j)
  static constexpr int QUU = KQ + 42;              // [9] Quu, [3] Qu
  static constexpr int MM = QUU + 12;              // whole-warp team only: [10][SS] M = S*[A|B], [10] q = [A|B]'*s
  static constexpr int QV = MM + 10 * SS;
  static constexpr int BWD_END = QUU + 12 + (W >= 32 ? 10 * SS + 12 : 0);
  static constexpr int FWD = 0;                    // [2][W][FWD_REC] staged chunks of the forward pass (overlay)
  static constexpr int FWD_END = 2 * W * FWD_REC;
  static constexpr int WORK = (BWD_END > FWD_END ? BWD_END : FWD_END) + ((BWD_END > FWD_END ? BWD_END : FWD_END) & 1);
  static constexpr int TRIAL = WORK;               // the trial's TrialIn block (read-only during the solve)
  static constexpr int TOTAL = WORK + 64;
};
// 876 doubles = 7008 B per narrow team.  876 = 12 (mod 16): the four teams of a warp run the same code on their own
// regions, and most of their shared-memory reads are team-wide broadcasts (one address per team); with regions a
// multiple of 128 B apart the four addresses of such a read share their banks (4 wavefronts), +-32 B of skew per team
// puts them on four different 8-byte slots (1 wavefront), and an 8-lane row (64 B per team) takes the minimum of 2.
constexpr int TEAM_SMEM_DOUBLES = SmL<TEAM>::TOTAL;
static_assert(!TS_SMEM_SKEW || TEAM_SMEM_DOUBLES % 16 == 4 || TEAM_SMEM_DOUBLES % 16 == 12, "narrow team regions must be skewed by 32 B (mod 128 B)");
static_assert(8 * (4 * TEAM_SMEM_DOUBLES * 8 + 1024) <= 233472, "eight four-team warps per SM must fit the 228 KB of shared memory");
static_assert(SmL<32>::TOTAL <= 4 * SmL<TEAM>::TOTAL, "the wide layout must fit the four narrow regions of a warp");
constexpr int SM_TRIAL = SmL<TEAM>::TRIAL;

struct TrialIn {
  int N;
  double dt;
  double x0[7], clk0;
  double xf[8], Qd[8], Qfd[8], Rd[3];
  Inertia I;
  const double* Bt;  // field table rows x 3
  long long B_rows;
  double index_scale, clock_rate;
  const double* U0;  // (N-1) x 3 or null
};
static_assert(sizeof(TrialIn) <= 64 * sizeof(double), "TrialIn must fit its shared-memory slot");
struct TrialWork {
  double* xu;    // [9][Nmax][10]  trajectory buffers (x7,u3) of this slot: current + 8 line-search candidates
  double* xu_warp;        // xu of the warp's first slot; buffer i of the warp = xu_warp + (i/9)*slot_stride + (i%9)*Nmax*10
  long long slot_stride;  // doubles between consecutive slots
  double* kd;    // [Nmax][24]     K column-major (21) + d (3)
  double* lam;   // [Nmax][6]      bound multipliers
  double* clk;   // [Nmax]         clock state
  double* bk;    // [Nmax][10]     field vectors of the three rk3 stages of each knot (9 used)
  long long Nmax;
};

// Teams that receive the Jacobian records of a chunk from a PRODUCER warp (k3_pair_kernel) declare
// `static constexpr bool EXT_LIN = true` and provide lin_begin / rec_wait / rec_release / lin_abort; every other team
// linearises its chunk itself.
template <class Team, class = void>
struct team_ext_lin {
  static constexpr bool value = false;
};
template <class Team>
struct team_ext_lin<Team, decltype((void)Team::EXT_LIN)> {
  static constexpr bool value = Team::EXT_LIN;
};

// Teams that run the QUATERNION-AWARE variant (ts_ilqr_opts.quat_error; SURVEY 8(f2), reference monte_carlo.jl:158,192 +
// quaternion_toolbox.jl:15-75) declare `static constexpr bool QUAT = true`: the backward pass then works on the error
// state [dw(3); dphi(3); 0] with A_e = E(x_k+1)' A E(x_k), B_e = E(x_k+1)' B, E = blkdiag(I3, G(q)) (7 x 7 here, last
// column zero), cost gradients / Hessians projected the same way, and the rollout feeds back
// dx = [w - wbar; MRP(conj(qbar) (x) q); 0].  A compile-time switch so that the default kernels do not change by a
// single instruction.  Requires equal LQR weights and an all-or-nothing goal mask on the four quaternion components
// (the reference's Bryson weights are): E' (c I4) E = c |q|^2 I3 is then diagonal and fits the diagonal-Q Riccati step.
template <class Team, class = void>
struct team_quat {
  static constexpr bool value = false;
};
template <class Team>
struct team_quat<Team, decltype((void)Team::QUAT)> {
  static constexpr bool value = Team::QUAT;
};
// Teams of the DIAGONAL-INERTIA kernels declare `static constexpr bool DIAGJ = true`: the host launches them when every
// trial's inertia matrix is diagonal (mul_J / mul_Jinv in ilqr_math.cuh: same values, a third of the operations).
template <class Team, class = void>
struct team_diagj {
  static constexpr bool value = false;
};
template <class Team>
struct team_diagj<Team, decltype((void)Team::DIAGJ)> {
  static constexpr bool value = Team::DIAGJ;
};
// G(q) = [-v'; s I + hat(v)] (4 x 3) of the raw quaternion q = (s, v)  (quaternion_toolbox.jl:22-27)
TS_HD void quat_G(const double q[4], double G[4][3]) {
  const double s_ = q[0], v1 = q[1], v2 = q[2], v3 = q[3];
  G[0][0] = -v1; G[0][1] = -v2; G[0][2] = -v3;
  G[1][0] = s_;  G[1][1] = -v3; G[1][2] = v2;
  G[2][0] = v3;  G[2][1] = s_;  G[2][2] = -v1;
  G[3][0] = -v2; G[3][1] = v1;  G[3][2] = s_;
}

// Work pointers always address global memory; when a TrialWork lives in shared memory (k3_wide_kernel) the compiler
// can no longer infer that from the kernel parameters, and would fall back to generic LD/ST.
template <class T>
TS_HD T* gptr(T* p) {
#ifdef __CUDA_ARCH__
  __builtin_assume(__isGlobal(p));
#endif
  return p;
}

// trajectory buffer i in the warp's buffer space: slot i/9, buffer i%9 (a team that owns a single slot uses 0..8)
template <int W>
TS_HD double* xu_buf(const TrialWork& w, int i) {
  return gptr(w.xu_warp + (long long)(i / 9) * w.slot_stride + (long long)(i % 9) * (w.Nmax * 10));
}

TS_HD int sym_idx(int i, int j) { return (i <= j) ? (i * 7 - i * (i - 1) / 2 + (j - i)) : (j * 7 - j * (j - 1) / 2 + (i - j)); }

TS_HD bool inv3_gj(const double A[9], double out[9]) {
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
    if (M[p][c] == 0.0) return false;
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
  return true;
}

// Cholesky of a symmetric 3x3 -- the PD test of the backward pass.  L holds the strictly-lower
// entries at [3],[6],[7] and the RECIPROCALS of the diagonal at [0],[4],[8] so that the two
// triangular solves per lane need no division (3 divisions per knot instead of 15).
TS_HD bool chol3(const double A[9], double L[9]) {
  // straight-line: the three pivot tests are combined at the end (a non-positive pivot makes the later entries
  // NaN/inf, which nobody reads because the factorisation is then rejected) -- no branch on the critical path
  L[1] = L[2] = L[5] = 0.0;
  const double s0 = A[0];
  L[0] = rnorm(s0);
  L[3] = A[3] * L[0];
  L[6] = A[6] * L[0];
  const double s1 = A[4] - L[3] * L[3];
  L[4] = rnorm(s1);
  L[7] = (A[7] - L[6] * L[3]) * L[4];
  const double s2 = A[8] - L[6] * L[6] - L[7] * L[7];
  L[8] = rnorm(s2);
  return (s0 > 0.0) & (s1 > 0.0) & (s2 > 0.0);
}
TS_HD void chol3_solve(const double L[9], const double b[3], double x[3]) {
  double y[3];
  y[0] = b[0] * L[0];
  y[1] = (b[1] - L[3] * y[0]) * L[4];
  y[2] = (b[2] - L[6] * y[0] - L[7] * y[1]) * L[8];
  x[2] = y[2] * L[8];
  x[1] = (y[1] - L[7] * x[2]) * L[4];
  x[0] = (y[0] - L[3] * x[1] - L[6] * x[2]) * L[0];
}

// The 3x3 system of the backward pass as it sits on the critical path of every knot.  Default (TS_QUU_SOLVER = 1): the
// symmetric cofactor matrix and ONE reciprocal of the determinant -- cofactors (2 dependent FP64 operations), determinant
// (3), reciprocal, and a solve is three independent 3-term dot products scaled by 1/det, which do not wait for the
// reciprocal: ~15 dependent operations for "factor + solve" instead of ~50 with three chained rsqrt in the Cholesky
// factor and the two triangular sweeps.  The PD test is Sylvester's criterion on the same matrix (leading minors
// a00, a00 a11 - a01^2, det > 0), which is the Cholesky pivot test (s0 = a00, s1 = m2 / a00, s2 = det / m2) in exact
// arithmetic.  TS_QUU_SOLVER = 0 compiles the reciprocal-Cholesky version back in (A/B and flop counting).
#ifndef TS_QUU_SOLVER
#define TS_QUU_SOLVER 1
#endif
TS_HD bool quu_factor(const double A[9], double F[9]) {
#if TS_QUU_SOLVER == 0
  return chol3(A, F);
#else
  const double a00 = A[0], a01 = A[3], a02 = A[6], a11 = A[4], a12 = A[7], a22 = A[8];   // lower triangle, as chol3 reads it
  const double c00 = a11 * a22 - a12 * a12;
  const double c01 = a02 * a12 - a01 * a22;
  const double c02 = a01 * a12 - a02 * a11;
  const double c11 = a00 * a22 - a02 * a02;
  const double c12 = a01 * a02 - a00 * a12;
  const double c22 = a00 * a11 - a01 * a01;
  const double det = a00 * c00 + a01 * c01 + a02 * c02;
  F[0] = c00; F[1] = c01; F[2] = c02; F[3] = c11; F[4] = c12; F[5] = c22;
#ifdef __CUDA_ARCH__
  F[6] = __drcp_rn(det);
#else
  F[6] = 1.0 / det;
#endif
  F[7] = F[8] = 0.0;
  return (a00 > 0.0) & (c22 > 0.0) & (det > 0.0);
#endif
}
TS_HD void quu_solve(const double F[9], const double b[3], double x[3]) {
#if TS_QUU_SOLVER == 0
  chol3_solve(F, b, x);
#else
  x[0] = (F[0] * b[0] + F[1] * b[1] + F[2] * b[2]) * F[6];
  x[1] = (F[1] * b[0] + F[3] * b[1] + F[4] * b[2]) * F[6];
  x[2] = (F[2] * b[0] + F[4] * b[1] + F[5] * b[2]) * F[6];
#endif
}

struct StageAL {  // stage cost pieces at (x,u)
  double l;       // 0.5 e'Qe + 0.5 u'Ru (unscaled)
  double c[6];
};
TS_HD void bound_c(const ts_ilqr_opts_dev& o, const double u[3], double c[6]) {
  for (int i = 0; i < 3; ++i) {
    c[i] = u[i] - o.u_max;
    c[3 + i] = o.u_min - u[i];
  }
}

// A2: an inequality is active when c > 0 (default) or c >= 0; `c >= 0` is `c > -(smallest subnormal)`, so the switch
// costs one uniform select instead of a second comparison per constraint.
TS_HD double active_threshold(const ts_ilqr_opts_dev& o) { return o.a2_active_ge ? -4.9406564584124654e-324 : 0.0; }

// Adds one knot's AL stage cost to Jc in the oracle's summation order; updates cmax.
TS_HD void add_stage_cost(const TrialIn& in, const ts_ilqr_opts_dev& o, double sc, double mu, const double x[7], double e8,
                          const double u[3], const double lam[6], double& Jc, double& cmax) {
  double l = 0.0;
  for (int i = 0; i < 7; ++i) {
    const double e = x[i] - in.xf[i];
    l += 0.5 * in.Qd[i] * e * e;
  }
  if (in.Qd[7] != 0.0) l += 0.5 * in.Qd[7] * e8 * e8;
  for (int i = 0; i < 3; ++i) l += 0.5 * in.Rd[i] * u[i] * u[i];
  Jc += l * sc;
  double c[6];
  bound_c(o, u, c);
  const double act_thr = active_threshold(o);
  for (int i = 0; i < 6; ++i) {
    const bool act = (c[i] > act_thr) || (lam[i] > 0.0);
    Jc += lam[i] * c[i] + (act ? 0.5 * mu * c[i] * c[i] : 0.0);
    cmax = (c[i] > cmax) ? c[i] : cmax;   // == fmax(cmax, fmax(0, c)): cmax starts at 0 and only grows; a NaN c is skipped either way
  }
}
TS_HD void add_terminal_cost(const TrialIn& in, const ts_ilqr_opts_dev& o, double mu, const double x[7], double e8,
                             const double lam_g[8], double& Jc, double& cmax) {
  for (int i = 0; i < 8; ++i) {
    const double e = (i < 7) ? (x[i] - in.xf[i]) : e8;
    Jc += 0.5 * in.Qfd[i] * e * e;
    if (o.goal_mask & (1 << i)) {
      Jc += lam_g[i] * e + 0.5 * mu * e * e;
      cmax = fmax(cmax, fabs(e));
    }
  }
}

struct Reg {
  double rho, drho;
};
TS_HD void reg_increase(const ts_ilqr_opts_dev& o, Reg& r) {
  r.drho = fmax(r.drho * o.bp_reg_increase, o.bp_reg_increase);
  r.rho = fmax(r.rho * r.drho, o.bp_reg_min);
}
TS_HD void reg_decrease(const ts_ilqr_opts_dev& o, Reg& r) {
  r.drho = fmin(r.drho / o.bp_reg_increase, 1.0 / o.bp_reg_increase);
  r.rho = r.rho * r.drho * ((r.rho * r.drho > o.bp_reg_min) ? 1.0 : 0.0);
}

// ----------------------------------------------------------------------------------------
// Jacobian phase for one knot (executed by ONE lane): fills a shared-memory knot record
//   rec[c*7 + i] = [A|B](i,c)  (column-major, c = 0..9), rec[70+i] = lx, rec[77+i] = lu, rec[80+i] = luu
template <class Team>
TS_FN_NOINLINE void linearise_knot(const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w, const double* xu_cur,
                                   int k, double sc, double mu, double* rec) {
  // all global inputs of the knot are loaded up front (one memory round trip, not one per use)
  const double* p = xu_cur + (long long)k * 10;
  const double* bp = gptr(w.bk) + (long long)k * 10;
  const double* lp_ = gptr(w.lam) + (long long)k * 6;
  double x[7], u[3], b[9], lam[6];
  for (int i = 0; i < 7; ++i) x[i] = p[i];
  for (int i = 0; i < 3; ++i) u[i] = p[7 + i];
  for (int i = 0; i < 9; ++i) b[i] = bp[i];
  for (int i = 0; i < 6; ++i) lam[i] = lp_[i];
  if (!team_ext_lin<Team>::value) rk3_jac7_jvp<team_diagj<Team>::value>(in.I, x, u, b, b + 3, b + 6, in.dt, rec);   // else: written by the producer warp
  for (int i = 0; i < 7; ++i) rec[70 + i] = sc * in.Qd[i] * (x[i] - in.xf[i]);
  double c6[6];
  bound_c(o, u, c6);
  const double act_thr = active_threshold(o);
  for (int i = 0; i < 3; ++i) {
    double lu = sc * in.Rd[i] * u[i];
    double luu = sc * in.Rd[i];
    const double lp = lam[i], ln = lam[3 + i];
    const bool ap = (c6[i] > act_thr) || (lp > 0.0);
    const bool an = (c6[3 + i] > act_thr) || (ln > 0.0);
    lu += (lp + (ap ? mu * c6[i] : 0.0)) - (ln + (an ? mu * c6[3 + i] : 0.0));
    luu += (ap ? mu : 0.0) + (an ? mu : 0.0);
    rec[77 + i] = lu;
    rec[80 + i] = luu;
  }
  if constexpr (team_quat<Team>::value) {
    // error coordinates (in place, in the knot's shared-memory record): columns 3..6 of [A] times G(q_k), then rows
    // 3..6 of [A|B] times G(q_k+1)'; the 7th row / column of the error state is identically zero
    double G0[4][3], G1[4][3];
    quat_G(x + 3, G0);
    quat_G(p + 10 + 3, G1);   // the next knot of the nominal trajectory (k <= N-2)
    for (int i = 0; i < 7; ++i) {
      const double a0 = rec[3 * 7 + i], a1 = rec[4 * 7 + i], a2 = rec[5 * 7 + i], a3 = rec[6 * 7 + i];
      for (int j = 0; j < 3; ++j) rec[(3 + j) * 7 + i] = a0 * G0[0][j] + a1 * G0[1][j] + a2 * G0[2][j] + a3 * G0[3][j];
      rec[6 * 7 + i] = 0.0;
    }
    for (int c = 0; c < 10; ++c) {
      const double r0 = rec[c * 7 + 3], r1 = rec[c * 7 + 4], r2 = rec[c * 7 + 5], r3 = rec[c * 7 + 6];
      for (int j = 0; j < 3; ++j) rec[c * 7 + 3 + j] = G1[0][j] * r0 + G1[1][j] * r1 + G1[2][j] * r2 + G1[3][j] * r3;
      rec[c * 7 + 6] = 0.0;
    }
    {
      const double l0 = rec[73], l1 = rec[74], l2 = rec[75], l3 = rec[76];
      for (int j = 0; j < 3; ++j) rec[73 + j] = G0[0][j] * l0 + G0[1][j] * l1 + G0[2][j] * l2 + G0[3][j] * l3;
      rec[76] = 0.0;
    }
    rec[83] = sc * in.Qd[3] * (x[3] * x[3] + x[4] * x[4] + x[5] * x[5] + x[6] * x[6]);   // E' (c I4) E = c |q|^2 I3
  }
}

// Backward Riccati sweep over the current trajectory.  Returns false if the regularisation ran away.
template <class Team>
TS_FN bool backward_pass(Team& tm, const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w, const double* xu_cur,
                         double sc, double mu, const double lam_g[8], Reg& reg, double& dV1, double& dV2, long long& cyc_lin) {
  typedef SmL<Team::W> L;
  constexpr int W = Team::W;
  double* sm = tm.smem();
  const int lane = tm.lane();
  const int N = in.N;
  int restarts = 0;
  for (;;) {  // regularisation restart loop
    dV1 = 0.0;
    dV2 = 0.0;
    // terminal value function -> shared memory (the per-knot loop loads S at its top, so the 35 doubles of
    // S/s are NOT live in registers across the register-hungry linearisation phase)
    tm.sync();
    if (lane < 7) {
      const double* xN = xu_cur + (long long)(N - 1) * 10;
      const double e = xN[lane] - in.xf[lane];
      double sxx = in.Qfd[lane], sx = in.Qfd[lane] * e;
      if (o.goal_mask & (1 << lane)) {
        sxx += mu;
        sx += lam_g[lane] + mu * e;
      }
      if constexpr (team_quat<Team>::value) {
        if (lane >= 3) {   // E_N' (.) E_N: attitude error coordinates 3..5, nothing in 6
          double G[4][3], v[4];
          quat_G(xN + 3, G);
          for (int r = 0; r < 4; ++r) {
            const double er = xN[3 + r] - in.xf[3 + r];
            v[r] = in.Qfd[3 + r] * er;
            if (o.goal_mask & (1 << (3 + r))) v[r] += lam_g[3 + r] + mu * er;
          }
          const int a_ = (lane < 6) ? lane - 3 : 0;
          const double w3 = in.Qfd[3] + ((o.goal_mask & 8) ? mu : 0.0);
          sxx = (lane < 6) ? w3 * (xN[3] * xN[3] + xN[4] * xN[4] + xN[5] * xN[5] + xN[6] * xN[6]) : 0.0;
          sx = (lane < 6) ? G[0][a_] * v[0] + G[1][a_] * v[1] + G[2][a_] * v[2] + G[3][a_] * v[3] : 0.0;
        }
      }
      for (int i = 0; i < 7; ++i) sm[L::SCOL + lane * L::SS + i] = (i == lane) ? sxx : 0.0;
      sm[L::SVEC + lane] = sx;
    }
    bool not_pd = false;
    const int n_chunks = (N - 1 + W - 1) / W;
    int pos = 0;   // position of the chunk in this sweep (0 = last chunk of the trajectory)
    if constexpr (team_ext_lin<Team>::value) tm.lin_begin(xu_cur, gptr(w.bk), N);
    TS_NO_UNROLL
    for (int ch = n_chunks - 1; ch >= 0 && !not_pd; --ch) {
      const int base = ch * W;
      tm.sync();  // previous chunk's records fully consumed
      const long long tl0 = ts_clock();
      double* recs = sm + L::REC0;
      if constexpr (team_ext_lin<Team>::value) recs = tm.rec_wait(pos);   // Jacobians of this chunk from the producer warp
      if (base + lane < N - 1) linearise_knot<Team>(in, o, w, xu_cur, base + lane, sc, mu, recs + lane * REC);
      tm.sync();
      cyc_lin += ts_clock() - tl0;
      if (!team_ext_lin<Team>::value && base >= W) {  // L2 prefetch of the next (lower) chunk's linearisation inputs: hidden behind the Riccati steps
        const int kn = base - W + lane;
        tm.prefetch_l2(xu_cur + (long long)kn * 10);
        tm.prefetch_l2(gptr(w.bk) + (long long)kn * 10);
        tm.prefetch_l2(gptr(w.lam) + (long long)kn * 6);
      }
      int kk_hi = N - 2 - base;
      if (kk_hi > W - 1) kk_hi = W - 1;
      TS_NO_UNROLL
      for (int kk = kk_hi; kk >= 0; --kk) {
        const double* rec = recs + kk * REC;
        const int k = base + kk;
        if constexpr (W >= 32) {
          // ================= whole-warp team: the knot step spread over 30 lanes =================
          // The narrow team gives each of its lanes a whole column (119 FMAs in a row); a warp that works on ONE
          // trial has lanes to spare, so here every lane computes at most three 7-term dot products per stage:
          //   A  M(i,c) = S(i,:)*[A|B](:,c)      lane (i = lane%7, g = lane/7 < 4) takes c = g, g+4, g+8;
          //      q(c)   = [A|B](:,c)'*s           lanes 28..31
          //   B  G(r,c) = [A|B](:,r)'*M(:,c)      lane (i,g): Qxx(i,j) for j = g, g+4 (kept in registers for P3);
          //                                       lanes 0..20 one entry of Qux, lanes 21..29 one entry of Quu
          //   P2 3x3 Cholesky in every lane; each lane solves the (at most three) gain columns it needs itself
          //   P3 lane (i,g): S_new(i,j) for j = g, g+4; the lanes with i == j also s_new(j)
          // Every dot product and sum is evaluated in the order of the narrow path below: same results bit for bit.
          // (written without divergent branches: lanes that have no task in a stage compute a clamped duplicate
          //  and only their stores are predicated -- a divergent side branch costs its full latency again)
          const int li = lane % 7, lg = lane / 7;
          const bool rowlane = lane < 28;
          const int j0 = lg < 4 ? lg : 3, j1 = lg + 4 < 7 ? lg + 4 : 6;   // clamped; validity in has_j1
          const bool has_j1 = rowlane && lg + 4 < 7;
          {  // ---- stage A: lanes 0..27 one row of S against up to three columns; lanes 28..31 the vector s
            double X[7];
            for (int l = 0; l < 7; ++l) {
              const double srow = 0.5 * (sm[L::SCOL + l * L::SS + li] + sm[L::SCOL + li * L::SS + l]);
              X[l] = rowlane ? srow : sm[L::SVEC + l];
            }
            const int c0 = rowlane ? lg : lane - 28;
            for (int q = 0; q < 3; ++q) {
              const int c = c0 + 4 * q;
              const int cc = c < 10 ? c : 9;
              double t = 0.0;
              for (int l = 0; l < 7; ++l) t += X[l] * rec[cc * 7 + l];
              if (c < 10) sm[rowlane ? (L::MM + c * L::SS + li) : (L::QV + c)] = t;
            }
          }
          tm.sync();
          double Qxx0, Qxx1;
          {  // ---- stage B
            double arow[7];
            for (int l = 0; l < 7; ++l) arow[l] = rec[li * 7 + l];
            double t = 0.0;
            for (int l = 0; l < 7; ++l) t += arow[l] * sm[L::MM + j0 * L::SS + l];
            if constexpr (team_quat<Team>::value) {   // l_xx(li, li) in error coordinates
              const double qd_li = (li < 3) ? sc * in.Qd[li] : ((li < 6) ? rec[83] : 0.0);
              Qxx0 = t + ((li == j0) ? qd_li : 0.0);
            } else {
              Qxx0 = t + ((li == j0) ? sc * in.Qd[li] : 0.0);
            }
            t = 0.0;
            for (int l = 0; l < 7; ++l) t += arow[l] * sm[L::MM + j1 * L::SS + l];
            if constexpr (team_quat<Team>::value) {
              const double qd_li = (li < 3) ? sc * in.Qd[li] : ((li < 6) ? rec[83] : 0.0);
              Qxx1 = t + ((li == j1) ? qd_li : 0.0);
            } else {
              Qxx1 = t + ((li == j1) ? sc * in.Qd[li] : 0.0);
            }
            const bool isux = lane < 21;
            const int u = isux ? lane : (lane < 30 ? lane - 21 : 0);
            const int rr = u % 3, cc = isux ? u / 3 : 7 + u / 3;
            t = 0.0;
            for (int l = 0; l < 7; ++l) t += rec[(7 + rr) * 7 + l] * sm[L::MM + cc * L::SS + l];
            const double tq = t + ((rr == cc - 7) ? rec[80 + rr] : 0.0);
            if (lane < 30) sm[isux ? (L::KQ + cc * 3 + rr) : (L::QUU + rr * 3 + (cc - 7))] = isux ? t : tq;   // Qux(rr,cc) | Quu(rr,cc-7)
          }
          tm.sync();
          double Quu[9], Qu[3], Qr[9], Lc[9];
          for (int i = 0; i < 9; ++i) Quu[i] = sm[L::QUU + i];
          for (int i = 0; i < 3; ++i) Qu[i] = rec[77 + i] + sm[L::QV + 7 + i];
          for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) Qr[i * 3 + j] = 0.5 * (Quu[i * 3 + j] + Quu[j * 3 + i]) + ((i == j) ? reg.rho : 0.0);
          if (!quu_factor(Qr, Lc)) {
            not_pd = true;  // identical decision in every lane
            break;
          }
          double d[3], Quud[3];
          {
            const double nb[3] = {-Qu[0], -Qu[1], -Qu[2]};
            quu_solve(Lc, nb, d);
            for (int i = 0; i < 3; ++i) Quud[i] = Quu[i * 3 + 0] * d[0] + Quu[i * 3 + 1] * d[1] + Quu[i * 3 + 2] * d[2];
          }
          for (int l = 0; l < 3; ++l) {
            dV1 += d[l] * Qu[l];
            dV2 += 0.5 * d[l] * Quud[l];
          }
          double* kdk = gptr(w.kd) + (long long)k * 24;
          {  // ---- gains this lane needs, then its entries of the new value function
            double Quxi[3], Ki[3];
            for (int c = 0; c < 3; ++c) Quxi[c] = sm[L::KQ + li * 3 + c];
            {
              const double nb[3] = {-Quxi[0], -Quxi[1], -Quxi[2]};
              quu_solve(Lc, nb, Ki);
            }
            if (lane < 7)
              for (int c = 0; c < 3; ++c) kdk[li * 3 + c] = Ki[c];
            if (lane == 7)
              for (int c = 0; c < 3; ++c) kdk[21 + c] = d[c];
            for (int q = 0; q < 2; ++q) {
              const int j = q ? j1 : j0;
              const bool valid = q ? has_j1 : rowlane;
              double Quxj[3], Kj[3], QuuK[3];
              for (int c = 0; c < 3; ++c) Quxj[c] = sm[L::KQ + j * 3 + c];
              const double nb[3] = {-Quxj[0], -Quxj[1], -Quxj[2]};
              quu_solve(Lc, nb, Kj);
              for (int i = 0; i < 3; ++i) QuuK[i] = Quu[i * 3 + 0] * Kj[0] + Quu[i * 3 + 1] * Kj[1] + Quu[i * 3 + 2] * Kj[2];
              double t = q ? Qxx1 : Qxx0;
              for (int l = 0; l < 3; ++l) t += Ki[l] * QuuK[l];
              for (int l = 0; l < 3; ++l) t += Ki[l] * Quxj[l];
              for (int l = 0; l < 3; ++l) t += Quxi[l] * Kj[l];
              if (valid) sm[L::SCOL + j * L::SS + li] = t;
            }
            // new s(li) from this lane's own gain column (K(:,li), Qux(:,li)); lanes 0..6 store the seven entries
            double ts = rec[70 + li] + sm[L::QV + li];
            for (int l = 0; l < 3; ++l) ts += Ki[l] * Quud[l];
            for (int l = 0; l < 3; ++l) ts += Ki[l] * Qu[l];
            for (int l = 0; l < 3; ++l) ts += Quxi[l] * d[l];
            if (lane < 7) sm[L::SVEC + li] = ts;
          }
          tm.sync();
        } else {
          // ---- P0: value function of knot k+1 from shared memory, symmetrised (App. C: Sxx = (Sxx+Sxx')/2)
          double S[28], s[7];
          for (int i = 0; i < 7; ++i)
            for (int j = i; j < 7; ++j) S[sym_idx(i, j)] = 0.5 * (sm[L::SCOL + j * L::SS + i] + sm[L::SCOL + i * L::SS + j]);
          for (int i = 0; i < 7; ++i) s[i] = sm[L::SVEC + i];
          // ---- P1: column products
          double Qxxc[7], Quxc[3], Qx = 0.0;
          if (lane < 7) {
            double a[7], m[7];
            for (int i = 0; i < 7; ++i) a[i] = rec[lane * 7 + i];
            for (int i = 0; i < 7; ++i) {
              double t = 0.0;
              for (int l = 0; l < 7; ++l) t += S[sym_idx(i, l)] * a[l];
              m[i] = t;
            }
            for (int i = 0; i < 7; ++i) {
              double t = 0.0;
              for (int l = 0; l < 7; ++l) t += rec[i * 7 + l] * m[l];
              if constexpr (team_quat<Team>::value) {   // l_xx(i, i) in error coordinates: c |q|^2 on 3..5, nothing on 6
                const double qd_i = (i < 3) ? sc * in.Qd[i] : ((i < 6) ? rec[83] : 0.0);
                Qxxc[i] = t + ((i == lane) ? qd_i : 0.0);
              } else {
                Qxxc[i] = t + ((i == lane) ? sc * in.Qd[i] : 0.0);
              }
            }
            for (int c = 0; c < 3; ++c) {
              double t = 0.0;
              for (int l = 0; l < 7; ++l) t += rec[(7 + c) * 7 + l] * m[l];
              Quxc[c] = t;
            }
            double t = 0.0;
            for (int l = 0; l < 7; ++l) t += a[l] * s[l];
            Qx = rec[70 + lane] + t;
          }
          if (lane < 3) {
            double b[7], m[7];
            for (int i = 0; i < 7; ++i) b[i] = rec[(7 + lane) * 7 + i];
            for (int i = 0; i < 7; ++i) {
              double t = 0.0;
              for (int l = 0; l < 7; ++l) t += S[sym_idx(i, l)] * b[l];
              m[i] = t;
            }
            for (int c = 0; c < 3; ++c) {
              double t = 0.0;
              for (int l = 0; l < 7; ++l) t += rec[(7 + c) * 7 + l] * m[l];
              sm[L::QUU + c * 3 + lane] = t + ((c == lane) ? rec[80 + c] : 0.0);
            }
            double t = 0.0;
            for (int l = 0; l < 7; ++l) t += b[l] * s[l];
            sm[L::QUU + 9 + lane] = rec[77 + lane] + t;
          }
          tm.sync();
          // ---- P2: 3x3 solve (every lane, redundantly)
          double Quu[9], Qu[3], Qr[9], L[9];
          for (int i = 0; i < 9; ++i) Quu[i] = sm[L::QUU + i];
          for (int i = 0; i < 3; ++i) Qu[i] = sm[L::QUU + 9 + i];
          for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) Qr[i * 3 + j] = 0.5 * (Quu[i * 3 + j] + Quu[j * 3 + i]) + ((i == j) ? reg.rho : 0.0);
          if (!quu_factor(Qr, L)) {
            not_pd = true;  // identical decision in every lane of the team
            break;
          }
          double Kc[3] = {0.0, 0.0, 0.0}, d[3], Quud[3], QuuK[3] = {0.0, 0.0, 0.0};
          {
            const double nb[3] = {-Qu[0], -Qu[1], -Qu[2]};
            quu_solve(L, nb, d);
            for (int i = 0; i < 3; ++i) Quud[i] = Quu[i * 3 + 0] * d[0] + Quu[i * 3 + 1] * d[1] + Quu[i * 3 + 2] * d[2];
          }
          double* kdk = gptr(w.kd) + (long long)k * 24;
          if (lane < 7) {
            const double nb[3] = {-Quxc[0], -Quxc[1], -Quxc[2]};
            quu_solve(L, nb, Kc);
            for (int i = 0; i < 3; ++i) QuuK[i] = Quu[i * 3 + 0] * Kc[0] + Quu[i * 3 + 1] * Kc[1] + Quu[i * 3 + 2] * Kc[2];
            for (int c = 0; c < 3; ++c) {
              sm[L::KQ + lane * 6 + c] = Kc[c];
              sm[L::KQ + lane * 6 + 3 + c] = Quxc[c];
              kdk[lane * 3 + c] = Kc[c];
            }
          }
          if (lane == 7)  // (predicated stores, not an else-branch: a divergent side path costs its latency again)
            for (int c = 0; c < 3; ++c) kdk[21 + c] = d[c];
          for (int l = 0; l < 3; ++l) {
            dV1 += d[l] * Qu[l];
            dV2 += 0.5 * d[l] * Quud[l];
          }
          tm.sync();
          // ---- P3: new S column / s entry
          if (lane < 7) {
            for (int i = 0; i < 7; ++i) {
              const double* kq = sm + L::KQ + i * 6;
              double t = Qxxc[i];
              for (int l = 0; l < 3; ++l) t += kq[l] * QuuK[l];
              for (int l = 0; l < 3; ++l) t += kq[l] * Quxc[l];
              for (int l = 0; l < 3; ++l) t += kq[3 + l] * Kc[l];
              sm[L::SCOL + lane * L::SS + i] = t;
            }
            double t = Qx;
            for (int l = 0; l < 3; ++l) t += Kc[l] * Quud[l];
            for (int l = 0; l < 3; ++l) t += Kc[l] * Qu[l];
            for (int l = 0; l < 3; ++l) t += Quxc[l] * d[l];
            sm[L::SVEC + lane] = t;
          }
          tm.sync();
        }
      }
      if constexpr (team_ext_lin<Team>::value) {
        if (!not_pd) {   // chunk consumed: hand its buffer back (the producer fills it for the chunk after next)
          tm.rec_release(pos, pos + 2 < n_chunks);
          ++pos;
        }
      }
    }
    if constexpr (team_ext_lin<Team>::value) {
      if (not_pd) tm.lin_abort(pos, n_chunks);   // regularisation restart: drain the producer, then start the sweep again
    }
    if (!not_pd) break;
    reg_increase(o, reg);
    if (reg.rho > o.bp_reg_max || ++restarts > 200) return false;
  }
  reg_decrease(o, reg);
  return true;
}

// AL cost + c_max of a stored trajectory, knots spread over the lanes (tree-summed).
template <class Team>
TS_FN double trajectory_cost(Team& tm, const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w, const double* xu,
                             double sc, double mu, const double lam_g[8], double& cmax_out) {
  double Jc = 0.0, cmax = 0.0;
  const int N = in.N;
  // knots are dealt to the first TEAM lanes whatever the team width: the 8 partial sums and the tree below are
  // then bit-identical for an 8-lane team and a whole warp (lanes >= 8 contribute exact zeros), so a trial's
  // iteration path does not depend on where it runs (straggler hand-over, k3_wide_kernel)
  if (tm.lane() < TEAM)
    for (int k = tm.lane(); k < N - 1; k += TEAM) {
      const double* p = xu + (long long)k * 10;
      const double e8 = (in.Qd[7] != 0.0) ? (gptr(w.clk)[k] - in.xf[7]) : 0.0;
      add_stage_cost(in, o, sc, mu, p, e8, p + 7, gptr(w.lam) + (long long)k * 6, Jc, cmax);
    }
  if (tm.lane() == 0) add_terminal_cost(in, o, mu, xu + (long long)(N - 1) * 10, gptr(w.clk)[N - 1] - in.xf[7], lam_g, Jc, cmax);
  cmax_out = tm.max(cmax);
  return tm.sum(Jc);
}

// One batch of speculative line-search rollouts: lane a rolls out its own step size alpha; the
// per-knot inputs every lane needs (x_k,u_k | K_k,d_k | lambda_k | stage field vectors) are
// staged through shared memory in double-buffered 8-knot chunks (asynchronous copies issued one
// chunk ahead, so the ~1 us HBM/L2 latency is off the sequential critical path).
struct RollOut {
  double J, cmax;
  bool ok;
};
// The gradient measure of the convergence test, mean_k max_i |d_k,i| / (|u_k,i| + 1), of a STORED trajectory (the
// accepted line-search candidate, or the kept one when the line search is exhausted).  It used to be accumulated inside
// every speculative rollout (three |.|, a cross-multiplied maximum and a division per knot and candidate: 7 % of the
// rollout loop's instructions, needed for one candidate in 21).  Lane l evaluates knot base + l; the terms are then
// added up on the first TEAM lanes in ascending knot order per (k mod TEAM) class, whatever the team width, so the sum
// does not depend on where a trial runs.
template <class Team>
TS_FN double trajectory_grad(Team& tm, const ts_ilqr_opts_dev& o, const TrialWork& w, const double* xu, int N) {
  constexpr int W = Team::W;
  const int lane = tm.lane();
  double g = 0.0;
#ifdef __CUDA_ARCH__
#pragma unroll 4   // the loads of four steps in flight (the candidate was written a moment ago: L2 latency)
#endif
  for (int base = 0; base < N - 1; base += W) {
    const int k = base + lane;
    double m = 0.0;
    if (k < N - 1) {
      const double* p = xu + (long long)k * 10;
      const double* kd = gptr(w.kd) + (long long)k * 24;
      for (int i = 0; i < 3; ++i) m = fmax(m, fabs(kd[21 + i]) / (fabs(p[7 + i]) + 1.0));
    }
    for (int j = 0; j < W / TEAM; ++j) {
      const double mj = (W > TEAM) ? tm.bcast(m, (lane % TEAM) + TEAM * j) : m;
      if (lane < TEAM) g += mj;
    }
  }
  return tm.sum(g) / (double)(o.a3_grad_over_N ? N : N - 1);
}
template <class Team>
TS_FN void stage_chunk(Team& tm, const TrialWork& w, const double* xu_cur, int base, int N, double* buf) {
  const int k = base + tm.lane();
  if (k < N - 1) {
    double* dst = buf + tm.lane() * FWD_REC;
    tm.stage16(dst, xu_cur + (long long)k * 10, 5);
    tm.stage16(dst + 10, gptr(w.kd) + (long long)k * 24, 12);
    tm.stage16(dst + 34, gptr(w.lam) + (long long)k * 6, 3);
    tm.stage16(dst + 40, gptr(w.bk) + (long long)k * 10, 5);
  }
  tm.stage_commit();
}
template <class Team>
TS_FN_NOINLINE RollOut forward_batch(Team& tm, const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w, const double* xu_cur,
                                     double* xu_cand, bool live, double alpha, double sc, double mu, const double lam_g[8],
                                     double clk_absmax) {
  RollOut r;
  r.ok = live;
  double Jc = 0.0, cmax = 0.0;
  double xb[7];
  for (int i = 0; i < 7; ++i) xb[i] = in.x0[i];
  const int N = in.N;
  typedef SmL<Team::W> L;
  constexpr int W = Team::W;
  double* sm = tm.smem() + L::FWD;
  const int n_chunks = (N - 1 + W - 1) / W;
  const bool clk_bad = !(clk_absmax < o.max_state_value);   // the analytic clock state takes part in the max |x| test
  tm.sync();
  stage_chunk(tm, w, xu_cur, 0, N, sm);
  TS_NO_UNROLL
  for (int ch = 0; ch < n_chunks; ++ch) {
    const int base = ch * W;
    if (ch + 1 < n_chunks) {
      stage_chunk(tm, w, xu_cur, base + W, N, sm + ((ch + 1) & 1) * W * FWD_REC);
      tm.stage_wait(1);
    } else {
      tm.stage_wait(0);
    }
    tm.sync();
    const double* buf = sm + (ch & 1) * W * FWD_REC;
    int kk_n = N - 1 - base;
    if (kk_n > W) kk_n = W;
    if (r.ok) {
      TS_NO_UNROLL
      for (int kk = 0; kk < kk_n; ++kk) {
        const int k = base + kk;
        const double* p = buf + kk * FWD_REC;
        const double* kd = p + 10;
        double ub[3];
        double dx[7];
        if constexpr (team_quat<Team>::value) {   // quaternion_error(x, xbar), quaternion_toolbox.jl:63-75
          for (int i = 0; i < 3; ++i) dx[i] = xb[i] - p[i];
          const double qi[4] = {p[3], -p[4], -p[5], -p[6]};
          double qe[4];
          qmult(qi, xb + 3, qe);
          const double inv = 1.0 / (1.0 + qe[0]);
          for (int i = 0; i < 3; ++i) dx[3 + i] = qe[1 + i] * inv;
          dx[6] = 0.0;
        } else {
          for (int i = 0; i < 7; ++i) dx[i] = xb[i] - p[i];
        }
        for (int i = 0; i < 3; ++i) {
          double t = p[7 + i];
          for (int j = 0; j < 7; ++j) t += kd[j * 3 + i] * dx[j];
          t += alpha * kd[21 + i];
          ub[i] = t;
        }
        const double e8 = (in.Qd[7] != 0.0) ? (gptr(w.clk)[k] - in.xf[7]) : 0.0;
        add_stage_cost(in, o, sc, mu, xb, e8, ub, p + 34, Jc, cmax);
        double* q = xu_cand + (long long)k * 10;
        for (int i = 0; i < 7; ++i) q[i] = xb[i];
        for (int i = 0; i < 3; ++i) q[7 + i] = ub[i];
        double xn[7];
        rk3_step7<0, team_diagj<Team>::value>(in.I, xb, ub, p + 40, p + 43, p + 46, in.dt, xn);
        // max |x|, max |u| (NaN counts as infinite) against the limits, as ten predicate tests: a NaN fails `<`
        bool bad = clk_bad;
        for (int i = 0; i < 7; ++i) {
          xb[i] = xn[i];
          bad |= !(fabs(xn[i]) < o.max_state_value);
        }
        for (int i = 0; i < 3; ++i) bad |= !(fabs(ub[i]) < o.max_control_value);
        if (bad) {
          r.ok = false;
          break;
        }
      }
    }
    tm.sync();  // chunk buffer free for the copy issued two chunks ahead
  }
  if (r.ok) {
    double* q = xu_cand + (long long)(N - 1) * 10;
    for (int i = 0; i < 7; ++i) q[i] = xb[i];
    q[7] = q[8] = q[9] = 0.0;
    add_terminal_cost(in, o, mu, xb, gptr(w.clk)[N - 1] - in.xf[7], lam_g, Jc, cmax);
  }
  r.J = Jc;
  r.cmax = cmax;
  return r;
}

// ----------------------------------------------------------------------------------------
// Solver state of one trial between phases.  In the persistent kernel it lives in registers; in the
// phase-split ("phased") launch mode it is stored to / loaded from global memory between kernels.
enum { PH_BACKWARD = 0, PH_FORWARD = 1, PH_DONE = 2 };
struct TrialState {
  double mu, lam_g[8];
  double J_prev, J, J_true, c_max, c_max_prev, rho, drho, dV1, dV2, clk_absmax;
  long long cyc_bwd, cyc_fwd, cyc_lin;
  int it, outer, dJ_zero, inner_total, ls_total, status, cur, phase, b0, pad_;
};

// the trial's tables: clock trajectory + stage field vectors of every knot (sequential, exact replica); returns max |clock|
// in every lane.  Shared by a fresh start (solve_init) and a continuation (park_import_kernel, CS3).
template <class Team>
TS_FN double solve_tables(Team& tm, const TrialIn& in, const TrialWork& w) {
  const int N = in.N;
  double clk_absmax = 0.0;
  if (tm.lane() == 0) {
    double x8 = in.clk0;
    for (int k = 0; k < N - 1; ++k) {
      const ClockStep cs = clock_rk3(x8, in.clock_rate, in.dt);
      gptr(w.clk)[k] = x8;
      clk_absmax = fmax(clk_absmax, fabs(x8));
      const double tt[3] = {cs.t1, cs.t2, cs.t3};
      for (int s3 = 0; s3 < 3; ++s3) {
        const double* br = in.Bt + (long long)field_row(tt[s3], in.index_scale, in.B_rows) * 3;
        for (int c = 0; c < 3; ++c) gptr(w.bk)[(long long)k * 10 + s3 * 3 + c] = br[c];
      }
      gptr(w.bk)[(long long)k * 10 + 9] = 0.0;
      x8 = cs.next;
    }
    gptr(w.clk)[N - 1] = x8;
    clk_absmax = fmax(clk_absmax, fabs(x8));
  }
  return tm.bcast(clk_absmax, 0);
}

// setup: tables, multipliers, initial rollout, J_prev
template <class Team>
TS_FN void solve_init(Team& tm, const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w, TrialState& st) {
  const int lane = tm.lane();
  const int N = in.N;
  const double sc = o.stage_cost_dt ? in.dt : 1.0;
  const double clk_absmax = solve_tables(tm, in, w);
  for (int i = lane; i < (N - 1) * 6; i += Team::W) gptr(w.lam)[i] = 0.0;
  tm.sync();
  if (lane == 0) {
    double* xu = gptr(w.xu);
    double xb[7];
    for (int i = 0; i < 7; ++i) xb[i] = in.x0[i];
    for (int k = 0; k < N - 1; ++k) {
      double u[3];
      for (int i = 0; i < 3; ++i) u[i] = in.U0 ? in.U0[(long long)k * 3 + i] : 0.0;
      double* q = xu + (long long)k * 10;
      for (int i = 0; i < 7; ++i) q[i] = xb[i];
      for (int i = 0; i < 3; ++i) q[7 + i] = u[i];
      const double* b = gptr(w.bk) + (long long)k * 10;
      double xn[7];
      rk3_step7<0, team_diagj<Team>::value>(in.I, xb, u, b, b + 3, b + 6, in.dt, xn);
      for (int i = 0; i < 7; ++i) xb[i] = xn[i];
    }
    double* q = xu + (long long)(N - 1) * 10;
    for (int i = 0; i < 7; ++i) q[i] = xb[i];
    q[7] = q[8] = q[9] = 0.0;
  }
  tm.sync();
  st.mu = o.penalty_initial;
  for (int i = 0; i < 8; ++i) st.lam_g[i] = 0.0;
  st.status = ST_MAX_OUTER;
  st.outer = 1;
  st.inner_total = 0;
  st.ls_total = 0;
  st.rho = 0.0;
  st.drho = 0.0;
  st.it = 0;
  st.dJ_zero = 0;
  st.cur = 0;
  st.b0 = 0;
  st.pad_ = 0;
  st.dV1 = st.dV2 = 0.0;
  st.cyc_bwd = st.cyc_fwd = st.cyc_lin = 0;
  st.clk_absmax = clk_absmax;
  st.c_max = 0.0;
  st.c_max_prev = INFINITY;
  st.J_prev = trajectory_cost(tm, in, o, w, gptr(w.xu), sc, st.mu, st.lam_g, st.c_max);
  st.J = st.J_prev;
  st.J_true = st.J_prev;
  st.phase = (o.max_outer < 1) ? PH_DONE : PH_BACKWARD;
}

// start of the next outer iteration on the trajectory xu_c, after an outer update (mu, lam_g and the bound multipliers
// already updated).  Also the resume step of a continued solve (CS3, park_import_kernel).
template <class Team>
TS_FN void solve_next_outer(Team& tm, const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w, TrialState& st,
                            const double* xu_c, double sc) {
  ++st.outer;
  st.it = 0;
  st.dJ_zero = 0;
  st.rho = 0.0;
  st.drho = 0.0;
  double cm;
  // J_true: the current trajectory's cost under the NEW multipliers; J_prev: the line-search reference of the next
  // iteration -- the same number in the default reading, the carried-over cost under A7
  st.J_true = trajectory_cost(tm, in, o, w, xu_c, sc, st.mu, st.lam_g, cm);
  st.J_prev = o.a7_carry_cost ? st.J : st.J_true;
}

// inner-iteration bookkeeping once a forward pass has produced (Jn, grad): convergence tests, outer AL update
template <class Team>
TS_FN void solve_after_forward(Team& tm, const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w, TrialState& st,
                               double Jn, double grad) {
  const int lane = tm.lane();
  const int N = in.N;
  const double sc = o.stage_cost_dt ? in.dt : 1.0;
  const bool last = (st.outer == o.max_outer) || o.a4_no_intermediate;
  const double ctol = last ? o.cost_tol : o.cost_tol_intermediate;
  const double gtol = last ? o.grad_tol : o.grad_tol_intermediate;
  st.phase = PH_BACKWARD;
  st.b0 = 0;
  bool inner_done = false;
  if (!(Jn == Jn)) {
    st.status = ST_NAN;
    st.J = Jn;
    st.phase = PH_DONE;
    return;
  }
  if (Jn > o.max_cost_value) {
    st.status = ST_COST_BLOWUP;
    st.J = Jn;
    st.phase = PH_DONE;
    return;
  }
  const double dJ = fabs(Jn - st.J_prev);
  st.J_prev = Jn;
  if (dJ == 0.0) ++st.dJ_zero; else st.dJ_zero = 0;
  if ((0.0 < dJ && dJ < ctol) || grad < gtol || st.dJ_zero > o.dJ_counter_limit || st.it >= o.max_inner) inner_done = true;
  st.J = Jn;
  if (!inner_done) return;
  // ---- outer update: duals (A5), penalty (A6), convergence
  const double* xu_c = xu_buf<Team::W>(w, st.cur);
  for (int k = lane; k < N - 1; k += Team::W) {
    double c6[6];
    bound_c(o, xu_c + (long long)k * 10 + 7, c6);
    double* lam = gptr(w.lam) + (long long)k * 6;
    for (int i = 0; i < 6; ++i) {
      const double l0 = lam[i];
      double l = l0 + st.mu * c6[i];
      l = fmin(fmax(l, -o.dual_max), o.dual_max);
      if (o.a5_dual_active_only && !((c6[i] > active_threshold(o)) || (l0 > 0.0))) l = l0;
      lam[i] = fmax(0.0, l);
    }
  }
  for (int i = 0; i < 8; ++i) {
    if (!(o.goal_mask & (1 << i))) continue;
    const double e = ((i < 7) ? xu_c[(long long)(N - 1) * 10 + i] : gptr(w.clk)[N - 1]) - in.xf[i];
    const double l = st.lam_g[i] + st.mu * e;
    st.lam_g[i] = fmin(fmax(l, -o.dual_max), o.dual_max);
  }
  if (!o.a6_penalty_conditional || st.c_max > o.constraint_decrease_ratio * st.c_max_prev)
    st.mu = fmin(st.mu * o.penalty_scaling, o.penalty_max);
  st.c_max_prev = st.c_max;
  tm.sync();
  if (st.c_max < o.constraint_tol) {
    st.status = ST_CONVERGED;
    st.phase = PH_DONE;
  } else if (st.outer >= o.max_outer) {
    st.phase = PH_DONE;
  } else {
    solve_next_outer(tm, in, o, w, st, xu_c, sc);
  }
}

// phase BACKWARD: one Riccati sweep (with regularisation restarts)
template <class Team>
TS_FN void solve_backward(Team& tm, const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w, TrialState& st) {
  const double sc = o.stage_cost_dt ? in.dt : 1.0;
  ++st.it;
  ++st.inner_total;
  const long long t0 = ts_clock();
  Reg reg;
  reg.rho = st.rho;
  reg.drho = st.drho;
  const bool ok = backward_pass(tm, in, o, w, xu_buf<Team::W>(w, st.cur), sc, st.mu, st.lam_g, reg, st.dV1, st.dV2, st.cyc_lin);
  st.rho = reg.rho;
  st.drho = reg.drho;
  st.cyc_bwd += ts_clock() - t0;
  if (!ok) {
    st.status = ST_REG_MAX;
    st.phase = PH_DONE;
    return;
  }
  tm.sync();  // gains visible to every lane
  st.phase = PH_FORWARD;
  st.b0 = 0;
}

// phase FORWARD: one batch of 8 speculative line-search candidates c = b0 + lane, alpha = 2^-c
template <class Team>
TS_FN void solve_forward(Team& tm, const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w, TrialState& st) {
  const int lane = tm.lane();
  const int N = in.N;
  const double sc = o.stage_cost_dt ? in.dt : 1.0;
  const long long t0 = ts_clock();
  const double* xu_cur = xu_buf<Team::W>(w, st.cur);
  const int n_cand = o.max_linesearch + 1;
  const int c = st.b0 + lane;
  const bool live = (c < n_cand);
  const int bufi = (lane < st.cur) ? lane : lane + 1;
  double alpha = 1.0;
  for (int i = 0; i < c; ++i) alpha /= 2.0;
  const RollOut r = forward_batch(tm, in, o, w, xu_cur, xu_buf<Team::W>(w, bufi), live, alpha, sc, st.mu, st.lam_g, st.clk_absmax);
  bool acc = false;
  if (live && r.ok) {
    const double expected = -alpha * (st.dV1 + alpha * st.dV2);
    const double z = (expected > 0.0) ? (st.J_prev - r.J) / expected : -1.0;
    acc = !((z <= o.ls_lower || z > o.ls_upper) && (r.J >= st.J_prev));
  }
  const unsigned bits = tm.ballot(acc);
  if (bits) {
    int a = 0;
    while (!((bits >> a) & 1u)) ++a;
    st.ls_total += st.b0 + a + 1;
    const double Jn = tm.bcast(r.J, a);
    st.c_max = tm.bcast(r.cmax, a);
    st.cur = (a < st.cur) ? a : a + 1;
    tm.sync();   // the accepted lane's trajectory is visible to the team
    const double grad = trajectory_grad(tm, o, w, xu_buf<Team::W>(w, st.cur), N);
    st.cyc_fwd += ts_clock() - t0;
    solve_after_forward(tm, in, o, w, st, Jn, grad);
    return;
  }
  tm.sync();
  st.b0 += Team::W;
  if (st.b0 < n_cand) {  // next batch of candidates
    st.cyc_fwd += ts_clock() - t0;
    return;
  }
  // line search exhausted: keep the trajectory, raise the regularisation (App. C step 4)
  st.ls_total += n_cand;
  Reg reg;
  reg.rho = st.rho;
  reg.drho = st.drho;
  reg_increase(o, reg);
  reg.rho += o.bp_reg_fp;
  st.rho = reg.rho;
  st.drho = reg.drho;
  const double grad = trajectory_grad(tm, o, w, xu_cur, N);
  st.cyc_fwd += ts_clock() - t0;
  // the kept trajectory's cost under the current multipliers (the oracle re-evaluates al_cost of the unchanged
  // trajectory): J_prev, except in the first iteration of an inner solve under A7, where J_prev is the carried-over value
  solve_after_forward(tm, in, o, w, st, (st.it == 1) ? st.J_true : st.J_prev, grad);
}

TS_HD void solve_finish(const TrialIn& in, const TrialState& st, ts_trial_outcome_dev& out) {
  out.status = st.status;
  out.outer_iters = st.outer;
  out.inner_iters = st.inner_total;
  out.ls_rollouts = st.ls_total;
  out.N = in.N;
  out.J = st.J;
  out.c_max = st.c_max;
  out.t_final = 0.0;    // filled by the fused Monte-Carlo path; the low-level solve has no field pass / replay
  out.slew_time = 0.0;
  out.flops = 0.0;
}
// CS1: the exported state of a finished trial is what the solver holds after its final outer update (at a MAX_OUTER end
// solve_after_forward has applied the dual, goal-multiplier and penalty updates before it stops)
TS_HD void solve_export(const TrialState& st, ts_al_state_dev& s) {
  s.mu = st.mu;
  for (int i = 0; i < 8; ++i) s.lam_goal[i] = st.lam_g[i];
  s.J = st.J;
  s.c_max = st.c_max;
  s.status = st.status;
  s.outer_iters = st.outer;
  s.inner_iters = st.inner_total;
  s.ls_rollouts = st.ls_total;
}
// CS3: resume a trial exported at a MAX_OUTER end.  Expects the trajectory in buffer 0 of w and the bound multipliers in
// w.lam; rebuilds the tables as solve_init does and then runs the start of the next outer iteration exactly as
// solve_after_forward does.  Counters and costs carry on from the exported values.
template <class Team>
TS_FN void solve_import(Team& tm, const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w, const ts_al_state_dev& s,
                        TrialState& st) {
  st.clk_absmax = solve_tables(tm, in, w);
  tm.sync();
  st.mu = s.mu;
  for (int i = 0; i < 8; ++i) st.lam_g[i] = s.lam_goal[i];
  st.J = s.J;
  st.c_max = s.c_max;
  st.c_max_prev = s.c_max;
  st.status = ST_MAX_OUTER;
  st.outer = s.outer_iters;
  st.inner_total = s.inner_iters;
  st.ls_total = s.ls_rollouts;
  st.cur = 0;
  st.b0 = 0;
  st.pad_ = 0;
  st.dV1 = st.dV2 = 0.0;
  st.cyc_bwd = st.cyc_fwd = st.cyc_lin = 0;
  st.phase = PH_BACKWARD;
  solve_next_outer(tm, in, o, w, st, xu_buf<Team::W>(w, 0), o.stage_cost_dt ? in.dt : 1.0);
}
// per-trial SM-cycle diagnostics (ts_k3_last_cycles): backward pass, forward pass, linearisation share of the backward pass
TS_HD void solve_diag(const TrialState& st, double* diag3) {
  diag3[0] = (double)st.cyc_bwd;
  diag3[1] = (double)st.cyc_fwd;
  diag3[2] = (double)st.cyc_lin;
}

// The whole solve as one loop over phases (persistent-kernel mode and the host lane-emulator).
template <class Team>
TS_FN void alilqr_solve_team(Team& tm, const TrialIn& in, const ts_ilqr_opts_dev& o, const TrialWork& w,
                             ts_trial_outcome_dev& out, int& cur_out) {
  TrialState st;
  solve_init(tm, in, o, w, st);
  // One loop iteration = one iLQR iteration: a backward sweep, then forward batches until a step is
  // taken.  Keeping this shape (rather than "run whatever phase I am in") keeps the four teams of a warp
  // in the same phase: a team that needs an extra line-search batch makes its siblings wait at the
  // reconvergence point instead of drifting into the other phase (which would serialise both code paths).
  while (st.phase != PH_DONE) {
    if (st.phase == PH_BACKWARD) solve_backward(tm, in, o, w, st);
    while (st.phase == PH_FORWARD) solve_forward(tm, in, o, w, st);
  }
  solve_finish(in, st, out);
  cur_out = st.cur;
  tm.sync();
}

}  // namespace ts
