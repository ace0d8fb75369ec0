// K4 -- batched TVLQR replay in four launches (tvlqr_solver.cuh): K4a linearisation, one thread per (trial, knot);
// K4b backward Riccati sweep, one thread per trial; K4n stage records (noise, perturbation quaternions, field rows), one
// thread per (trial, step, stage); K4c closed-loop replay, one thread per trial -- plus the eigen-axis-slew /
// Bryson-weight preparation kernel.
//   attitude_simulation(...)      reference src/attitude_controller.jl:1-48 (+ :50-145)
//   eigen_axis_slew(x0,xf,t)      src/eigen_axis_slew.jl:1-38
//   Bryson weights                src/TortoiseSat.jl:157-168, src/monte_carlo.jl:165-176
// Round 1 ran all three phases in one thread per trial (255 registers, 5.5 KB of stack, 80 ms per 4096 trials and
// 780 ms on the ragged sweep): the Jacobians were 70% of the work and sat inside the sequential scan.  They are now
// their own fully parallel launch, and the two sequential scans are light (6x6 blocks, no spills in the loop).
#pragma once
#include "common.cuh"
#include "tvlqr_solver.cuh"

namespace ts {

struct K4Args {
  int64_t n_trials;
  const int64_t* N_i;
  const int64_t* offs;
  const double* X_lqr;   // ragged N x 8 at offs*8
  const double* U_lqr;   // ragged (N-1) x 3 at offs*3
  const double* x0_lqr;  // 8 per trial
  const double* Jmat;    // 9
  const double* B_eci;
  const int64_t* B_offs;
  const int64_t* B_rows;
  const double* index_scale;
  const double* clock_rate;
  const double* t_final;      // per trial (tf of t_sim and the "fail" sentinel)
  const double* q_final;      // 4 per trial
  const uint32_t* stream_id;  // Philox stream per trial (global trial id), nullable -> t
  ts_tvlqr_opts_dev opts;
  const double* noise;   // explicit: ragged (N x 36) at offs*36, nullable
  double* X_sim;         // nullable, ragged N x 8
  double* U_sim;         // nullable, ragged N x 3
  double* dX;            // nullable, ragged N x 6
  double* K;             // ragged N x 18 (scratch if the caller passes none)
  int64_t* N_sim;        // nullable
  double* slew_time;     // nullable
  // linearisation scratch: AB[lin_total x 54] = projected (A 6x6 | B 6x3) per knot, lin_offs[t] = first knot of trial t
  double* AB;
  double* clk;             // [lin_total] replay clock state per step (written by K4b, read by K4n)
  const int64_t* lin_offs;
  int64_t lin_total;
};

// ---- K4a: the linearisation, one thread per (trial, knot) -- ~70% of the replay's FLOPs and embarrassingly parallel
// over knots (every knot's Jacobian depends only on the optimised trajectory).  lin_offs[t] = sum_{t' < t} (N_t' - 1).
__global__ void __launch_bounds__(128) k4a_linearise_kernel(const K4Args a) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.lin_total) return;
  // trial of knot g: largest t with lin_offs[t] <= g
  int64_t lo = 0, hi = a.n_trials - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (a.lin_offs[mid] <= g) lo = mid; else hi = mid - 1;
  }
  const int64_t t = lo;
  const int64_t k = g - a.lin_offs[t];
  Inertia I;
  for (int i = 0; i < 9; ++i) I.J[i] = a.Jmat[t * 9 + i];
  inv3_gj(I.J, I.Jinv);
  const double* X = a.X_lqr + a.offs[t] * 8;
  const double* U = a.U_lqr + a.offs[t] * 3;
  const double h = a.opts.dt_squared ? a.opts.dt * a.opts.dt : a.opts.dt;
  double AB[54];
  tvlqr_linearise_knot(I, X + k * 8, X + (k + 1) * 8, U + k * 3, a.B_eci + a.B_offs[t] * 3, a.B_rows[t], a.index_scale[t],
                       a.clock_rate[t], h, AB);
  double* o = a.AB + g * 54;
  for (int i = 0; i < 54; ++i) o[i] = AB[i];
}

// ---- per-thread staging ring for the two sequential kernels.  One thread owns one slew and walks its knots in order; what
// a knot needs (54 doubles of [A|B] for the Riccati step, 69 for a replay step) sits in arrays laid out per slew, so the
// 32 threads of a warp touch 32 unrelated addresses per load and every knot used to wait out several DRAM round trips
// (ncu on the round-2 first cut: long-scoreboard 81 % of the replay's warp-cycles, ~10 k cycles per knot).  Each thread
// now copies the inputs of the knot K4_RING_D steps ahead into its own slice of shared memory with 8-byte cp.async and
// waits only for the oldest copy: the DRAM latency is off the dependent chain.  (W odd: the lanes' slices start on
// different banks.)
constexpr int K4_RING_D = 4;
constexpr int K4B_W = 55;   // 54 used
constexpr int K4C_W = 71;   // 8 + 18 + 40 + 3 = 69 used
constexpr int K4B_SMEM_BYTES = K4_RING_D * 32 * K4B_W * 8;
constexpr int K4C_SMEM_BYTES = K4_RING_D * 32 * K4C_W * 8;
__device__ __forceinline__ void k4_cp8(double* dst_smem, const double* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"((unsigned)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void k4_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void k4_wait_oldest() { asm volatile("cp.async.wait_group %0;\n" ::"n"(K4_RING_D - 1) : "memory"); }

// ---- K4b: the backward Riccati sweep (sequential in k), one thread per trial, over the stored linearisations
__global__ void __launch_bounds__(32) k4b_riccati_kernel(const K4Args a) {
  extern __shared__ __align__(16) double k4_smem[];
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.n_trials) return;
  const int N = (int)a.N_i[t];
  double S[36];
  for (int i = 0; i < 36; ++i) S[i] = 0.0;
  for (int i = 0; i < 6; ++i) S[i * 6 + i] = a.opts.Qfd[i];
  const double* ab = a.AB + a.lin_offs[t] * 54;
  double* K = a.K + a.offs[t] * 18;
  double* ring = k4_smem + threadIdx.x * K4B_W;
  auto issue = [&](int k) {   // knot k -> slot (k mod D); an empty group when k is out of range keeps the group count uniform
    if (k >= 0) {
      double* dst = ring + (k % K4_RING_D) * 32 * K4B_W;
      const double* src = ab + (long long)k * 54;
#pragma unroll
      for (int i = 0; i < 54; ++i) k4_cp8(dst + i, src + i);
    }
    k4_commit();
  };
  for (int d = 0; d < K4_RING_D; ++d) issue(N - 2 - d);
#pragma unroll 1
  for (int k = N - 2; k >= 0; --k) {
    k4_wait_oldest();
    tvlqr_riccati_step(a.opts, ring + (k % K4_RING_D) * 32 * K4B_W, S, K + (long long)k * 18);
    issue(k - K4_RING_D);
  }
  // the replay's clock state at every step (the reference accumulates it through rk4: sequential, exact replica), so
  // that K4n can look the stage field rows up in parallel
  double x8 = a.x0_lqr[t * 8 + 7];
  double* clk = a.clk + a.lin_offs[t];
#pragma unroll 1
  for (int k = 0; k < N - 1; ++k) {
    clk[k] = x8;
    double tcl[4], nxt;
    clock_rk4(x8, a.clock_rate[t], a.opts.dt, tcl, nxt);
    x8 = nxt;
  }
}

// ---- K4b as a TEAM kernel: 16 lanes per slew (two slews per warp).  The Riccati step is a chain of small dense products
// whose columns are independent: lane c < 6 owns column c of A (S A, B'S A, its gain column, its closed-loop column,
// S Acl, its column of the new S), lanes 6..8 own the columns of B (S B, B'S B); three exchanges through the team's
// shared memory per step (B'SB | K, Acl | new S).  Every dot product keeps the summation order of tvlqr_riccati_step, so
// the gains are bit-identical to the one-thread version (which the host emulator and the oracle tests run); one thread
// per slew needed ~1200 dependent-issue FMAs per knot (2.6 k cycles), a lane of the team ~220.  [A|B] records are staged
// K4_RING_D steps ahead by the team's lanes with 16-byte cp.async (27 pieces per record).
constexpr int K4B_TEAM = 16;
constexpr int K4B_TEAMS_PER_BLOCK = 4;
constexpr int K4B_XB = K4_RING_D * 54;                 // exchange area behind the ring: BSB 9 (+pad) | K 18 (+pad) | Acl 36 | Sn 36
constexpr int K4B_TEAM_DOUBLES = K4B_XB + 12 + 20 + 36 + 36;
static_assert(K4B_TEAM_DOUBLES % 2 == 0 && (K4B_XB % 2) == 0, "16-byte alignment of the team regions");
__global__ void __launch_bounds__(K4B_TEAM * K4B_TEAMS_PER_BLOCK) k4b_riccati_team_kernel(const K4Args a) {
  __shared__ __align__(16) double sm_all[K4B_TEAMS_PER_BLOCK * K4B_TEAM_DOUBLES];
  const int team = threadIdx.x / K4B_TEAM, c = threadIdx.x % K4B_TEAM;
  const int64_t t = (int64_t)blockIdx.x * K4B_TEAMS_PER_BLOCK + team;
  if (t >= a.n_trials) return;   // the whole team leaves together
#define K4B_QD(i) a.opts.Qd[i]
#define K4B_QFD(i) a.opts.Qfd[i]
#define K4B_RD(i) a.opts.Rd[i]
#define K4B_GAINS a.K
#define K4B_CLOCK true
#include "k4b_riccati_body.inc"
}

// ---- K4w gains: K4b's team step with one team per (slew, weighting) of a weight-sweep ensemble (ts_mc_weight_ensemble,
// WE2 of DESIGN.md section 4, K4).  The teams of one slew are adjacent and share its [A|B] records in L2.  Team (t, w)
// reads weighting w (Qd 6 | Qfd 6 | Rd 3 doubles at sets + 15 w) into registers and writes its gains at K + w k_stride +
// offs[t] * 18; the team of weighting 0 alone writes the slew's replay clock sequence.
struct K4wGainsArgs {
  K4Args a;                          // the selected slews' K4 arguments (a.K unused)
  const double* sets;                // n_sets x 15
  int64_t n_sets, k_stride;          // k_stride: doubles per weighting's gains region
  double* K;
};
__global__ void __launch_bounds__(K4B_TEAM * K4B_TEAMS_PER_BLOCK) k4w_riccati_sets_kernel(const K4wGainsArgs aw) {
  __shared__ __align__(16) double sm_all[K4B_TEAMS_PER_BLOCK * K4B_TEAM_DOUBLES];
  const K4Args& a = aw.a;
  const int team = threadIdx.x / K4B_TEAM, c = threadIdx.x % K4B_TEAM;
  const int64_t g = (int64_t)blockIdx.x * K4B_TEAMS_PER_BLOCK + team;
  if (g >= a.n_trials * aw.n_sets) return;   // the whole team leaves together
  const int64_t t = g / aw.n_sets, ws = g - t * aw.n_sets;
  double wq[15];
#pragma unroll
  for (int i = 0; i < 15; ++i) wq[i] = aw.sets[ws * 15 + i];
#define K4B_QD(i) wq[i]
#define K4B_QFD(i) wq[6 + (i)]
#define K4B_RD(i) wq[12 + (i)]
#define K4B_GAINS (aw.K + ws * aw.k_stride)
#define K4B_CLOCK (ws == 0)
#include "k4b_riccati_body.inc"
}

// ---- K4n: the stage records of the replay (tvlqr_solver.cuh): for every rk4 stage of every step the disturbance draws of
// simulator.jl:5,10,22 (Philox4x32-10 + Box-Muller, counter-based on (seed, trial, step, stage)), the perturbation
// quaternion (sincos) and the perturbed field row of the stage's clock value -- one thread per (trial, step, stage).  In
// round 1 all of this sat inside the sequential replay, where FP64 log / sincos / divisions were ~80% of its instructions.
// The records (40 doubles per step) overwrite the linearisation scratch (54 per step), which K4b has consumed by then.
__global__ void __launch_bounds__(128) k4n_records_kernel(const K4Args a) {
  const int64_t g4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t g = g4 >> 2;
  const int s4 = (int)(g4 & 3);
  if (g >= a.lin_total) return;
  int64_t lo = 0, hi = a.n_trials - 1;
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (a.lin_offs[mid] <= g) lo = mid; else hi = mid - 1;
  }
  const int64_t t = lo;
  const int64_t k = g - a.lin_offs[t];
  double tcl[4], nxt;
  clock_rk4(a.clk[g], a.clock_rate[t], a.opts.dt, tcl, nxt);
  const double* Bn = a.B_eci + (a.B_offs[t] + field_row(tcl[s4], a.index_scale[t], a.B_rows[t])) * 3;
  double nzb[9];
  const double* nz = nullptr;
  if (a.opts.noise_mode == 1) nz = a.noise + a.offs[t] * 36 + (k * 4 + s4) * 9;
  if (a.opts.noise_mode == 2) {
    tvlqr_noise(a.opts.seed, a.stream_id ? a.stream_id[t] : (uint32_t)t, (uint32_t)k, (uint32_t)s4, nzb);
    nz = nzb;
  }
  double rec[TV_REC];
  tvlqr_stage_record(nz, Bn, rec);
  double* o = a.AB + a.lin_offs[t] * 54 + (k * 4 + s4) * TV_REC;
  for (int i = 0; i < TV_REC; ++i) o[i] = rec[i];
}

// ---- K4c: the closed-loop replay (sequential in k) + slew-time rule, one thread per trial
struct K4cRingSrc {   // the replay's input policy (tvlqr_replay_src): step k from the staging ring, step k + D requested behind it
  const double *X, *U, *K, *recs;
  double* ring;
  long long n_steps;   // steps 0 .. N-2 have inputs
  __device__ __forceinline__ void issue(long long k) const {
    if (k < n_steps) {
      double* dst = ring + (int)(k % K4_RING_D) * 32 * K4C_W;
      const double* x = X + k * 8;
      const double* g = K + k * 18;
      const double* r = recs + k * (4 * TV_REC);
      const double* u = U + k * 3;
#pragma unroll
      for (int i = 0; i < 8; ++i) k4_cp8(dst + i, x + i);
#pragma unroll
      for (int i = 0; i < 18; ++i) k4_cp8(dst + 8 + i, g + i);
#pragma unroll
      for (int i = 0; i < 4 * TV_REC; ++i) k4_cp8(dst + 26 + i, r + i);
#pragma unroll
      for (int i = 0; i < 3; ++i) k4_cp8(dst + 26 + 4 * TV_REC + i, u + i);
    }
    k4_commit();
  }
  __device__ __forceinline__ void fetch(long long k, const double*& xr, const double*& Kk, const double*& ul, const double*& rk) const {
    k4_wait_oldest();
    const double* p = ring + (int)(k % K4_RING_D) * 32 * K4C_W;
    xr = p;
    Kk = p + 8;
    rk = p + 26;
    ul = p + 26 + 4 * TV_REC;
  }
  __device__ __forceinline__ void done(long long k) const { issue(k + K4_RING_D); }
};
static_assert(4 * TV_REC == 40 && 26 + 4 * TV_REC + 3 <= K4C_W, "replay staging slot layout");
__global__ void __launch_bounds__(32) k4c_replay_kernel(const K4Args a) {
  extern __shared__ __align__(16) double k4_smem[];
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.n_trials) return;
  TvlqrIn in;
  in.N = (int)a.N_i[t];
  in.X_lqr = a.X_lqr + a.offs[t] * 8;
  in.U_lqr = a.U_lqr + a.offs[t] * 3;
  for (int i = 0; i < 8; ++i) in.x0[i] = a.x0_lqr[t * 8 + i];
  for (int i = 0; i < 9; ++i) in.I.J[i] = a.Jmat[t * 9 + i];
  inv3_gj(in.I.J, in.I.Jinv);
  in.Bt = a.B_eci + a.B_offs[t] * 3;
  in.B_rows = a.B_rows[t];
  in.index_scale = a.index_scale[t];
  in.clock_rate = a.clock_rate[t];
  in.noise = a.noise ? a.noise + a.offs[t] * 36 : nullptr;
  in.trial = a.stream_id ? a.stream_id[t] : (uint32_t)t;
  for (int i = 0; i < 4; ++i) in.q_final[i] = a.q_final[t * 4 + i];
  in.t_final = a.t_final[t];
  in.time_step = a.opts.dt;
  in.trial_index_1based = (long long)in.trial + 1;
  ts_tvlqr_opts_dev o = a.opts;
  o.tf = a.t_final[t];
  K4cRingSrc src;
  src.X = in.X_lqr;
  src.U = in.U_lqr;
  src.K = a.K + a.offs[t] * 18;
  src.recs = a.AB + a.lin_offs[t] * 54;
  src.ring = k4_smem + threadIdx.x * K4C_W;
  src.n_steps = in.N - 1;
  for (int d = 0; d < K4_RING_D; ++d) src.issue(d);
  double slew = 0.0;
  const long long ns = tvlqr_replay_src<true>(in, o, src, a.X_sim ? a.X_sim + a.offs[t] * 8 : nullptr, a.U_sim ? a.U_sim + a.offs[t] * 3 : nullptr,
                                              a.dX ? a.dX + a.offs[t] * 6 : nullptr, &slew);
  asm volatile("cp.async.wait_all;\n" ::: "memory");   // copies requested past the last simulated step
  if (a.N_sim) a.N_sim[t] = ns;
  if (a.slew_time) a.slew_time[t] = slew;
}

// host: the three launches of K4 (a.AB / a.lin_offs / a.lin_total must be set)
// Zeroes the X_sim / U_sim rows of the trials about to be replayed again (ts_mc_continue): one block per trial.  A
// replay writes only its first N_sim rows, and the kept arrays promise zeros from there on.
__global__ void __launch_bounds__(256) k4_clear_rows_kernel(int64_t n_trials, const int64_t* N_i, const int64_t* offs, double* X_sim,
                                                            double* U_sim) {
  const int64_t t = blockIdx.x;
  if (t >= n_trials) return;
  double* xs = X_sim + offs[t] * 8;
  double* us = U_sim + offs[t] * 3;
  const int64_t n8 = N_i[t] * 8, n3 = N_i[t] * 3;
  for (int64_t i = threadIdx.x; i < n8; i += blockDim.x) xs[i] = 0.0;
  for (int64_t i = threadIdx.x; i < n3; i += blockDim.x) us[i] = 0.0;
}

// K4a + K4b: the gains and the replay clock sequence
inline void k4_gains_launch(ts_ctx* c, const K4Args& a) {
  if (a.lin_total > 0) k4a_linearise_kernel<<<(unsigned)((a.lin_total + 127) / 128), 128, 0, c->stream>>>(a);
  // (a per-device attribute: set on every launch -- ts_create_multi drives several devices from one process)
  cudaFuncSetAttribute(k4b_riccati_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, K4B_SMEM_BYTES);
  cudaFuncSetAttribute(k4c_replay_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, K4C_SMEM_BYTES);
  if (a.lin_total > 0)
    k4b_riccati_team_kernel<<<(unsigned)((a.n_trials + K4B_TEAMS_PER_BLOCK - 1) / K4B_TEAMS_PER_BLOCK), K4B_TEAM * K4B_TEAMS_PER_BLOCK, 0,
                              c->stream>>>(a);
  else
    k4b_riccati_kernel<<<(unsigned)((a.n_trials + 31) / 32), 32, K4B_SMEM_BYTES, c->stream>>>(a);
  c->launches += 2;
}

inline void k4_launch(ts_ctx* c, const K4Args& a) {
  k4_gains_launch(c, a);
  if (a.lin_total > 0) k4n_records_kernel<<<(unsigned)((4 * a.lin_total + 127) / 128), 128, 0, c->stream>>>(a);
  k4c_replay_kernel<<<(unsigned)((a.n_trials + 31) / 32), 32, K4C_SMEM_BYTES, c->stream>>>(a);
  c->launches += 2;
}

// ---- K4e: the disturbance ensemble of a kept Monte-Carlo run (ts_mc_replay_ensemble, RE1-RE5 of DESIGN.md section 4,
// K4).  One warp per (slew, 32 consecutive realisations), one realisation per lane, warps of the longest slews first.
// The reference row, the gain, the reference control and the clock state of a step (K4b's sequence) are the same for
// every lane: the warp stages them K4_RING_D steps ahead into one shared slot per step (30 doubles, one 8-byte cp.async
// per lane) and the lanes read them by broadcast.  The clock state is noise-free, so the four stage field rows are the
// same for every lane too (uniform loads).  The stage records cannot be pre-generated as K4n does (40 doubles per step
// and realisation): each lane builds its own at the step, with K4n's Philox / Box-Muller / stage-record code and its
// realisation's counters, into its own slice of shared memory (one stage at a time, so the draws never compete with
// the integration for registers), and then runs K4c's replay step and slew-time rule on them (tvlqr_replay_src<true>).
// Stored and reloaded like K4n's records, the draws enter the integration exactly as in the kept run (RE3).
constexpr int K4E_W = 32;            // ring slot: x_ref 8 | K 18 | u_ref 3 | clock 1
constexpr int K4E_R = 4 * TV_REC + 1;   // a lane's stage records (odd stride: 64-bit accesses without bank conflicts)
constexpr int K4E_WARPS = 4;
struct K4eArgs {
  int64_t n_sel;                     // selected active trials, compacted (longest horizon first)
  const int64_t *N_i, *offs, *B_offs, *B_rows;
  const double *X_lqr, *U_lqr, *K;   // kept trajectories (knot offsets offs), gains of K4a + K4b
  const double* clk;                 // K4b's replay clock sequence, at lin_offs
  const int64_t* lin_offs;
  const double *x0, *x0_lqr, *Jmat, *B_eci, *index_scale, *clock_rate, *t_final, *q_final;
  const uint32_t* stream_id;
  ts_tvlqr_opts_dev opts;            // the run's options after the fused path's overrides, noise_mode 2
  int64_t n_real, r_first, n_blk;    // n_blk = ceil(n_real / 32) warps per trial
  double q_noise_scale;
  double* slew_time;                 // n_sel x n_real
  double* x_final;                   // n_sel x n_real x 8, nullable
};
// The K4e arguments over the trials, kept trajectories, gains and options of a's replay (x0: the trials' unperturbed
// initial states); the realisations and the outputs are left to the caller.
inline K4eArgs k4e_args(const K4Args& a, const double* x0) {
  K4eArgs e;
  e.n_sel = a.n_trials; e.N_i = a.N_i; e.offs = a.offs; e.B_offs = a.B_offs; e.B_rows = a.B_rows;
  e.X_lqr = a.X_lqr; e.U_lqr = a.U_lqr; e.K = a.K;
  e.clk = a.clk; e.lin_offs = a.lin_offs;
  e.x0 = x0; e.x0_lqr = a.x0_lqr; e.Jmat = a.Jmat; e.B_eci = a.B_eci; e.index_scale = a.index_scale;
  e.clock_rate = a.clock_rate; e.t_final = a.t_final; e.q_final = a.q_final; e.stream_id = a.stream_id;
  e.opts = a.opts;
  return e;
}
template <bool DISP>
struct K4eWarpSrc {
  const TvlqrIn* in;
  const ts_tvlqr_opts_dev* o;
  const double *X, *U, *K, *clk;
  double* ring;                      // this warp's K4_RING_D slots of K4E_W doubles
  double* recs;                      // this lane's K4E_R doubles
  long long n_steps;
  int lane;
  __device__ __forceinline__ void issue(long long k) const {
    if (k < n_steps && lane < 30) {
      const double* src = lane < 8 ? X + k * 8 + lane
                        : lane < 26 ? K + k * 18 + (lane - 8)
                        : lane < 29 ? U + k * 3 + (lane - 26)
                                    : clk + k;
      k4_cp8(ring + (int)(k % K4_RING_D) * K4E_W + lane, src);
    }
    k4_commit();
  }
  __device__ __forceinline__ void fetch(long long k, const double*& xr, const double*& Kk, const double*& ul, const double*& rk) const {
    k4_wait_oldest();
    __syncwarp();                    // the other lanes' copies of slot k are complete and visible
    const double* p = ring + (int)(k % K4_RING_D) * K4E_W;
    double tcl[4], nxt;
    clock_rk4(p[29], in->clock_rate, o->dt, tcl, nxt);
#pragma unroll 1
    for (int s = 0; s < 4; ++s) {
      double rec[TV_REC];
      const double tc = s == 0 ? tcl[0] : (s == 3 ? tcl[3] : tcl[1]);   // (no dynamic index: tcl stays in registers)
      tvlqr_stage_record_at<DISP>(*in, *o, k, s, tc, rec);
#pragma unroll
      for (int i = 0; i < TV_REC; ++i) recs[s * TV_REC + i] = rec[i];
    }
    xr = p;
    Kk = p + 8;
    ul = p + 26;
    rk = recs;
  }
  __device__ __forceinline__ void done(long long k) const {
    __syncwarp();                    // every lane has read slot k: it may be refilled
    issue(k + K4_RING_D);
  }
};
// K4d: the dispersion ensemble of a kept run (ts_mc_dispersion_ensemble, DE1-DE6): K4e's layout, ring and replay; each
// lane draws its realisation's truth-model parameters once before the step loop (dispersion_params, tvlqr_disp_setup:
// truth inertia in TvlqrIn::I, gains of the nominal model).  Per stage the lane transforms the (uniformly loaded) field
// row of its record and scales the torque (tvlqr_disp_field, simulator7_rec<true>).
struct K4dArgs {
  K4eArgs e;
  double sigma[4];                   // sigma_inertia, sigma_torquer, sigma_field_scale, sigma_field_angle
  double* params;                    // n_sel x n_real x DISP_NP, nullable
};
// K4w: the weight-sweep ensemble of a kept run (ts_mc_weight_ensemble, WE1-WE7): K4d's replay (DISP = true; a null
// dispersion is four zero sigmas) with one warp per (slew, weighting, 32 realisations).  The warps of one slew are
// adjacent, its weightings in order, so they share the slew's reference rows in L2; the staging ring reads weighting w's
// gains (K4w gains layout).  CLAMP: the torquer limit u_limit (WE4).
struct K4wArgs {
  K4dArgs d;                         // d.e.n_sel slews; d.params unused
  int64_t n_sets, k_stride;
  double u_limit;
};
__global__ void __launch_bounds__(32 * K4E_WARPS) k4e_ensemble_replay_kernel(const K4eArgs a) {
  constexpr bool DISP = false, CLAMP = false;
  constexpr int64_t n_sets = 1, k_stride = 0;
  constexpr double u_limit = 0.0;
  const double* sigma = nullptr;
  double* params = nullptr;
#include "k4e_replay_body.inc"
}
__global__ void __launch_bounds__(32 * K4E_WARPS) k4d_dispersion_replay_kernel(const K4dArgs ad) {
  constexpr bool DISP = true, CLAMP = false;
  constexpr int64_t n_sets = 1, k_stride = 0;
  constexpr double u_limit = 0.0;
  const K4eArgs& a = ad.e;
  const double* sigma = ad.sigma;
  double* params = ad.params;
#include "k4e_replay_body.inc"
}
template <bool CLAMP>
__global__ void __launch_bounds__(32 * K4E_WARPS) k4w_weight_replay_kernel(const K4wArgs aw) {
  constexpr bool DISP = true;
  const int64_t n_sets = aw.n_sets, k_stride = aw.k_stride;
  const double u_limit = aw.u_limit;
  const K4eArgs& a = aw.d.e;
  const double* sigma = aw.d.sigma;
  double* params = nullptr;
#include "k4e_replay_body.inc"
}

// eigen_axis_slew + Bryson weights, one thread per trial.  t_k = t0 + k*dt, k = 0..nt-1 with
// nt = length(t0:dt:t_final).  Optional guess outputs (ragged nt x 3 / nt x 4 at goffs).
struct PrepArgs {
  int64_t n_trials;
  const double* x0;       // 8 per trial (omega, q, clock)
  const double* xf;       // 8
  const double* Jmat;     // 9
  const double* t_final;  // per trial
  double t0, dt, alpha, beta;
  int conj_fix;           // 0: the reference's literal qmult(q_f, q_0) (eigen_axis_slew.jl:16); 1: conj(q_f) (x) q_0
  double* Qd;             // 8 per trial
  double* Qfd;
  double* Rd;             // 3
  const int64_t* goffs;   // nullable
  double* w_guess;        // nullable
  double* q_guess;        // nullable
};

__global__ void __launch_bounds__(128) k_slew_prep(const PrepArgs a) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.n_trials) return;
  const double PI = 3.141592653589793;
  const double* x0 = a.x0 + t * 8;
  const double* xf = a.xf + t * 8;
  const double* J = a.Jmat + t * 9;
  const double q1[4] = {x0[3], x0[4], x0[5], x0[6]};
  // eigen_axis_slew.jl:16 passes the 7-vector [q2; -q2[2:4]] to qmult, which reads entries 1 and 2:4 only: the literal
  // error quaternion is qmult(q2, q1), NOT conj(q2) (x) q1.  Reproduced by default; conj_fix = 1 is the evident intent.
  const double sg = a.conj_fix ? -1.0 : 1.0;
  const double q2c[4] = {xf[3], sg * xf[4], sg * xf[5], sg * xf[6]};
  double qe[4];
  qmult(q2c, q1, qe);
  const double theta_f = 2 * acos(qe[0]);
  const double sh = sin(theta_f / 2);
  const double axis[3] = {-qe[1] / sh, -qe[2] / sh, -qe[3] / sh};
  const long long nt = range_len(a.t0, a.dt, a.t_final[t]);
  const double t_end = a.t0 + a.dt * (double)(nt - 1);
  const double al = PI / t_end;
  const double tstep = (a.t0 + a.dt * 1.0) - (a.t0 + a.dt * 0.0);  // t[2]-t[1]
  double w_max = 0.0, tau_max = -INFINITY;
  double th_prev = theta_f * 1 / 2 * (1.0 - cos(al * (a.t0 + a.dt * 0.0)));
  double dth_prev = 0.0, w_prev[3] = {0, 0, 0};
  double* wg = (a.w_guess && a.goffs) ? a.w_guess + a.goffs[t] * 3 : nullptr;
  double* qg = (a.q_guess && a.goffs) ? a.q_guess + a.goffs[t] * 4 : nullptr;
  for (long long i = 0; i < nt; ++i) {
    double dth;
    double th_next = 0.0;
    if (i + 1 < nt) {
      th_next = theta_f * 1 / 2 * (1.0 - cos(al * (a.t0 + a.dt * (double)(i + 1))));
      dth = (th_next - th_prev) / tstep;
    } else {
      dth = dth_prev;  // push!(d_theta, d_theta[end])
    }
    double w[3];
    for (int c = 0; c < 3; ++c) {
      w[c] = dth * axis[c];
      w_max = fmax(w_max, fabs(w[c]));
    }
    if (i > 0) {
      const double dw[3] = {w[0] - w_prev[0], w[1] - w_prev[1], w[2] - w_prev[2]};
      for (int r = 0; r < 3; ++r) {
        double s = J[r * 3 + 0] * dw[0];
        s += J[r * 3 + 1] * dw[1];
        s += J[r * 3 + 2] * dw[2];
        tau_max = fmax(tau_max, s / a.dt);
      }
    }
    if (wg)
      for (int c = 0; c < 3; ++c) wg[i * 3 + c] = w[c];
    if (qg) {
      const double hs = sin(th_prev / 2);
      const double qa[4] = {cos(th_prev / 2), axis[0] * hs, axis[1] * hs, axis[2] * hs};
      qmult(q1, qa, qg + i * 4);
    }
    for (int c = 0; c < 3; ++c) w_prev[c] = w[c];
    dth_prev = dth;
    th_prev = th_next;
  }
  const double m_max = tau_max / 1.e-5 * 1.e2;
  double* Qd = a.Qd + t * 8;
  double* Qfd = a.Qfd + t * 8;
  for (int i = 0; i < 3; ++i) {
    Qd[i] = a.alpha / (w_max * w_max);
    Qfd[i] = a.alpha / (w_max * w_max) * 10;
  }
  for (int i = 3; i < 7; ++i) {
    Qd[i] = a.alpha * a.beta;
    Qfd[i] = a.alpha * a.beta * 10;
  }
  Qd[7] = 0.0;
  Qfd[7] = 0.0;
  for (int i = 0; i < 3; ++i) a.Rd[t * 3 + i] = 1 / (m_max * m_max);
}

}  // namespace ts
