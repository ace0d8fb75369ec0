// K3 -- batched AL-iLQR, two launches.
//
// k3_alilqr_kernel: persistent warps; each warp runs FOUR trials at a time, one per 8-lane team (ilqr_solver.cuh),
// pulling groups of four trials from an atomic queue (trials pre-sorted by horizon on the host so that the four
// teams of a warp have similar trip counts, then dealt by slew angle).  Finished teams lend their lanes and
// trajectory buffers to the unfinished trials of their warp.
// k3_wide_kernel: once the queue is empty, trials that have used their allowance of knot-iterations are parked by
// the first kernel and finished here, ONE trial per warp (32-lane team), longest remaining budget first.
//
// Why 8-lane teams first and not one trial per warp throughout: an FP64 warp instruction occupies the SM
// sub-partition's 16-lane DFMA pipe for 2 issue cycles whatever the number of active lanes, and the sequential
// parts of iLQR (Riccati recursion, rollouts) expose limited parallelism per knot, so four trials per warp are the
// throughput-efficient mapping (3.9 vs 7.4 warp-ms per trial-iteration).  But a single-wave ensemble ends with a
// long tail of stragglers whose LATENCY is the makespan, and a whole warp per trial halves that latency
// (DESIGN.md, "K3"; measurements in profiles/README.md).
//
// Working set per trial (HBM/L2, streamed): 9 trajectory buffers (current + 8 line-search candidates; a wide warp
// uses the 36 buffers of its four slots) x N x 10, gains N x 24, multipliers N x 6 doubles.
// Shared memory per 8-lane team: 6912 B (knot records of the current 8-knot chunk, Riccati exchange buffers,
// staged forward-pass chunks, the trial's read-only parameters); 26 KB per wide warp.
#pragma once
#include "common.cuh"
#include "ilqr_solver.cuh"

namespace ts {

struct GpuTeam {
  static constexpr int W = TEAM;
  unsigned mask;
  int ln, shift;
  double* sm;
  __device__ __forceinline__ int lane() const { return ln; }
  __device__ __forceinline__ double* smem() const {
    double* p = sm;
    __builtin_assume(__isShared(p));  // lets ptxas emit LDS/STS instead of generic LD/ST
    return p;
  }
  __device__ __forceinline__ void sync() const { __syncwarp(mask); }
  __device__ __forceinline__ double bcast(double v, int src) const { return __shfl_sync(mask, v, src, TEAM); }
  __device__ __forceinline__ unsigned ballot(bool p) const { return (__ballot_sync(mask, p) >> shift) & 0xffu; }
  // asynchronous global->shared copies (cp.async / LDGSTS), 16 B per piece
  __device__ __forceinline__ void stage16(double* dst, const double* src, int n16) const {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
#pragma unroll
    for (int i = 0; i < n16; ++i)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d + 16u * i), "l"(src + 2 * i) : "memory");
  }
  __device__ __forceinline__ void prefetch_l2(const void* p) const { asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p)); }
  __device__ __forceinline__ void stage_commit() const { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
  __device__ __forceinline__ void stage_wait(int pending) const {
    if (pending == 0)
      asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    else
      asm volatile("cp.async.wait_group 1;\n" ::: "memory");
  }
  __device__ __forceinline__ double sum(double v) const {
    v += __shfl_xor_sync(mask, v, 4, TEAM);
    v += __shfl_xor_sync(mask, v, 2, TEAM);
    v += __shfl_xor_sync(mask, v, 1, TEAM);
    return v;
  }
  __device__ __forceinline__ double max(double v) const {
    v = fmax(v, __shfl_xor_sync(mask, v, 4, TEAM));
    v = fmax(v, __shfl_xor_sync(mask, v, 2, TEAM));
    v = fmax(v, __shfl_xor_sync(mask, v, 1, TEAM));
    return v;
  }
};

// The whole warp as ONE team of 32 lanes: used by k3_wide_kernel for the stragglers the persistent kernel parks.
// 32 knots are linearised per chunk and all 21 line-search candidates are rolled out in a single batch.
// (Round-1 measurement: switching to this team INSIDE the persistent kernel doubled its code and registers and
// slowed every other warp, 14.6 s -> 19.4 s on the 4096-trial ensemble; as a separate launch it costs nothing
// there.  The solver is width-generic and tested at W = 32 in tests/hostsim.)
struct GpuWideTeam {
  static constexpr int W = 32;
  int ln;
  double* sm;
  __device__ __forceinline__ int lane() const { return ln; }
  __device__ __forceinline__ double* smem() const {
    double* p = sm;
    __builtin_assume(__isShared(p));
    return p;
  }
  __device__ __forceinline__ void sync() const { __syncwarp(); }
  __device__ __forceinline__ double bcast(double v, int src) const { return __shfl_sync(0xffffffffu, v, src); }
  __device__ __forceinline__ unsigned ballot(bool p) const { return __ballot_sync(0xffffffffu, p); }
  __device__ __forceinline__ void stage16(double* dst, const double* src, int n16) const {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
#pragma unroll
    for (int i = 0; i < n16; ++i)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d + 16u * i), "l"(src + 2 * i) : "memory");
  }
  __device__ __forceinline__ void prefetch_l2(const void* p) const { asm volatile("prefetch.global.L2 [%0];\n" ::"l"(p)); }
  __device__ __forceinline__ void stage_commit() const { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
  __device__ __forceinline__ void stage_wait(int pending) const {
    if (pending == 0)
      asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    else
      asm volatile("cp.async.wait_group 1;\n" ::: "memory");
  }
  __device__ __forceinline__ double sum(double v) const {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  }
  __device__ __forceinline__ double max(double v) const {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
  }
};

// Solver state in and out (ts_alilqr_solve_state_batch; CS1-CS3 in DESIGN.md section 4, K3).  Kept behind one pointer
// of K3Args: the four-per-warp kernel sits at the register limit, and its allocation is sensitive to the parameter block.
struct K3StateIO {
  ts_al_state_dev* state_out;       // nullable; n_trials records
  double* lam_out;                  // with state_out; ragged N x 6 at offs*6 (last row of a trial zero)
  const ts_al_state_dev* state_in;  // continuation: n_trials records
  const double* lam_in;             // continuation: ragged like lam_out
  int64_t n_import;                 // continuation: trials park_import_kernel parks (places 0..n_import-1)
  int64_t lam_doubles;              // continuation: length of lam_in / lam_out (host side only)
};
struct K3Args {
  int64_t n_trials;
  const int64_t* order;  // trial permutation (sorted by horizon), n_trials entries
  const int64_t* N_i;
  const int64_t* offs;
  const double* x0;      // 8 per trial
  const double* xf;      // 8
  const double* Jmat;    // 9
  const double* Qd;      // 8
  const double* Qfd;     // 8
  const double* Rd;      // 3
  const double* B_eci;
  const int64_t* B_offs;
  const int64_t* B_rows;
  const double* index_scale;
  const double* clock_rate;
  double dt;
  const double* U0;      // nullable, ragged like U
  ts_ilqr_opts_dev opts;
  double* X;             // ragged N x 8
  double* U;             // ragged (N-1) x 3 at offs*3
  double* K;             // nullable, ragged (N-1) x 3 x 8 at offs*24
  ts_trial_outcome_dev* out;
  double* diag;          // nullable; 3 per trial: SM cycles in the backward pass, the forward pass, the linearisation
  // work arena of the first launch: one contiguous block per team slot [xu 9x | kd | lam | bk | clk], RAGGED by warp:
  // warp w starts with the w-th group of four of the horizon-sorted queue and only ever pulls shorter trials later,
  // so its four slots are sized for that first group (warp_cap[w] knots, even) and start at w_base + warp_off[w].
  // A single long-horizon outlier therefore costs one warp's worth of memory, not (slots x its horizon).
  double* w_base;
  const long long* warp_off;  // [warps] doubles
  const int* warp_cap;        // [warps] knots (even)
  int64_t n_warps;            // warps of the first launch (the dynamic queue starts behind their static first groups)
  int64_t Nmax;               // longest horizon of the ensemble, padded to even
  // region pool of the second launch: a wide warp takes k3_wide_doubles_per_knot() x N doubles per trial ([22 buffers
  // x 10 | kd 24 | lam 6 | bk 10 | clk 1] x N = 261 N by default), bump-allocated, and keeps its region for later trials
  // that fit
  double* pool;
  unsigned long long* pool_used;  // doubles handed out
  long long pool_cap;             // doubles
  unsigned long long* queue;
  int tail_share; // 1: finished siblings lend lanes + buffers to the line search of the group's last trial
  // straggler hand-over (k3_wide_kernel): once the queue is empty, a trial that has used its allowance of
  // knot-iterations (inner iterations x horizon: the unit of sequential work) is parked -- solver state + live
  // arrays copied out -- and finished by a whole warp in the second launch
  long long park_budget;      // knot-iterations; 0: never park
  long long park_budget_early; // a trial past this many knot-iterations is parked even while the queue still has work
  int park_cap;               // parking places
  unsigned* park_count;       // places handed out (may overshoot park_cap)
  TrialState* park_state;     // [park_cap]
  int64_t* park_trial;        // [park_cap] trial index
  long long* park_off;        // [park_cap] offset of the trial's arrays in park_data (doubles)
  double* park_data;          // bump-allocated, 27 * N(even) doubles per parked trial:
                              //   current trajectory 10N | multipliers 6N | stage fields 10N | clock N
  long long park_data_cap;    // doubles
  unsigned long long* park_used;  // doubles handed out
  unsigned long long* queue2; // work queue of the second launch
  int* park_order;            // [park_cap] parking places, longest remaining work first
  const struct K3StateIO* sio;   // nullable: solver state in and out (ts_alilqr_solve_state_batch), in device memory
};


// Fills the team's shared-memory TrialIn block for trial t (lane 0 writes, team syncs).
template <class Team>
__device__ __forceinline__ const TrialIn& k3_load_trial(const Team& tm, const K3Args& a, int64_t t) {
  TrialIn* inp = reinterpret_cast<TrialIn*>(tm.smem() + SmL<Team::W>::TRIAL);
  __builtin_assume(__isShared(inp));
  tm.sync();
  if (tm.ln == 0) {
    inp->N = (int)a.N_i[t];
    inp->dt = a.dt;
    for (int i = 0; i < 7; ++i) inp->x0[i] = a.x0[t * 8 + i];
    inp->clk0 = a.x0[t * 8 + 7];
    for (int i = 0; i < 8; ++i) {
      inp->xf[i] = a.xf[t * 8 + i];
      inp->Qd[i] = a.Qd[t * 8 + i];
      inp->Qfd[i] = a.Qfd[t * 8 + i];
    }
    for (int i = 0; i < 3; ++i) inp->Rd[i] = a.Rd[t * 3 + i];
    double Jm[9], Ji[9];
    for (int i = 0; i < 9; ++i) Jm[i] = a.Jmat[t * 9 + i];
    inv3_gj(Jm, Ji);
    for (int i = 0; i < 9; ++i) {
      inp->I.J[i] = Jm[i];
      inp->I.Jinv[i] = Ji[i];
    }
    inp->Bt = a.B_eci + a.B_offs[t] * 3;
    inp->B_rows = a.B_rows[t];
    inp->index_scale = a.index_scale[t];
    inp->clock_rate = a.clock_rate[t];
    inp->U0 = a.U0 ? a.U0 + a.offs[t] * 3 : nullptr;
  }
  tm.sync();
  return *inp;
}

// The four-per-warp kernels that export the solver state are instantiations of their own (Team::EXPORT): that kernel sits
// at the register limit, and the export code changes its allocation in the per-knot loops, so the solves that export
// nothing run kernels without it.  The general-inertia exporting instantiation also declares NO_LEND: without tail
// sharing (which does not change results, tests/test_gpu_ilqr.py) its per-knot loops stay free of local memory; with it,
// one reload landed in the rollout loop.
template <class Team, class = void>
struct team_export {
  static constexpr bool value = false;
};
template <class Team>
struct team_export<Team, decltype((void)Team::EXPORT)> {
  static constexpr bool value = Team::EXPORT;
};
template <class Team, class = void>
struct team_no_lend {
  static constexpr bool value = false;
};
template <class Team>
struct team_no_lend<Team, decltype((void)Team::NO_LEND)> {
  static constexpr bool value = Team::NO_LEND;
};

// Writes a finished trial's results in the reference's shapes: X (N x 8 incl. clock), U, K (3 x 8 per knot).
template <class Team>
__device__ __forceinline__ void k3_store_results(const Team& tm, const K3Args& a, int64_t t, const TrialWork& w, int N, int cur,
                                                 const ts_trial_outcome_dev& oc, const TrialState& st) {
  if (tm.ln == 0 && a.diag) solve_diag(st, a.diag + t * 3);
  if ((Team::W == 32 || team_export<Team>::value) && a.sio) {   // CS1 export
    if (tm.ln == 0) solve_export(st, a.sio->state_out[t]);
    double* Lo = a.sio->lam_out + a.offs[t] * 6;
    for (int k = tm.ln; k < N; k += Team::W)
      for (int i = 0; i < 6; ++i) Lo[(int64_t)k * 6 + i] = (k < N - 1) ? w.lam[(int64_t)k * 6 + i] : 0.0;
  }
  const double* xu = xu_buf<Team::W>(w, cur);
  double* Xo = a.X + a.offs[t] * 8;
  double* Uo = a.U + a.offs[t] * 3;
  for (int k = tm.ln; k < N; k += Team::W) {
    for (int i = 0; i < 7; ++i) Xo[(int64_t)k * 8 + i] = xu[(int64_t)k * 10 + i];
    Xo[(int64_t)k * 8 + 7] = w.clk[k];
    if (k < N - 1) {
      for (int i = 0; i < 3; ++i) Uo[(int64_t)k * 3 + i] = xu[(int64_t)k * 10 + 7 + i];
      if (a.K) {
        double* Ko = a.K + (a.offs[t] + k) * 24;
        const double* kd = w.kd + (int64_t)k * 24;
        for (int i = 0; i < 3; ++i) {
          for (int j = 0; j < 7; ++j) Ko[i * 8 + j] = kd[j * 3 + i];
          Ko[i * 8 + 7] = 0.0;
        }
      }
    } else {  // the ragged layout keeps N rows per trial: the unused last row of U and K is defined (zero)
      for (int i = 0; i < 3; ++i) Uo[(int64_t)k * 3 + i] = 0.0;
      if (a.K)
        for (int i = 0; i < 24; ++i) a.K[(a.offs[t] + k) * 24 + i] = 0.0;
    }
  }
  if (tm.ln == 0) a.out[t] = oc;
}

constexpr int K3_WARPS_PER_BLOCK = 1;
constexpr int K3_SLOT_DOUBLES_PER_KNOT = 90 + 24 + 6 + 10 + 1;      // narrow team slot: 9 buffers x 10 | kd | lam | bk | clk
// wide team: current trajectory + one buffer per line-search candidate of a batch (max_linesearch + 1 = 21 by default,
// at most 32 per batch), then kd | lam | bk | clk
__host__ __device__ inline int k3_wide_buffers(int max_linesearch) { return (max_linesearch + 1 < 32 ? max_linesearch + 1 : 32) + 1; }
__host__ __device__ inline int k3_wide_doubles_per_knot(int max_linesearch) { return k3_wide_buffers(max_linesearch) * 10 + 24 + 6 + 10 + 1; }
constexpr int K3_SMEM_BYTES = K3_WARPS_PER_BLOCK * 4 * TEAM_SMEM_DOUBLES * 8;

// index of the n-th set bit (n = 0, 1, ...) of a 4-bit mask
__device__ __forceinline__ int k3_nth_bit(unsigned m, int n) {
  int idx = 0;
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    if (m & (1u << b)) {
      if (n == 0) idx = b;
      --n;
    }
  }
  return idx;
}
__device__ __forceinline__ double k3_shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
__device__ __forceinline__ int k3_shfl_i(int v, int src) { return __shfl_sync(0xffffffffu, v, src); }
__device__ __forceinline__ long long k3_shfl_ll(long long v, int src) { return __shfl_sync(0xffffffffu, v, src); }

struct GpuTeamQuat : GpuTeam {   // the quaternion-aware variant (ts_ilqr_opts.quat_error; team_quat in ilqr_solver.cuh)
  static constexpr bool QUAT = true;
};
struct GpuTeamDiag : GpuTeam {   // every trial's inertia matrix is diagonal (team_diagj in ilqr_solver.cuh)
  static constexpr bool DIAGJ = true;
};
#define K3_BODY_TEAM GpuTeam
__global__ void __launch_bounds__(K3_WARPS_PER_BLOCK * 32, 1) k3_alilqr_kernel(const K3Args a) {
#include "k3_alilqr_body.inc"
}
#undef K3_BODY_TEAM
#define K3_BODY_TEAM GpuTeamDiag
__global__ void __launch_bounds__(K3_WARPS_PER_BLOCK * 32, 1) k3_alilqr_diag_kernel(const K3Args a) {
#include "k3_alilqr_body.inc"
}
#undef K3_BODY_TEAM
#define K3_BODY_TEAM GpuTeamQuat
__global__ void __launch_bounds__(K3_WARPS_PER_BLOCK * 32, 1) k3_alilqr_quat_kernel(const K3Args a) {
#include "k3_alilqr_body.inc"
}
#undef K3_BODY_TEAM
struct GpuTeamQuatDiag : GpuTeamQuat {
  static constexpr bool DIAGJ = true;
};
#define K3_BODY_TEAM GpuTeamQuatDiag
__global__ void __launch_bounds__(K3_WARPS_PER_BLOCK * 32, 1) k3_alilqr_quat_diag_kernel(const K3Args a) {
#include "k3_alilqr_body.inc"
}
#undef K3_BODY_TEAM
// the instantiations that export the solver state (K3StateIO)
struct GpuTeamX : GpuTeam {
  static constexpr bool EXPORT = true;
  static constexpr bool NO_LEND = true;
};
#define K3_BODY_TEAM GpuTeamX
__global__ void __launch_bounds__(K3_WARPS_PER_BLOCK * 32, 1) k3_alilqr_export_kernel(const K3Args a) {
#include "k3_alilqr_body.inc"
}
#undef K3_BODY_TEAM
struct GpuTeamDiagX : GpuTeamDiag {
  static constexpr bool EXPORT = true;
};
struct GpuTeamQuatX : GpuTeamQuat {
  static constexpr bool EXPORT = true;
};
struct GpuTeamQuatDiagX : GpuTeamQuatDiag {
  static constexpr bool EXPORT = true;
};
#define K3_BODY_TEAM GpuTeamDiagX
__global__ void __launch_bounds__(K3_WARPS_PER_BLOCK * 32, 1) k3_alilqr_diag_export_kernel(const K3Args a) {
#include "k3_alilqr_body.inc"
}
#undef K3_BODY_TEAM
#define K3_BODY_TEAM GpuTeamQuatX
__global__ void __launch_bounds__(K3_WARPS_PER_BLOCK * 32, 1) k3_alilqr_quat_export_kernel(const K3Args a) {
#include "k3_alilqr_body.inc"
}
#undef K3_BODY_TEAM
#define K3_BODY_TEAM GpuTeamQuatDiagX
__global__ void __launch_bounds__(K3_WARPS_PER_BLOCK * 32, 1) k3_alilqr_quat_diag_export_kernel(const K3Args a) {
#include "k3_alilqr_body.inc"
}
#undef K3_BODY_TEAM
// ---------------------------------------------------------------------------------------------
// Second launch: every parked straggler is finished by ONE WHOLE WARP (32-lane team): 32 knots linearised per
// chunk, all 21 line-search candidates in one batch, one warp per SM sub-partition when few trials are left.
// The makespan of a single-wave ensemble is the latency of its slowest trial (the ~7% of slews that use all
// max_outer x max_inner iterations), and a lone 8-lane team leaves 3/4 of its warp's issue slots empty.
// The per-trial arithmetic is that of the width-generic solver: outcomes do not depend on where a trial ran
// (tests/test_hostsim_*.py run the same source at W = 8 and W = 32).
// Between the two launches: order the parked trials by their remaining BUDGET of knot-iterations (remaining
// inner iterations x horizon), largest first (counting sort, one block).  The trials that will use every remaining iteration (the non-converging ones sit at a low
// outer count) then start in the first wave, and the short ones fill the warps that free up: longest-
// processing-time-first on the only estimate available.
__global__ void __launch_bounds__(1024, 1) k3_park_order_kernel(const K3Args a) {
  __shared__ int hist[1024];
  __shared__ int start[1024];
  unsigned n = *a.park_count;
  if (n > (unsigned)a.park_cap) n = (unsigned)a.park_cap;
  const int tid = threadIdx.x;
  hist[tid] = 0;
  __syncthreads();
  const double full = (double)a.opts.max_outer * a.opts.max_inner * (double)a.Nmax;
  auto bin_of = [&](unsigned i) {
    const TrialState& st = a.park_state[i];
    long long rem = (long long)(a.opts.max_outer - st.outer) * a.opts.max_inner + (a.opts.max_inner - st.it);
    if (rem < 0) rem = 0;
    double f = (double)rem * (double)a.N_i[a.park_trial[i]] / (full > 0.0 ? full : 1.0);   // remaining knot-iterations, relative
    if (f > 1.0) f = 1.0;
    return 1023 - (int)(f * 1023.0);   // bin 0 = most remaining work
  };
  for (unsigned i = tid; i < n; i += 1024) atomicAdd(&hist[bin_of(i)], 1);
  __syncthreads();
  if (tid == 0) {
    int acc = 0;
    for (int b = 0; b < 1024; ++b) {
      start[b] = acc;
      acc += hist[b];
    }
  }
  __syncthreads();
  for (unsigned i = tid; i < n; i += 1024) a.park_order[atomicAdd(&start[bin_of(i)], 1)] = (int)i;
}

// ---------------------------------------------------------------------------------------------
// Continuation (ts_alilqr_solve_state_batch with a state): one 8-lane team per continuing trial builds that trial's
// parked form -- TrialState + the 27 N-double record k3_wide_kernel / k3_pair_kernel resume from -- in the park
// buffers: the trial's tables (as solve_init builds them), the imported trajectory and multipliers, and the start of
// its next outer iteration (CS3, solve_import).  Place i holds trial park_trial[i] at park_off[i] (set by the host).
// Continuing trials are stragglers by construction: they go straight to the one-warp-per-trial launch.
__global__ void __launch_bounds__(32, 1) park_import_kernel(const K3Args a) {
  extern __shared__ __align__(16) double k3_smem[];
  const int lane32 = threadIdx.x & 31;
  const int team = lane32 >> 3;
  const int64_t i = (int64_t)blockIdx.x * 4 + team;
  if (i >= a.sio->n_import) return;   // team-uniform: the teams of a warp never synchronise with each other here
  GpuTeam tm;
  tm.ln = lane32 & 7;
  tm.shift = team * 8;
  tm.mask = 0xffu << tm.shift;
  tm.sm = k3_smem + team * TEAM_SMEM_DOUBLES;
  const int64_t t = a.park_trial[i];
  const TrialIn& in = k3_load_trial(tm, a, t);
  const int N = in.N;
  const long long Ne = N + (N & 1);
  double* pd = a.park_data + a.park_off[i];
  TrialWork w;
  w.Nmax = Ne;
  w.xu = w.xu_warp = pd;
  w.slot_stride = 0;
  w.kd = nullptr;
  w.lam = pd + 10 * Ne;
  w.bk = pd + 16 * Ne;
  w.clk = pd + 26 * Ne;
  const double* X = a.X + a.offs[t] * 8;
  const double* U = a.U + a.offs[t] * 3;
  const double* L = a.sio->lam_in + a.offs[t] * 6;
  for (int k = tm.ln; k < N; k += TEAM) {
    const bool stage = k < N - 1;
    for (int j = 0; j < 7; ++j) pd[(long long)k * 10 + j] = X[(long long)k * 8 + j];
    for (int j = 0; j < 3; ++j) pd[(long long)k * 10 + 7 + j] = stage ? U[(long long)k * 3 + j] : 0.0;
    for (int j = 0; j < 6; ++j) w.lam[(long long)k * 6 + j] = stage ? L[(long long)k * 6 + j] : 0.0;
  }
  TrialState st;
  solve_import(tm, in, a.opts, w, a.sio->state_in[t], st);
  if (tm.ln == 0) a.park_state[i] = st;
}

struct GpuWideQuatTeam : GpuWideTeam {
  static constexpr bool QUAT = true;
};
struct GpuWideDiagTeam : GpuWideTeam {
  static constexpr bool DIAGJ = true;
};
#define K3_BODY_TEAM GpuWideTeam
__global__ void __launch_bounds__(32, 1) k3_wide_kernel(const K3Args a) {
#include "k3_wide_body.inc"
}
#undef K3_BODY_TEAM
#define K3_BODY_TEAM GpuWideDiagTeam
__global__ void __launch_bounds__(32, 1) k3_wide_diag_kernel(const K3Args a) {
#include "k3_wide_body.inc"
}
#undef K3_BODY_TEAM
#define K3_BODY_TEAM GpuWideQuatTeam
__global__ void __launch_bounds__(32, 1) k3_wide_quat_kernel(const K3Args a) {
#include "k3_wide_body.inc"
}
#undef K3_BODY_TEAM
struct GpuWideQuatDiagTeam : GpuWideQuatTeam {
  static constexpr bool DIAGJ = true;
};
#define K3_BODY_TEAM GpuWideQuatDiagTeam
__global__ void __launch_bounds__(32, 1) k3_wide_quat_diag_kernel(const K3Args a) {
#include "k3_wide_body.inc"
}
#undef K3_BODY_TEAM
constexpr int K3_WIDE_SMEM_BYTES = SmL<32>::TOTAL * 8;

// ---------------------------------------------------------------------------------------------
// k3_pair_kernel: the one-warp-per-trial solver with a PRODUCER warp.  A straggler's latency is what ends the run, and
// of the ~4.4 k cycles a whole warp spends per knot-iteration ~0.6 k is the linearisation of the next 32-knot chunk --
// pure throughput work (one knot per lane, no dependence on the Riccati recursion) that sits on the critical path only
// because the same warp does it.  Here a second warp computes the Jacobian records [A|B] of chunk c-1 into the other
// half of a double buffer while the solver warp runs the 32 sequential Riccati steps of chunk c: the solver warp issues
// one instruction every ~3 cycles (dependent FP64 chains), so the producer's instructions fill issue slots and FP64 pipe
// cycles that would otherwise idle.
// Geometry: ONE block of 8 warps per SM (192 KB of shared memory, 255 registers): warps 0..3 are solver warps, warp 4+i
// is the producer of solver i; with the hardware's round-robin warp placement each SM sub-partition hosts exactly one
// solver and one producer -- a solver never shares its sub-partition with another solver (at 8 solver warps per SM a
// trial-iteration costs 7.7 ms, alone 4.6 ms).
// Hand-over through named barriers, 4 per pair (bar.arrive / bar.sync on 64 threads):
//   EMPTY_b  solver arrives when buffer b may be (re)filled: at the start of a sweep for both buffers, afterwards when
//            it has consumed the chunk in it; producer syncs before producing
//   FULL_b   producer arrives when buffer b holds a chunk, solver syncs before reading it
// A regularisation restart (Quu not positive definite) at sweep position j drains position j+1 (always produced) and
// tells the producer to stop before position j+2 (abort_pos; a position tag, not a flag, so that the producer's decision
// does not depend on when it happens to look).  Same solver source, same arithmetic as k3_wide_kernel.
struct K3PairCmd {
  const double* xu;    // trajectory to linearise
  const double* bk;    // stage field vectors
  int N;
  int type;            // 1 = sweep, 0 = exit
  volatile int abort_pos;  // -1, or the first sweep position the producer must NOT produce any more
  int pad_;
};
__device__ __forceinline__ void k3p_bar_sync(int id) { asm volatile("barrier.sync %0, 64;\n" ::"r"(id) : "memory"); }
__device__ __forceinline__ void k3p_bar_arrive(int id) { asm volatile("barrier.arrive %0, 64;\n" ::"r"(id) : "memory"); }

struct GpuPairTeam : GpuWideTeam {
  static constexpr bool EXT_LIN = true;
  double* rec1;        // second record buffer (the first is SmL<32>::REC0 of the pair's region)
  K3PairCmd* cmd;
  int bar0;            // first of the pair's four barrier ids: FULL_0, FULL_1, EMPTY_0, EMPTY_1
  __device__ __forceinline__ void lin_begin(const double* xu, const double* bk, int N) const {
    if (ln == 0) {
      cmd->xu = xu;
      cmd->bk = bk;
      cmd->N = N;
      cmd->type = 1;
      cmd->abort_pos = -1;
    }
    __syncwarp();
    __threadfence_block();
    k3p_bar_arrive(bar0 + 2);                       // both buffers are free: the producer starts on positions 0 and 1
    if (N - 1 > 32) k3p_bar_arrive(bar0 + 3);
  }
  __device__ __forceinline__ double* rec_wait(int pos) const {
    k3p_bar_sync(bar0 + (pos & 1));
    double* p = (pos & 1) ? rec1 : sm + SmL<32>::REC0;
    __builtin_assume(__isShared(p));
    return p;
  }
  __device__ __forceinline__ void rec_release(int pos, bool more) const {
    if (more) {
      __threadfence_block();
      k3p_bar_arrive(bar0 + 2 + (pos & 1));
    }
  }
  // abort at sweep position pos (whose FULL barrier has been passed): the producer produces position pos+1 in any case
  __device__ __forceinline__ void lin_abort(int pos, int n_pos) const {
    if (ln == 0) cmd->abort_pos = pos + 2;
    __syncwarp();
    __threadfence_block();
    if (pos + 1 < n_pos) k3p_bar_sync(bar0 + ((pos + 1) & 1));     // drain position pos+1
    if (pos + 2 < n_pos) k3p_bar_arrive(bar0 + 2 + (pos & 1));     // wake the producer at pos+2: it sees abort_pos and stops
  }
};
constexpr int K3_PAIRS_PER_BLOCK = 4;
constexpr int K3_PAIR_REGION_DOUBLES = SmL<32>::TOTAL + 32 * REC + 8 + 8;   // solver layout | second record buffer | cmd | TrialWork
static_assert(sizeof(K3PairCmd) <= 64 && sizeof(TrialWork) <= 64, "pair control blocks");
constexpr int K3_PAIR_SMEM_BYTES = K3_PAIRS_PER_BLOCK * K3_PAIR_REGION_DOUBLES * 8;

template <class PairTeam>
__device__ __forceinline__ void k3_pair_body(const K3Args& a) {
  extern __shared__ __align__(16) double k3_smem[];
  const int lane32 = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int pair = warp & (K3_PAIRS_PER_BLOCK - 1);
  const bool is_producer = warp >= K3_PAIRS_PER_BLOCK;
  double* region = k3_smem + pair * K3_PAIR_REGION_DOUBLES;
  double* rec1 = region + SmL<32>::TOTAL;
  K3PairCmd* cmd = reinterpret_cast<K3PairCmd*>(region + SmL<32>::TOTAL + 32 * REC);
  TrialWork& w = *reinterpret_cast<TrialWork*>(region + SmL<32>::TOTAL + 32 * REC + 8);
  const int bar0 = pair * 4;
  if (is_producer) {
    // ------------------------------------------------------------------ producer warp
    const TrialIn* inp = reinterpret_cast<const TrialIn*>(region + SmL<32>::TRIAL);
    __builtin_assume(__isShared(inp));
    for (;;) {
      // a sweep starts when the solver frees buffer 0 (lin_begin); the command block is valid from then on
      int pos = 0, n_pos = 1;
      bool done = false;
#pragma unroll 1
      for (; pos < n_pos; ++pos) {
        const int b = pos & 1;
        k3p_bar_sync(bar0 + 2 + b);
        if (pos == 0) {
          if (cmd->type == 0) {
            done = true;
            break;
          }
          n_pos = (cmd->N - 1 + 31) / 32;
        }
        const int ap = cmd->abort_pos;
        if (ap >= 0 && pos >= ap) break;
        const int N = cmd->N;
        const int k = (n_pos - 1 - pos) * 32 + lane32;
        if (k < N - 1) {
          double* rec = (b ? rec1 : region + SmL<32>::REC0) + lane32 * REC;
          __builtin_assume(__isShared(rec));
          const double* p = gptr(cmd->xu) + (long long)k * 10;
          const double* bp = gptr(cmd->bk) + (long long)k * 10;
          double x[7], u[3], bb[9];
          // (L2 loads: the solver warp wrote this trajectory with plain stores a moment ago)
          for (int i = 0; i < 7; ++i) x[i] = __ldcg(p + i);
          for (int i = 0; i < 3; ++i) u[i] = __ldcg(p + 7 + i);
          for (int i = 0; i < 9; ++i) bb[i] = __ldcg(bp + i);
          rk3_jac7_jvp<team_diagj<PairTeam>::value>(inp->I, x, u, bb, bb + 3, bb + 6, inp->dt, rec);
        }
        __syncwarp();
        __threadfence_block();
        k3p_bar_arrive(bar0 + b);
      }
      if (done) break;
    }
    return;
  }
  // -------------------------------------------------------------------- solver warp (as k3_wide_kernel)
  PairTeam tm;
  tm.ln = lane32;
  tm.sm = region;
  tm.rec1 = rec1;
  tm.cmd = cmd;
  tm.bar0 = bar0;
  if (lane32 == 0) {
    w.Nmax = 0;
    w.xu = w.xu_warp = w.kd = w.lam = w.bk = w.clk = nullptr;
    w.slot_stride = 0;
  }
  __syncwarp();
  long long region_cap = 0;
  const int nbuf = k3_wide_buffers(a.opts.max_linesearch);
  const long long dpk = k3_wide_doubles_per_knot(a.opts.max_linesearch);
  unsigned n_parked = *a.park_count;
  if (n_parked > (unsigned)a.park_cap) n_parked = (unsigned)a.park_cap;
  for (;;) {
    unsigned long long qpos = 0;
    if (lane32 == 0) qpos = atomicAdd(a.queue2, 1ull);
    qpos = __shfl_sync(0xffffffffu, qpos, 0);
    if (qpos >= n_parked) break;
    const int64_t idx = a.park_order[qpos];
    const int64_t t = a.park_trial[idx];
    const TrialIn& in = k3_load_trial(tm, a, t);
    const int N = in.N;
    const long long Ne = N + (N & 1);
    if (Ne > region_cap) {
      unsigned long long off = 0;
      if (lane32 == 0) off = atomicAdd(a.pool_used, (unsigned long long)(Ne * dpk));
      off = __shfl_sync(0xffffffffu, off, 0);
      if ((long long)(off + Ne * dpk) > a.pool_cap) {
        if (lane32 == 0) {
          ts_trial_outcome_dev oc = {};
          oc.status = ST_NAN;
          oc.N = N;
          a.out[t] = oc;
        }
        continue;
      }
      region_cap = Ne;
      __syncwarp();
      if (lane32 == 0) {
        w.Nmax = Ne;
        w.slot_stride = 9 * Ne * 10;
        w.xu = w.xu_warp = a.pool + off;
        w.kd = w.xu + (long long)nbuf * 10 * Ne;
        w.lam = w.kd + 24 * Ne;
        w.bk = w.lam + 6 * Ne;
        w.clk = w.bk + 10 * Ne;
      }
      __syncwarp();
    }
    const double* pd = a.park_data + a.park_off[idx];
    for (int i = lane32; i < N * 10; i += 32) w.xu[i] = pd[i];
    for (int i = lane32; i < N * 6; i += 32) w.lam[i] = pd[10 * Ne + i];
    for (int i = lane32; i < N * 10; i += 32) w.bk[i] = pd[16 * Ne + i];
    for (int i = lane32; i < N; i += 32) w.clk[i] = pd[26 * Ne + i];
    TrialState st = a.park_state[idx];
    st.cur = 0;
    __syncwarp();
    __threadfence_block();   // the producer reads the trajectory and field vectors this warp just wrote
    while (st.phase != PH_DONE) {
      if (st.phase == PH_BACKWARD) solve_backward(tm, in, a.opts, w, st);
      while (st.phase == PH_FORWARD) solve_forward(tm, in, a.opts, w, st);
    }
    ts_trial_outcome_dev oc;
    solve_finish(in, st, oc);
    k3_store_results(tm, a, t, w, N, st.cur, oc, st);
    __syncwarp();
  }
  if (lane32 == 0) cmd->type = 0;
  __syncwarp();
  __threadfence_block();
  k3p_bar_arrive(bar0 + 2);   // wakes the producer at the start of a sweep: it sees type == 0 and exits
}
struct GpuPairDiagTeam : GpuPairTeam {
  static constexpr bool DIAGJ = true;
};
__global__ void __launch_bounds__(64 * K3_PAIRS_PER_BLOCK, 1) k3_pair_kernel(const K3Args a) { k3_pair_body<GpuPairTeam>(a); }
__global__ void __launch_bounds__(64 * K3_PAIRS_PER_BLOCK, 1) k3_pair_diag_kernel(const K3Args a) { k3_pair_body<GpuPairDiagTeam>(a); }

}  // namespace ts
