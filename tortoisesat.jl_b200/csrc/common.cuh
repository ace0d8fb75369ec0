// Context, error plumbing and small helpers shared by every kernel file.
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/tortoise_b200.h"

namespace ts {
// Grow-only device scratch slots of a context.  Most slots hold one call's working storage and are shared between
// entries: whatever a call leaves in them is dead once it returns.  Storage that a later call reads (the readers are
// ts_k3_last_*, ts_mc_fetch_trajectories, ts_mc_fetch_state and ts_mc_continue) lives in a slot that no other entry
// writes.
enum Slot : int {
  SLOT_POSITIONS,                          // K2 orbit positions (ts_magnetic_simulation_batch without `pos`, Monte-Carlo)
  SLOT_ARGS_A, SLOT_ARGS_B, SLOT_ARGS_C,   // a call's small per-trial inputs; C also K3 outcomes and slew-prep outputs
  SLOT_CUTOFF,                             // gramian / condition-time cutoffs
  SLOT_PER_TRIAL,                          // tf_index, the K3 queue order, K4 N_sim + slew_time
  SLOT_K3_ARENA, SLOT_ROWS_A, SLOT_ROWS_B, // K3 trajectory arena; per-row outputs (slew-prep guesses, Monte-Carlo scoping field)
  SLOT_K4_GAINS,                           // K4 gains when the caller passes none
  SLOT_ORBIT_BLOCK, SLOT_ROW_LIMITS,       // Monte-Carlo per-orbit block and table row limits
  SLOT_PACKED_I64, SLOT_PACKED_F64,        // Monte-Carlo packed per-trial arrays (read by ts_mc_continue)
  SLOT_STREAM_IDS,                         // Monte-Carlo Philox stream ids (the run's own replay)
  SLOT_PARK_STATE, SLOT_PARK_DATA,         // K3 parking places (read by ts_k3_last_parked) and parked trajectories
  SLOT_PIPE_A, SLOT_PIPE_B,                // K1 host-pointer pipeline stages
  SLOT_K3_CYCLES,                          // K3 cycle counters (read by ts_k3_last_cycles)
  SLOT_KEPT_XSIM, SLOT_KEPT_USIM, SLOT_KEPT_BLOCK,   // Monte-Carlo kept trajectories, field tables, weights and outcomes
                                                     // (read by ts_mc_fetch_trajectories and ts_mc_continue)
  SLOT_K3_WARP_OFFS, SLOT_K3_WARP_CAPS, SLOT_K3_POOL, // K3 per-warp arena offsets and capacities, straggler pool
  SLOT_LIN_RECORDS,                        // K4 linearisation records
  SLOT_TABLE,                              // a call's lookup table: K4 linearisation offsets, K8 padded coefficients
  SLOT_K3_COUNTERS,                        // K3 queue and park counters (read by ts_k3_last_split / ts_k3_last_parked)
  SLOT_AL_STATES,                          // K3 continuation: a call's imported and exported solver states
  SLOT_KEPT_STATE,                         // Monte-Carlo kept solver states + multipliers (ts_mc_fetch_state, ts_mc_continue)
  SLOT_ENSEMBLE_OUT,                       // an ensemble's slew times, final states and parameters (ts_mc_replay_ensemble, ts_mc_dispersion_ensemble)
  SLOT_WEIGHT_SETS,                        // a weight-sweep ensemble's weightings (ts_mc_weight_ensemble)
  SLOT_COUNT
};

// The per-trial inputs of a fused Monte-Carlo run's n active trials, packed column by column: hi holds the int64 columns
// and then the run's total knot count, hf the double columns, column k at [F_COL[k] * n, F_COL[k + 1] * n) (trial a's
// entries at F_COL[k] * n + width(k) * a).  ts_monte_carlo_run fills and uploads it, and ts_mc_continue and
// ts_mc_replay_ensemble compact the kept copy to the trials they replay.
enum McColI : int { I_N, I_OFFS, I_B_OFFS, I_B_ROWS, I_COLS };
enum McColF : int { F_X0, F_XF, F_JMAT, F_T_FINAL, F_INDEX_SCALE, F_CLOCK_RATE, F_X0LQR, F_Q_FINAL, F_COLS };
constexpr size_t F_COL[F_COLS + 1] = {0, 8, 16, 25, 26, 27, 28, 36, 40};

struct McPacked {
  size_t n;
  std::vector<int64_t> hi;
  std::vector<double> hf;
  std::vector<uint32_t> sid;   // Philox stream ids
  McPacked(size_t n = 0) : n(n), hi(I_COLS * n + 1), hf(F_COL[F_COLS] * n), sid(n) {}
  static size_t width(McColF k) { return F_COL[k + 1] - F_COL[k]; }
  int64_t* col(McColI k) { return hi.data() + k * n; }
  const int64_t* col(McColI k) const { return hi.data() + k * n; }
  double* at(McColF k, size_t a) { return hf.data() + F_COL[k] * n + width(k) * a; }
  const double* at(McColF k, size_t a) const { return hf.data() + F_COL[k] * n + width(k) * a; }
  // the trials sel (indices, repeats allowed) alone; their knot and row offsets keep pointing into the full arrays
  McPacked compact(const std::vector<int64_t>& sel) const {
    McPacked p(sel.size());
    for (size_t k = 0; k < p.n; ++k) {
      const size_t a = (size_t)sel[k];
      for (int j = 0; j < I_COLS; ++j) p.col((McColI)j)[k] = col((McColI)j)[a];
      for (int j = 0; j < F_COLS; ++j) memcpy(p.at((McColF)j, k), at((McColF)j, a), width((McColF)j) * sizeof(double));
      p.sid[k] = sid[a];
    }
    p.hi.back() = hi.back();
    return p;
  }
};

// an uploaded McPacked: the columns as device pointers
struct McPackedView {
  const int64_t* i = nullptr;
  const double* f = nullptr;
  size_t n = 0;
  const int64_t* col(McColI k) const { return i + k * n; }
  const double* col(McColF k) const { return f + F_COL[k] * n; }
};
}  // namespace ts

struct ts_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev_k3[3] = {nullptr, nullptr, nullptr};  // K3: start | persistent kernel done | straggler kernel done
  unsigned* d_k3_parked = nullptr;                     // device word holding the number of parked trials of the last K3 run
  bool k3_timed = false;
  int k3_park_cap = 0;                                 // parking places of the last K3 run
  int64_t k3_diag_n = 0;                               // trials covered by the K3 cycle diagnostics (SLOT_K3_CYCLES)
  cudaStream_t pipe[2] = {nullptr, nullptr};           // K1 host-pointer path: double-buffered copy/compute pipeline
  cudaEvent_t pipe_ev = nullptr;
  char err[512] = {0};
  char name[128] = {0};
  int64_t launches = 0;
  double last_kernel_ms = 0.0;
  double ens_ms[2] = {0.0, 0.0};  // the last replay / dispersion / weight ensemble: gains (K4a + K4b / K4w) | replay (K4e / K4d / K4w)
  double* d_tabG = nullptr;  // 104 x 25
  double* d_tabH = nullptr;  // 91 x 25
  double* d_tabGH = nullptr; // 3450 (igrf12syn)
  int* d_flag = nullptr;     // generic device error/flag word
  void* d_gh_stage = nullptr; // K1: the call's interpolated coefficient table (2 x 104 double2)
  // the last ts_monte_carlo_run with keep_trajectories, cleared when a run starts (device pointers into the kept slots).
  // The kept level cfg.keep_trajectories: 1 the trajectories and what ts_mc_replay_ensemble needs, 2 also ts_mc_continue's.
  struct McLast {
    ts_mc_config cfg = {};
    int64_t n = 0, knots = 0, rows = 0;
    std::vector<int64_t> knot_offs, row_offs;
    double *d_X = nullptr, *d_U = nullptr, *d_Xs = nullptr, *d_Us = nullptr, *d_B = nullptr;
    bool diag_inertia = false;
    std::vector<int64_t> act;       // active trials (caller indices); none reached the solver: no trajectories kept
    ts::McPacked in;                // their packed inputs and stream ids
    std::vector<ts_trial_outcome> out;
    // keep_trajectories = 2
    ts::McPackedView d_in;
    double *d_w = nullptr, *d_lam = nullptr;
    ts_trial_outcome* d_out = nullptr;
    ts_al_state* d_state = nullptr;
    void* d_sio = nullptr;          // the K3StateIO block of the kept states
  } mc_last;
  // grow-only scratch arenas
  void* scratch[ts::SLOT_COUNT] = {};
  size_t scratch_bytes[ts::SLOT_COUNT] = {};
};

namespace ts {

inline int fail(ts_ctx* ctx, int code, const char* fmt, ...) {
  if (ctx) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(ctx->err, sizeof(ctx->err), fmt, ap);
    va_end(ap);
  }
  return code;
}

// The sigmas a dispersion ensemble accepts (ts_mc_dispersion_ensemble): finite and >= 0, the three log-standard
// deviations <= 1 and the field angle <= pi.
inline bool dispersion_opts_ok(const ts_dispersion_opts* d) {
  const double s[4] = {d->sigma_inertia, d->sigma_torquer, d->sigma_field_scale, d->sigma_field_angle};
  for (int i = 0; i < 4; ++i)
    if (!std::isfinite(s[i]) || s[i] < 0.0 || s[i] > (i < 3 ? 1.0 : 3.14159265358979323846)) return false;
  return true;
}

// The weightings and torquer limit a weight-sweep ensemble accepts (ts_mc_weight_ensemble, WE7): n_sets >= 1, every Qd
// and Qfd entry finite and >= 0, every Rd entry finite and > 0 (B'SB + R stays invertible), u_limit finite and >= 0.
inline bool weight_sets_ok(int64_t n_sets, const ts_tvlqr_weights* sets, double u_limit) {
  if (n_sets < 1 || !sets || !std::isfinite(u_limit) || u_limit < 0.0) return false;
  for (int64_t w = 0; w < n_sets; ++w) {
    for (int i = 0; i < 6; ++i)
      if (!std::isfinite(sets[w].Qd[i]) || sets[w].Qd[i] < 0.0 || !std::isfinite(sets[w].Qfd[i]) || sets[w].Qfd[i] < 0.0) return false;
    for (int i = 0; i < 3; ++i)
      if (!std::isfinite(sets[w].Rd[i]) || !(sets[w].Rd[i] > 0.0)) return false;
  }
  return true;
}

#define TS_CUDA(ctx, call)                                                                              \
  do {                                                                                                  \
    cudaError_t e__ = (call);                                                                           \
    if (e__ != cudaSuccess)                                                                             \
      return ts::fail((ctx), TS_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

// grow-only device scratch slot
inline int scratch_reserve(ts_ctx* ctx, Slot slot, size_t bytes, void** out) {
  if (ctx->scratch_bytes[slot] < bytes) {
    if (ctx->scratch[slot]) cudaFree(ctx->scratch[slot]);
    ctx->scratch[slot] = nullptr;
    ctx->scratch_bytes[slot] = 0;
    cudaError_t e = cudaMalloc(&ctx->scratch[slot], bytes);
    if (e != cudaSuccess) return fail(ctx, TS_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    ctx->scratch_bytes[slot] = bytes;
  }
  *out = ctx->scratch[slot];
  return TS_OK;
}

// A call's arrays.  in / out pass device pointers through (pointers_are_device) or stage host arrays into device
// memory the call owns; out and back queue the copies of results into host arrays.  start() opens the timed window of
// ts_last_kernel_ms.  finish() ends the call: it closes that window, checks the launches, runs the queued copies,
// synchronises the stream once and reads the time.  The first failure sticks in rc and makes the rest no-ops.
struct Staging {
  struct Back {
    void* host;
    const void* dev;
    size_t bytes;
  };
  ts_ctx* c;
  const int pointers_are_device;
  int rc = TS_OK;
  bool timed = false;
  std::vector<void*> owned;
  std::vector<Back> backs;
  Staging(ts_ctx* ctx, int pointers_are_device) : c(ctx), pointers_are_device(pointers_are_device) {}
  ~Staging() {
    for (void* p : owned) cudaFree(p);
  }
  void* alloc(size_t bytes) {
    void* d = nullptr;
    if (rc) return nullptr;
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e != cudaSuccess) {
      rc = fail(c, TS_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
      return nullptr;
    }
    owned.push_back(d);
    return d;
  }
  template <class T> const T* in(const T* p, size_t count) {
    if (!p || pointers_are_device || count == 0) return p;
    T* d = (T*)alloc(count * sizeof(T));
    if (!d) return nullptr;
    cudaError_t e = cudaMemcpyAsync(d, p, count * sizeof(T), cudaMemcpyHostToDevice, c->stream);
    if (e != cudaSuccess) rc = fail(c, TS_ERR_CUDA, "H2D copy failed: %s", cudaGetErrorString(e));
    return d;
  }
  template <class T> T* out(T* p, size_t count) {
    if (!p || pointers_are_device || count == 0) return p;
    T* d = (T*)alloc(count * sizeof(T));
    back(p, d, count);
    return d;
  }
  // an array the call reads and writes in place: staged in, and copied back at finish()
  template <class T> T* inout(T* p, size_t count) {
    if (!p || pointers_are_device || count == 0) return p;
    T* d = const_cast<T*>(in((const T*)p, count));
    back(p, d, count);
    return d;
  }
  template <class T> void back(T* host, const T* dev, size_t count) {
    if (!rc && count) backs.push_back({host, dev, count * sizeof(T)});
  }
  void start() {
    timed = true;
    cudaEventRecord(c->ev0, c->stream);
  }
  int finish() {
    if (rc) return rc;
    if (timed) cudaEventRecord(c->ev1, c->stream);
    TS_CUDA(c, cudaGetLastError());
    for (const Back& b : backs) {
      cudaError_t e = cudaMemcpyAsync(b.host, b.dev, b.bytes, cudaMemcpyDeviceToHost, c->stream);
      if (e != cudaSuccess) return fail(c, TS_ERR_CUDA, "D2H copy failed: %s", cudaGetErrorString(e));
    }
    TS_CUDA(c, cudaStreamSynchronize(c->stream));
    float ms = 0.f;
    if (timed && cudaEventElapsedTime(&ms, c->ev0, c->ev1) == cudaSuccess) c->last_kernel_ms = ms;
    return TS_OK;
  }
};

// small host array -> device scratch slot
template <class T>
inline int upload(ts_ctx* c, Slot slot, const T* host, size_t count, T** dev) {
  void* d = nullptr;
  int rc = scratch_reserve(c, slot, count * sizeof(T) + 16, &d);
  if (rc) return rc;
  TS_CUDA(c, cudaMemcpyAsync(d, host, count * sizeof(T), cudaMemcpyHostToDevice, c->stream));
  *dev = (T*)d;
  return TS_OK;
}

// a call's N timing events, destroyed when it returns; ms(a, b) is the time between the a-th and the b-th
template <int N> struct Events {
  cudaEvent_t e[N];
  Events() { for (cudaEvent_t& x : e) cudaEventCreate(&x); }
  ~Events() { for (cudaEvent_t x : e) cudaEventDestroy(x); }
  cudaEvent_t operator[](int i) const { return e[i]; }
  float ms(int a, int b) const {
    float t = 0.f;
    cudaEventElapsedTime(&t, e[a], e[b]);
    return t;
  }
};

}  // namespace ts
