// Several GPUs of one node behind one handle (SURVEY.md section 8b/8e): one ts_ctx per device, one host thread per
// device while a call runs, one NCCL communicator per device.  Trials are independent (reference
// src/monte_carlo.jl:118: the loop body touches only index i), so the only exchange is the end-of-run
// ncclAllGather of the 64-byte outcome records and the ncclAllReduce of the statistics vector.
// NCCL is bound at run time (dlopen of libnccl.so.2 on the first ts_create_multi with n_devices > 1): the single-GPU
// entry points carry no NCCL dependency, and a process that already has NCCL loaded (PyTorch) shares that copy.
#pragma once
#include <dlfcn.h>

#include <thread>

#include "common.cuh"

extern "C" int ts_monte_carlo_run(ts_ctx* c, const ts_mc_config* cfg, const double* kep6, const ts_field_opts* fopts, const double* x0,
                                  const double* xf, const double* Jmat, const double* q_noise0, const uint32_t* stream_id,
                                  ts_trial_outcome* out, ts_mc_stats* stats);
extern "C" int ts_mc_continue(ts_ctx* c, int64_t n_trials, const ts_ilqr_opts* opts, ts_trial_outcome* out, ts_mc_stats* stats);
extern "C" int ts_create(ts_ctx** out, int device_id);
extern "C" void ts_destroy(ts_ctx* c);
extern "C" const char* ts_last_error(const ts_ctx* c);

namespace ts {
// the slice of the NCCL API this library uses (types as in nccl.h 2.x)
typedef struct ncclComm* nccl_comm_t;
enum { NCCL_SUCCESS = 0, NCCL_CHAR = 0, NCCL_F64 = 8, NCCL_SUM = 0, NCCL_MAX = 2 };
struct NcclApi {
  void* lib = nullptr;
  int (*CommInitAll)(nccl_comm_t*, int, const int*) = nullptr;
  int (*CommDestroy)(nccl_comm_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool load(char* err, size_t errlen) {
    if (lib) return true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (lib) break;
    }
    if (!lib) {
      snprintf(err, errlen, "ts_create_multi: cannot load libnccl.so.2 (%s)", dlerror());
      return false;
    }
    CommInitAll = (decltype(CommInitAll))dlsym(lib, "ncclCommInitAll");
    CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
    AllGather = (decltype(AllGather))dlsym(lib, "ncclAllGather");
    AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
    GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
    if (!CommInitAll || !CommDestroy || !AllGather || !AllReduce) {
      snprintf(err, errlen, "ts_create_multi: libnccl.so.2 lacks an expected symbol");
      return false;
    }
    return true;
  }
};
}  // namespace ts

struct ts_multi {
  int n = 0;
  std::vector<int> dev;
  std::vector<ts_ctx*> ctx;
  ts::NcclApi nccl;
  std::vector<ts::nccl_comm_t> comms;
  std::vector<void*> d_send, d_recv;   // per device: outcome shard / gathered outcomes + statistics
  std::vector<size_t> d_bytes;
  char err[512] = {0};
};

namespace ts {

// statistics block <-> flat vectors for the two all-reduces (sum, max)
constexpr int MS_SUM = 17, MS_MAX = 4;
inline void stats_pack(const ts_mc_stats& s, double* sum, double* mx) {
  sum[0] = (double)s.n_trials; sum[1] = (double)s.n_converged; sum[2] = (double)s.n_no_cutoff; sum[3] = (double)s.n_fail_slew;
  sum[4] = s.sum_slew_time; sum[5] = s.sum_slew_time_sq; sum[6] = s.sum_t_final; sum[7] = s.sum_inner_iters;
  sum[8] = s.sum_ls_rollouts; sum[9] = s.sum_knots; sum[10] = s.flops;
  for (int i = 0; i < 6; ++i) sum[11 + i] = (double)s.n_status[i];
  mx[0] = s.ms_field; mx[1] = s.ms_prep; mx[2] = s.ms_solve; mx[3] = s.ms_tvlqr;
}
inline void stats_unpack(const double* sum, const double* mx, ts_mc_stats& s) {
  s.n_trials = (int64_t)llround(sum[0]); s.n_converged = (int64_t)llround(sum[1]); s.n_no_cutoff = (int64_t)llround(sum[2]);
  s.n_fail_slew = (int64_t)llround(sum[3]);
  s.sum_slew_time = sum[4]; s.sum_slew_time_sq = sum[5]; s.sum_t_final = sum[6]; s.sum_inner_iters = sum[7];
  s.sum_ls_rollouts = sum[8]; s.sum_knots = sum[9]; s.flops = sum[10];
  for (int i = 0; i < 6; ++i) s.n_status[i] = (int64_t)llround(sum[11 + i]);
  s.ms_field = mx[0]; s.ms_prep = mx[1]; s.ms_solve = mx[2]; s.ms_tvlqr = mx[3];
}

// Runs `shard(g, c, ng, shard_out, shard_stats)` for every device's shard (trials g, g+G, g+2G, ...) on the device's own
// thread, then gathers the 64-byte outcome records with ncclAllGather and reduces the statistics with ncclAllReduce
// (sum; ms_* max).  `out` and `stats` are written only when every shard succeeded.
template <class Shard>
inline int multi_shards(ts_multi* m, int64_t n, Shard&& shard, ts_trial_outcome* out, ts_mc_stats* stats) {
  const int G = m->n;
  const int64_t per = (n + G - 1) / G;   // records per device in the gather (short shards are padded)
  std::vector<int> rcs(G, TS_OK);
  std::vector<std::vector<ts_trial_outcome>> shard_out(G);
  std::vector<ts_mc_stats> shard_stats(G);
  std::vector<std::vector<ts_trial_outcome>> gathered(G);
  std::vector<std::vector<double>> red(G);
  auto worker = [&](int g) {
    ts_ctx* c = m->ctx[g];
    const int64_t ng = (n - g + G - 1) / G;
    shard_out[g].assign((size_t)per, ts_trial_outcome{});
    memset(&shard_stats[g], 0, sizeof(ts_mc_stats));
    rcs[g] = ng > 0 ? shard(g, c, ng, shard_out[g].data(), &shard_stats[g]) : TS_OK;
    if (G == 1) return;
    // ---- exchange (every rank takes part even after a local failure, so that nobody hangs in the collective)
    cudaSetDevice(m->dev[g]);
    const size_t rec = sizeof(ts_trial_outcome);
    const size_t b_send = (size_t)per * rec, b_recv = (size_t)per * rec * G;
    const size_t b_red = (size_t)(MS_SUM + MS_MAX) * sizeof(double);
    const size_t need = b_recv + 2 * b_red + 256;
    if (m->d_bytes[g] < need) {
      if (m->d_send[g]) cudaFree(m->d_send[g]);
      if (m->d_recv[g]) cudaFree(m->d_recv[g]);
      cudaMalloc(&m->d_send[g], b_send + b_red + 256);
      cudaMalloc(&m->d_recv[g], need);
      m->d_bytes[g] = need;
    }
    double hsum[MS_SUM + MS_MAX];
    stats_pack(shard_stats[g], hsum, hsum + MS_SUM);
    char* ds = (char*)m->d_send[g];
    char* dr = (char*)m->d_recv[g];
    cudaMemcpyAsync(ds, shard_out[g].data(), b_send, cudaMemcpyHostToDevice, c->stream);
    cudaMemcpyAsync(ds + b_send, hsum, b_red, cudaMemcpyHostToDevice, c->stream);
    int e = m->nccl.AllGather(ds, dr, b_send, NCCL_CHAR, m->comms[g], c->stream);
    if (e == NCCL_SUCCESS) e = m->nccl.AllReduce(ds + b_send, dr + b_recv, MS_SUM, NCCL_F64, NCCL_SUM, m->comms[g], c->stream);
    if (e == NCCL_SUCCESS)
      e = m->nccl.AllReduce(ds + b_send + MS_SUM * sizeof(double), dr + b_recv + MS_SUM * sizeof(double), MS_MAX, NCCL_F64, NCCL_MAX,
                            m->comms[g], c->stream);
    if (e != NCCL_SUCCESS && rcs[g] == TS_OK) rcs[g] = TS_ERR_CUDA;
    gathered[g].resize((size_t)per * G);
    red[g].resize(MS_SUM + MS_MAX);
    cudaMemcpyAsync(gathered[g].data(), dr, b_recv, cudaMemcpyDeviceToHost, c->stream);
    cudaMemcpyAsync(red[g].data(), dr + b_recv, b_red, cudaMemcpyDeviceToHost, c->stream);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess && rcs[g] == TS_OK) rcs[g] = TS_ERR_CUDA;
  };
  std::vector<std::thread> th;
  for (int g = 0; g < G; ++g) th.emplace_back(worker, g);
  for (auto& t : th) t.join();
  for (int g = 0; g < G; ++g)
    if (rcs[g] != TS_OK) {
      snprintf(m->err, sizeof(m->err), "device %d: %s", m->dev[g], ts_last_error(m->ctx[g]));
      return rcs[g];
    }
  if (G == 1) {
    memcpy(out, shard_out[0].data(), (size_t)n * sizeof(ts_trial_outcome));
    if (stats) *stats = shard_stats[0];
    return TS_OK;
  }
  // every rank now holds all records (rank-major, `per` per rank): hand rank 0's copy back in the caller's trial order
  for (int g = 0; g < G; ++g)
    for (int64_t a = 0; g + a * G < n; ++a) out[g + a * G] = gathered[0][(size_t)g * per + a];
  if (stats) stats_unpack(red[0].data(), red[0].data() + MS_SUM, *stats);
  return TS_OK;
}

}  // namespace ts

extern "C" {

int ts_create_multi(ts_multi** out, const int* device_ids, int n_devices) {
  if (!out) return TS_ERR_ARG;
  *out = nullptr;
  if (!device_ids || n_devices < 1 || n_devices > 64) return TS_ERR_ARG;
  ts_multi* m = new ts_multi();
  m->n = n_devices;
  m->dev.assign(device_ids, device_ids + n_devices);
  for (int i = 0; i < n_devices; ++i) {
    ts_ctx* c = nullptr;
    const int rc = ts_create(&c, device_ids[i]);
    if (rc != TS_OK) {
      for (ts_ctx* p : m->ctx) ts_destroy(p);
      delete m;
      return rc;
    }
    m->ctx.push_back(c);
  }
  m->d_send.assign(n_devices, nullptr);
  m->d_recv.assign(n_devices, nullptr);
  m->d_bytes.assign(n_devices, 0);
  if (n_devices > 1) {
    if (!m->nccl.load(m->err, sizeof(m->err))) {
      fprintf(stderr, "%s\n", m->err);
      for (ts_ctx* p : m->ctx) ts_destroy(p);
      delete m;
      return TS_ERR_CUDA;
    }
    m->comms.assign(n_devices, nullptr);
    const int e = m->nccl.CommInitAll(m->comms.data(), n_devices, device_ids);
    if (e != ts::NCCL_SUCCESS) {
      fprintf(stderr, "ts_create_multi: ncclCommInitAll failed: %s\n", m->nccl.GetErrorString ? m->nccl.GetErrorString(e) : "?");
      for (ts_ctx* p : m->ctx) ts_destroy(p);
      delete m;
      return TS_ERR_CUDA;
    }
  }
  *out = m;
  return TS_OK;
}

void ts_destroy_multi(ts_multi* m) {
  if (!m) return;
  for (int i = 0; i < m->n; ++i) {
    cudaSetDevice(m->dev[i]);
    if (i < (int)m->comms.size() && m->comms[i]) m->nccl.CommDestroy(m->comms[i]);
    if (m->d_send[i]) cudaFree(m->d_send[i]);
    if (m->d_recv[i]) cudaFree(m->d_recv[i]);
    ts_destroy(m->ctx[i]);
  }
  delete m;
}

const char* ts_multi_last_error(const ts_multi* m) { return m ? m->err : "null handle"; }
int ts_multi_device_count(const ts_multi* m) { return m ? m->n : 0; }
ts_ctx* ts_multi_ctx(ts_multi* m, int i) { return (m && i >= 0 && i < m->n) ? m->ctx[i] : nullptr; }

int ts_multi_monte_carlo_run(ts_multi* m, const ts_mc_config* cfg, const double* kep6, const ts_field_opts* fopts, const double* x0,
                             const double* xf, const double* Jmat, const double* q_noise0, const uint32_t* stream_id,
                             ts_trial_outcome* out, ts_mc_stats* stats) {
  if (!m) return TS_ERR_ARG;
  if (!cfg || !kep6 || !fopts || !x0 || !xf || !Jmat || !out) {
    snprintf(m->err, sizeof(m->err), "ts_multi_monte_carlo_run: null argument");
    return TS_ERR_ARG;
  }
  const int G = m->n;
  const int64_t n = cfg->n_trials;
  if (stats) memset(stats, 0, sizeof(*stats));
  if (n <= 0) return n == 0 ? TS_OK : TS_ERR_ARG;
  auto shard = [&](int g, ts_ctx* c, int64_t ng, ts_trial_outcome* so, ts_mc_stats* ss) {
    ts_mc_config cg = *cfg;
    cg.n_trials = ng;
    std::vector<double> sx0((size_t)ng * 8), sxf((size_t)ng * 8), sJ((size_t)ng * 9), sq, skep;
    std::vector<uint32_t> sid((size_t)ng);
    std::vector<ts_field_opts> sfo;
    if (q_noise0) sq.resize((size_t)ng * 3);
    if (!cfg->shared_orbit) {
      skep.resize((size_t)ng * 6);
      sfo.resize((size_t)ng);
    }
    for (int64_t a = 0; a < ng; ++a) {
      const int64_t t = g + a * G;
      memcpy(&sx0[a * 8], x0 + t * 8, 64);
      memcpy(&sxf[a * 8], xf + t * 8, 64);
      memcpy(&sJ[a * 9], Jmat + t * 9, 72);
      if (q_noise0) memcpy(&sq[a * 3], q_noise0 + t * 3, 24);
      sid[a] = stream_id ? stream_id[t] : (uint32_t)t;   // Philox streams keyed by the GLOBAL trial id: results do not depend on G
      if (!cfg->shared_orbit) {
        memcpy(&skep[a * 6], kep6 + t * 6, 48);
        sfo[a] = fopts[t];
      }
    }
    return ts_monte_carlo_run(c, &cg, cfg->shared_orbit ? kep6 : skep.data(), cfg->shared_orbit ? fopts : sfo.data(), sx0.data(),
                              sxf.data(), sJ.data(), q_noise0 ? sq.data() : nullptr, sid.data(), so, ss);
  };
  return multi_shards(m, n, shard, out, stats);
}

int ts_multi_mc_continue(ts_multi* m, int64_t n_trials, const ts_ilqr_opts* opts, ts_trial_outcome* out, ts_mc_stats* stats) {
  if (!m) return TS_ERR_ARG;
  if (!opts || !out || n_trials < 0) {
    snprintf(m->err, sizeof(m->err), "ts_multi_mc_continue: null argument or n_trials < 0");
    return TS_ERR_ARG;
  }
  if (n_trials == 0) return TS_OK;
  auto shard = [&](int, ts_ctx* c, int64_t ng, ts_trial_outcome* so, ts_mc_stats* ss) { return ts_mc_continue(c, ng, opts, so, ss); };
  return multi_shards(m, n_trials, shard, out, stats);
}

// ts_multi_mc_replay_ensemble, ts_multi_mc_dispersion_ensemble (dispersed) and ts_multi_mc_weight_ensemble (ws): each
// trial on the device that holds it, all devices at once, rows back in the caller's order.  The argument checks of the
// single-device entry run before any device does: a failure leaves the outputs untouched.
static int multi_ensemble(ts_multi* m, const char* fn, int64_t n_trials, const ts_replay_ensemble_opts* opts, bool dispersed,
                          const ts_dispersion_opts* disp, int64_t n_sel, const int64_t* trials, double* slew_time, double* x_final,
                          double* params, const WeightSets* ws = nullptr) {
  if (!m) return TS_ERR_ARG;
  const int G = m->n;
  bool bad = n_trials < 0 || !opts || !slew_time || (trials ? n_sel < 0 : n_sel != n_trials) || (dispersed && !disp);
  if (!bad) bad = opts->n_real < 1 || opts->r_first < 0 || opts->r_first + opts->n_real > ((int64_t)1 << 30);
  if (!bad && disp) bad = !ts::dispersion_opts_ok(disp);
  if (!bad && ws) bad = !ts::weight_sets_ok(ws->n, ws->sets, ws->u_limit);
  for (int64_t p = 0; !bad && trials && p < n_sel; ++p) bad = trials[p] < 0 || trials[p] >= n_trials;
  if (bad) {
    snprintf(m->err, sizeof(m->err), "%s: bad argument", fn);
    return TS_ERR_ARG;
  }
  const size_t RR = (size_t)opts->n_real * (ws ? (size_t)ws->n : 1), NP = ts::DISP_NP;   // RR: slew times per trial
  std::vector<std::vector<int64_t>> pos(G), loc(G);   // caller rows and device-local trial indices per device
  for (int64_t p = 0; p < n_sel; ++p) {
    const int64_t t = trials ? trials[p] : p;
    pos[t % G].push_back(p);
    loc[t % G].push_back(t / G);
  }
  std::vector<int> rcs(G, TS_OK);
  std::vector<std::vector<double>> hs(G), hx(G), hp(G);
  auto worker = [&](int g) {
    if (pos[g].empty()) return;
    const int64_t ng = (n_trials - g + G - 1) / G;
    const size_t k = pos[g].size();
    hs[g].resize(k * RR);
    if (x_final) hx[g].resize(k * RR * 8);
    if (params) hp[g].resize(k * RR * NP);
    double* px = x_final ? hx[g].data() : nullptr;
    rcs[g] = ws          ? ts_mc_weight_ensemble(m->ctx[g], ng, opts, disp, ws->n, ws->sets, ws->u_limit, (int64_t)k, loc[g].data(),
                                                 hs[g].data(), px)
             : dispersed ? ts_mc_dispersion_ensemble(m->ctx[g], ng, opts, disp, (int64_t)k, loc[g].data(), hs[g].data(), px,
                                                     params ? hp[g].data() : nullptr)
                         : ts_mc_replay_ensemble(m->ctx[g], ng, opts, (int64_t)k, loc[g].data(), hs[g].data(), px);
  };
  std::vector<std::thread> th;
  for (int g = 0; g < G; ++g) th.emplace_back(worker, g);
  for (auto& t : th) t.join();
  for (int g = 0; g < G; ++g)
    if (rcs[g] != TS_OK) {
      snprintf(m->err, sizeof(m->err), "device %d: %s", m->dev[g], ts_last_error(m->ctx[g]));
      return rcs[g];
    }
  for (int g = 0; g < G; ++g)
    for (size_t k = 0; k < pos[g].size(); ++k) {
      const size_t p = (size_t)pos[g][k];
      memcpy(slew_time + p * RR, &hs[g][k * RR], RR * 8);
      if (x_final) memcpy(x_final + p * RR * 8, &hx[g][k * RR * 8], RR * 64);
      if (params) memcpy(params + p * RR * NP, &hp[g][k * RR * NP], RR * NP * 8);
    }
  return TS_OK;
}

int ts_multi_mc_replay_ensemble(ts_multi* m, int64_t n_trials, const ts_replay_ensemble_opts* opts, int64_t n_sel, const int64_t* trials,
                                double* slew_time, double* x_final) {
  return multi_ensemble(m, "ts_multi_mc_replay_ensemble", n_trials, opts, false, nullptr, n_sel, trials, slew_time, x_final, nullptr);
}

int ts_multi_mc_dispersion_ensemble(ts_multi* m, int64_t n_trials, const ts_replay_ensemble_opts* opts, const ts_dispersion_opts* disp,
                                    int64_t n_sel, const int64_t* trials, double* slew_time, double* x_final, double* params) {
  return multi_ensemble(m, "ts_multi_mc_dispersion_ensemble", n_trials, opts, true, disp, n_sel, trials, slew_time, x_final, params);
}

int ts_multi_mc_weight_ensemble(ts_multi* m, int64_t n_trials, const ts_replay_ensemble_opts* opts, const ts_dispersion_opts* disp,
                                int64_t n_sets, const ts_tvlqr_weights* sets, double u_limit, int64_t n_sel, const int64_t* trials,
                                double* slew_time, double* x_final) {
  const WeightSets ws = {n_sets, sets, u_limit};
  return multi_ensemble(m, "ts_multi_mc_weight_ensemble", n_trials, opts, false, disp, n_sel, trials, slew_time, x_final, nullptr, &ws);
}

}  // extern "C"
