// libtortoise_b200.so -- single translation unit: context + C-ABI entry points.
// Kernels live in the k*_*.cuh files included below.  sm_100a only; there is no
// CPU fallback anywhere in this library.
#include "common.cuh"
#include "igrf_device.cuh"
#include "k1_igrf.cuh"
#include "k2_field.cuh"
#include "k3_alilqr.cuh"
#include "k4_tvlqr.cuh"
#include "k5_unitops.cuh"
#include "k6_igrf12syn.cuh"
#include "k7_comparison.cuh"
#include "k8_field_map.cuh"

#include <algorithm>
#include <numeric>
#include <utility>

namespace ts {
#include "igrf12_tables.inc"
}

using namespace ts;

extern "C" {

int ts_version(void) { return 104; }

int ts_create(ts_ctx** out, int device_id) {
  if (!out) return TS_ERR_ARG;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return TS_ERR_CUDA;  // no GPU -> no library (no CPU fallback)
  if (device_id < 0 || device_id >= ndev) return TS_ERR_ARG;
  ts_ctx* c = new ts_ctx();
  c->device = device_id;
  if (cudaSetDevice(device_id) != cudaSuccess) {
    delete c;
    return TS_ERR_CUDA;
  }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device_id);
  c->sm_count = prop.multiProcessorCount;
  snprintf(c->name, sizeof(c->name), "%s", prop.name);
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess ||
      cudaEventCreate(&c->ev_k3[0]) != cudaSuccess || cudaEventCreate(&c->ev_k3[1]) != cudaSuccess ||
      cudaEventCreate(&c->ev_k3[2]) != cudaSuccess ||
      cudaMalloc(&c->d_tabG, sizeof(TS_IGRF12_G)) != cudaSuccess || cudaMalloc(&c->d_tabH, sizeof(TS_IGRF12_H)) != cudaSuccess ||
      cudaMalloc(&c->d_tabGH, sizeof(TS_IGRF12_GH)) != cudaSuccess || cudaMalloc(&c->d_flag, 64) != cudaSuccess ||
      cudaMalloc(&c->d_gh_stage, 2 * IGRF_NCOEF * sizeof(double2)) != cudaSuccess) {
    ts_destroy(c);
    return TS_ERR_CUDA;
  }
  cudaMemcpy(c->d_tabG, TS_IGRF12_G, sizeof(TS_IGRF12_G), cudaMemcpyHostToDevice);
  cudaMemcpy(c->d_tabH, TS_IGRF12_H, sizeof(TS_IGRF12_H), cudaMemcpyHostToDevice);
  cudaMemcpy(c->d_tabGH, TS_IGRF12_GH, sizeof(TS_IGRF12_GH), cudaMemcpyHostToDevice);
  IgrfConsts h;
  igrf_host_constants(h);
  if (cudaMemcpyToSymbol(c_igrf, &h, sizeof(h)) != cudaSuccess) {
    ts_destroy(c);
    return TS_ERR_CUDA;
  }
  cudaMemset(c->d_flag, 0, 64);
  *out = c;
  return TS_OK;
}

void ts_destroy(ts_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  for (int i = 0; i < SLOT_COUNT; ++i)
    if (c->scratch[i]) cudaFree(c->scratch[i]);
  if (c->d_tabG) cudaFree(c->d_tabG);
  if (c->d_tabH) cudaFree(c->d_tabH);
  if (c->d_tabGH) cudaFree(c->d_tabGH);
  if (c->d_flag) cudaFree(c->d_flag);
  if (c->d_gh_stage) cudaFree(c->d_gh_stage);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  for (int i = 0; i < 3; ++i)
    if (c->ev_k3[i]) cudaEventDestroy(c->ev_k3[i]);
  for (int i = 0; i < 2; ++i)
    if (c->pipe[i]) cudaStreamDestroy(c->pipe[i]);
  if (c->pipe_ev) cudaEventDestroy(c->pipe_ev);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

const char* ts_last_error(const ts_ctx* c) { return c ? c->err : "null context"; }
int64_t ts_launch_count(const ts_ctx* c) { return c ? c->launches : 0; }
double ts_last_kernel_ms(const ts_ctx* c) { return c ? c->last_kernel_ms : 0.0; }
int ts_k3_last_split(ts_ctx* c, double* persistent_ms, double* straggler_ms, int64_t* n_parked) {
  if (!c) return TS_ERR_ARG;
  if (persistent_ms) *persistent_ms = 0.0;
  if (straggler_ms) *straggler_ms = 0.0;
  if (n_parked) *n_parked = 0;
  if (!c->k3_timed) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  TS_CUDA(c, cudaStreamSynchronize(c->stream));
  float a = 0.f, b = 0.f;
  TS_CUDA(c, cudaEventElapsedTime(&a, c->ev_k3[0], c->ev_k3[1]));
  TS_CUDA(c, cudaEventElapsedTime(&b, c->ev_k3[1], c->ev_k3[2]));
  unsigned np = 0;
  if (c->d_k3_parked) TS_CUDA(c, cudaMemcpy(&np, c->d_k3_parked, sizeof(np), cudaMemcpyDeviceToHost));
  if (persistent_ms) *persistent_ms = a;
  if (straggler_ms) *straggler_ms = b;
  if (np > (unsigned)c->k3_park_cap) np = (unsigned)c->k3_park_cap;   // the device counter may overshoot the parking places
  if (n_parked) *n_parked = (int64_t)np;
  return TS_OK;
}

int ts_k3_last_parked(ts_ctx* c, int64_t cap, int64_t* trial, int32_t* outer_at_park, int32_t* inner_at_park, int64_t* n_out) {
  if (!c || !n_out || cap < 0 || (cap > 0 && (!trial || !outer_at_park || !inner_at_park))) return TS_ERR_ARG;
  *n_out = 0;
  if (!c->k3_timed || !c->d_k3_parked || c->k3_park_cap <= 0 || !c->scratch[SLOT_PARK_STATE]) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  TS_CUDA(c, cudaStreamSynchronize(c->stream));
  unsigned np = 0;
  TS_CUDA(c, cudaMemcpy(&np, c->d_k3_parked, sizeof(np), cudaMemcpyDeviceToHost));
  if (np > (unsigned)c->k3_park_cap) np = (unsigned)c->k3_park_cap;
  const size_t n = std::min<size_t>((size_t)np, (size_t)cap), pc = (size_t)c->k3_park_cap;
  std::vector<TrialState> st(n);
  std::vector<int64_t> tr(n);
  if (n) {
    TS_CUDA(c, cudaMemcpy(st.data(), c->scratch[SLOT_PARK_STATE], n * sizeof(TrialState), cudaMemcpyDeviceToHost));
    TS_CUDA(c, cudaMemcpy(tr.data(), (const char*)c->scratch[SLOT_PARK_STATE] + pc * sizeof(TrialState), n * 8, cudaMemcpyDeviceToHost));
  }
  for (size_t i = 0; i < n; ++i) {
    trial[i] = tr[i];
    outer_at_park[i] = st[i].outer;
    inner_at_park[i] = st[i].inner_total;
  }
  *n_out = (int64_t)n;
  return TS_OK;
}

int ts_k3_last_cycles(ts_ctx* c, int64_t n_trials, double* cycles3) {
  if (!c || !cycles3 || n_trials < 0) return TS_ERR_ARG;
  if (n_trials > c->k3_diag_n || !c->scratch[SLOT_K3_CYCLES]) return fail(c, TS_ERR_ARG, "ts_k3_last_cycles: the last solve covered %lld trials", (long long)c->k3_diag_n);
  TS_CUDA(c, cudaSetDevice(c->device));
  TS_CUDA(c, cudaStreamSynchronize(c->stream));
  TS_CUDA(c, cudaMemcpy(cycles3, c->scratch[SLOT_K3_CYCLES], (size_t)n_trials * 3 * sizeof(double), cudaMemcpyDeviceToHost));
  return TS_OK;
}

int ts_device_info(ts_ctx* c, int* sm_count, char* name, int name_len) {
  if (!c) return TS_ERR_ARG;
  if (sm_count) *sm_count = c->sm_count;
  if (name && name_len > 0) snprintf(name, (size_t)name_len, "%s", c->name);
  return TS_OK;
}

int ts_synchronize(ts_ctx* c) {
  if (!c) return TS_ERR_ARG;
  TS_CUDA(c, cudaSetDevice(c->device));
  TS_CUDA(c, cudaStreamSynchronize(c->stream));
  return TS_OK;
}

int ts_fp64_peak_probe(ts_ctx* c, double* tflops_out) {
  if (!c || !tflops_out) return TS_ERR_ARG;
  TS_CUDA(c, cudaSetDevice(c->device));
  const int iters = 4096, blocks = c->sm_count * 8, threads = 256;
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    Staging io(c, 0);
    io.start();
    fp64_peak_kernel<<<blocks, threads, 0, c->stream>>>((double*)c->d_flag + 1, iters, 1.0000001, 1e-9);
    c->launches++;
    if (int rc = io.finish()) return rc;
    const double flops = 2.0 * 8 * 16 * (double)iters * (double)blocks * threads;
    const double tf = flops / (c->last_kernel_ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  *tflops_out = best;
  return TS_OK;
}

int ts_fp64_latency_probe(ts_ctx* c, double* cycles4) {
  if (!c || !cycles4) return TS_ERR_ARG;
  TS_CUDA(c, cudaSetDevice(c->device));
  double* d = (double*)c->d_flag;   // 64 bytes
  for (int rep = 0; rep < 2; ++rep) {
    fp64_latency_kernel<<<1, 32, 0, c->stream>>>(d + 1, 2048, 1.0000001, 1e-9);
    c->launches++;
  }
  TS_CUDA(c, cudaGetLastError());
  TS_CUDA(c, cudaStreamSynchronize(c->stream));
  TS_CUDA(c, cudaMemcpy(cycles4, d + 1, 4 * sizeof(double), cudaMemcpyDeviceToHost));
  return TS_OK;
}

// the dates igrf12 / igrf12syn accept
static bool igrf_date_ok(double date) { return date >= 1900.0 && date <= 2025.0; }

// Reads back c->d_flag after the call's other results and turns a set flag into TS_ERR_DOMAIN (K1, K8).
static int finish_domain_checked(ts_ctx* c, Staging& io, const char* msg) {
  int bad = 0;
  io.back(&bad, (const int*)c->d_flag, 1);
  if (int rc = io.finish()) return rc;
  return bad ? fail(c, TS_ERR_DOMAIN, "%s", msg) : TS_OK;
}

static const char* const K1_DOMAIN_MSG =
    "The latitude must be between -pi/2 and +pi/2 rad and the longitude between -pi and +pi rad.";

// the call's coefficient table (c->d_gh_stage), queued on the context's stream ahead of the K1 launches that read it
static void k1_stage(ts_ctx* c, double date) {
  k1_stage_kernel<<<1, 128, 0, c->stream>>>(c->d_tabG, c->d_tabH, date, (double2*)c->d_gh_stage);
  c->launches++;
}
static void k1_launch(ts_ctx* c, cudaStream_t st, double date, int64_t n, const double* r, const double* la, const double* lo,
                      double* bn, double* be, double* bd) {
  const unsigned blocks = (unsigned)((n + K1_THREADS - 1) / K1_THREADS);
  const double2* gh = (const double2*)c->d_gh_stage;
  if (igrf_nmax_for_date(date) == 13)
    k1_igrf12_batch<13><<<blocks, K1_THREADS, 0, st>>>(gh, n, r, la, lo, bn, be, bd, c->d_flag);
  else
    k1_igrf12_batch<10><<<blocks, K1_THREADS, 0, st>>>(gh, n, r, la, lo, bn, be, bd, c->d_flag);
  c->launches++;
}

// Host-pointer path of ts_igrf12_batch: the call is PCIe-bound (24 B in + 24 B out per point against ~20 ns of
// FP64 work per 1000 points), so the points go through two device staging sets on two streams: the upload of
// chunk k+1 and the download of chunk k-1 overlap the kernel of chunk k (full-duplex link), and no device
// memory is allocated per call.
static int igrf12_host_pipeline(ts_ctx* c, double date, int64_t n, const double* r_m, const double* lat, const double* lon,
                                double* Bn, double* Be, double* Bd) {
  constexpr int64_t CHUNK = 1 << 22;
  for (int i = 0; i < 2; ++i)
    if (!c->pipe[i]) TS_CUDA(c, cudaStreamCreateWithFlags(&c->pipe[i], cudaStreamNonBlocking));
  if (!c->pipe_ev) TS_CUDA(c, cudaEventCreateWithFlags(&c->pipe_ev, cudaEventDisableTiming));
  const int64_t chunk = std::min<int64_t>(CHUNK, n);
  double* stage[2];
  int rc;
  for (int i = 0; i < 2; ++i) {
    void* p;
    if ((rc = scratch_reserve(c, i ? SLOT_PIPE_B : SLOT_PIPE_A, (size_t)chunk * 6 * sizeof(double), &p))) return rc;
    stage[i] = (double*)p;
  }
  TS_CUDA(c, cudaMemsetAsync(c->d_flag, 0, sizeof(int), c->stream));
  k1_stage(c, date);   // both pipeline streams wait for pipe_ev
  TS_CUDA(c, cudaEventRecord(c->pipe_ev, c->stream));
  const int64_t n_chunks = (n + chunk - 1) / chunk;
  std::vector<cudaEvent_t> ev((size_t)n_chunks * 2, nullptr);
  for (auto& e : ev) cudaEventCreate(&e);
  cudaError_t err = cudaSuccess;
  for (int i = 0; i < 2 && err == cudaSuccess; ++i) err = cudaStreamWaitEvent(c->pipe[i], c->pipe_ev, 0);
  for (int64_t k = 0; k < n_chunks && err == cudaSuccess; ++k) {
    cudaStream_t st = c->pipe[k & 1];
    double* d = stage[k & 1];
    const int64_t o = k * chunk, m = std::min<int64_t>(chunk, n - o);
    const size_t b = (size_t)m * sizeof(double);
    if (err == cudaSuccess) err = cudaMemcpyAsync(d, r_m + o, b, cudaMemcpyHostToDevice, st);
    if (err == cudaSuccess) err = cudaMemcpyAsync(d + chunk, lat + o, b, cudaMemcpyHostToDevice, st);
    if (err == cudaSuccess) err = cudaMemcpyAsync(d + 2 * chunk, lon + o, b, cudaMemcpyHostToDevice, st);
    cudaEventRecord(ev[(size_t)k * 2], st);
    k1_launch(c, st, date, m, d, d + chunk, d + 2 * chunk, d + 3 * chunk, d + 4 * chunk, d + 5 * chunk);
    cudaEventRecord(ev[(size_t)k * 2 + 1], st);
    if (err == cudaSuccess) err = cudaGetLastError();
    if (err == cudaSuccess) err = cudaMemcpyAsync(Bn + o, d + 3 * chunk, b, cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaMemcpyAsync(Be + o, d + 4 * chunk, b, cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaMemcpyAsync(Bd + o, d + 5 * chunk, b, cudaMemcpyDeviceToHost, st);
  }
  for (int i = 0; i < 2; ++i) {
    const cudaError_t e2 = cudaStreamSynchronize(c->pipe[i]);
    if (err == cudaSuccess) err = e2;
  }
  double ms_sum = 0.0;
  for (int64_t k = 0; k < n_chunks; ++k) {
    float ms = 0.f;
    if (err == cudaSuccess && cudaEventElapsedTime(&ms, ev[(size_t)k * 2], ev[(size_t)k * 2 + 1]) == cudaSuccess) ms_sum += ms;
  }
  for (auto& e : ev)
    if (e) cudaEventDestroy(e);
  if (err != cudaSuccess) return fail(c, TS_ERR_CUDA, "ts_igrf12_batch (host pipeline): %s", cudaGetErrorString(err));
  c->last_kernel_ms = ms_sum;
  Staging io(c, 0);
  return finish_domain_checked(c, io, K1_DOMAIN_MSG);
}

int ts_igrf12_batch(ts_ctx* c, double date, int64_t n, const double* r_m, const double* lat, const double* lon, double* Bn,
                    double* Be, double* Bd, int pointers_are_device) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || (n > 0 && (!r_m || !lat || !lon || !Bn || !Be || !Bd))) return fail(c, TS_ERR_ARG, "ts_igrf12_batch: null array or n<0");
  if (!igrf_date_ok(date))
    return fail(c, TS_ERR_DATE, "This IGRF version will not work for years outside the interval [1900, 2025).");
  if (n == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  if (!pointers_are_device) return igrf12_host_pipeline(c, date, n, r_m, lat, lon, Bn, Be, Bd);
  TS_CUDA(c, cudaMemsetAsync(c->d_flag, 0, sizeof(int), c->stream));
  Staging io(c, pointers_are_device);
  io.start();
  k1_stage(c, date);
  k1_launch(c, c->stream, date, n, r_m, lat, lon, Bn, Be, Bd);
  return finish_domain_checked(c, io, K1_DOMAIN_MSG);
}

// igrf12syn(isv,date,itype,alt,colat,elong) [src/igrf.jl:335-534] at n points
int ts_igrf12syn_batch(ts_ctx* c, int isv, double date, int itype, int64_t n, const double* alt_km, const double* colat_deg,
                       const double* elong_deg, double* x, double* y, double* z, double* f, int pointers_are_device) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || (n > 0 && (!alt_km || !colat_deg || !elong_deg || !x || !y || !z || !f))) return fail(c, TS_ERR_ARG, "ts_igrf12syn_batch: null array or n<0");
  if (isv != 0 && isv != 1) return fail(c, TS_ERR_ARG, "ts_igrf12syn_batch: isv must be 0 or 1");
  if (itype != 1 && itype != 2) return fail(c, TS_ERR_ARG, "ts_igrf12syn_batch: itype must be 1 (geodetic) or 2 (geocentric)");
  if (!igrf_date_ok(date))
    return fail(c, TS_ERR_DATE, "This IGRF version will not work for years outside the interval [1900, 2025).");
  if (n == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  Staging io(c, pointers_are_device);
  const size_t m = (size_t)n;
  const double *da = io.in(alt_km, m), *dc = io.in(colat_deg, m), *de = io.in(elong_deg, m);
  double *ox = io.out(x, m), *oy = io.out(y, m), *oz = io.out(z, m), *of = io.out(f, m);
  if (io.rc) return io.rc;
  const SynEpoch ep = igrf12syn_epoch(isv, date);
  io.start();
  k6_igrf12syn<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(c->d_tabGH, ep, itype, n, da, dc, de, ox, oy, oz, of);
  c->launches++;
  return io.finish();
}

// ---------------------------------------------------------------------------- K8
static int field_map_dims(ts_ctx* c, const char* fn, int64_t n0, int64_t n1) {
  if (n0 < 2 || n1 < 2 || n0 > K8_MAX_AXIS || n1 > K8_MAX_AXIS)
    return fail(c, TS_ERR_ARG, "%s: n0 = %lld and n1 = %lld must lie in [2, %lld]", fn, (long long)n0, (long long)n1,
                (long long)K8_MAX_AXIS);
  return TS_OK;
}

// FM1: Thomas solves along axis 1 (j) for every data row, then along axis 0 (i) for every padded column.  The j-lines
// are made columns by a tiled transpose into a (n1+2) x n0 x 3 buffer, solved in place, and transposed into rows
// 1..n0 of C, where the i-pass solves in place.
int ts_field_map_prefilter(ts_ctx* c, int64_t n0, int64_t n1, const double* grid, double* coefs, int pointers_are_device) {
  if (!c) return TS_ERR_ARG;
  if (!grid || !coefs) return fail(c, TS_ERR_ARG, "ts_field_map_prefilter: null array");
  int rc;
  if ((rc = field_map_dims(c, "ts_field_map_prefilter", n0, n1))) return rc;
  TS_CUDA(c, cudaSetDevice(c->device));
  std::vector<double> inv((size_t)(n0 + n1));
  k8_thomas_factors(n0, inv.data());
  k8_thomas_factors(n1, inv.data() + n0);
  Staging io(c, pointers_are_device), host(c, 0);   // the factors are always a host array
  const double* G = io.in(grid, (size_t)n0 * n1 * 3);
  double* Cf = io.out(coefs, (size_t)(n0 + 2) * (n1 + 2) * 3);
  const double* inv0 = host.in(inv.data(), inv.size());
  double* T = (double*)io.alloc((size_t)(n1 + 2) * n0 * 3 * sizeof(double));
  if (io.rc || host.rc) return io.rc ? io.rc : host.rc;
  const double* inv1 = inv0 + n0;
  const dim3 tb(K8_TILE, 8);
  io.start();
  k8_transpose3<<<dim3((unsigned)((n1 + K8_TILE - 1) / K8_TILE), (unsigned)((n0 + K8_TILE - 1) / K8_TILE)), tb, 0, c->stream>>>(
      G, n0, n1, T + n0 * 3, n0 * 3);
  k8_prefilter_cols<<<(unsigned)((n0 * 3 + 127) / 128), 128, 0, c->stream>>>(T, n1, n0 * 3, inv1);
  k8_transpose3<<<dim3((unsigned)((n0 + K8_TILE - 1) / K8_TILE), (unsigned)((n1 + 2 + K8_TILE - 1) / K8_TILE)), tb, 0, c->stream>>>(
      T, n1 + 2, n0, Cf + (n1 + 2) * 3, (n1 + 2) * 3);
  k8_prefilter_cols<<<(unsigned)(((n1 + 2) * 3 + 127) / 128), 128, 0, c->stream>>>(Cf, n0, (n1 + 2) * 3, inv0);
  c->launches += 4;
  return io.finish();
}

// FM2 + FM3 at n points; FM4 (the component index) is left to the caller: every row holds all three components.
int ts_field_map_eval_batch(ts_ctx* c, int64_t n0, int64_t n1, const double* coefs, int64_t n, const double* x0,
                            const double* x1, double* out, int pointers_are_device) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || !coefs || (n > 0 && (!x0 || !x1 || !out))) return fail(c, TS_ERR_ARG, "ts_field_map_eval_batch: null array or n<0");
  int rc;
  if ((rc = field_map_dims(c, "ts_field_map_eval_batch", n0, n1))) return rc;
  if (n == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  const int64_t nodes = (n0 + 2) * (n1 + 2);
  Staging io(c, pointers_are_device);
  const double *dc = io.in(coefs, (size_t)nodes * 3), *da = io.in(x0, (size_t)n), *db = io.in(x1, (size_t)n);
  double* dout = io.out(out, (size_t)n * 3);
  if (io.rc) return io.rc;
  void* c4;
  if ((rc = scratch_reserve(c, SLOT_TABLE, (size_t)nodes * 4 * sizeof(double), &c4))) return rc;
  TS_CUDA(c, cudaMemsetAsync(c->d_flag, 0, sizeof(int), c->stream));
  io.start();
  k8_pad4<<<(unsigned)((nodes + 255) / 256), 256, 0, c->stream>>>(dc, nodes, (double*)c4);
  k8_field_map_eval<<<(unsigned)((n + K8_THREADS - 1) / K8_THREADS), K8_THREADS, 0, c->stream>>>(
      (const double*)c4, n0, n1, n, da, db, dout, c->d_flag);
  c->launches += 2;
  return finish_domain_checked(c, io, "ts_field_map_eval_batch: non-finite index (the rows of those points are NaN)");
}

// ---------------------------------------------------------------------------- K2
static_assert(sizeof(ts_field_opts) == sizeof(ts_field_opts_dev), "field opts layout");

// K2b over `rows` table rows from row `lo` of n orbits: one launch per IGRF degree present (any13 / any10); `skip`
// (nullable) leaves out the orbits whose cutoff index is already set
static void k2b_launch(ts_ctx* c, bool any13, bool any10, int64_t n, int64_t rows, const ts_field_opts_dev* fo, const int64_t* offs,
                       const int64_t* lim, const double* pos, double* B, int64_t lo = 0, const int64_t* skip = nullptr) {
  const dim3 grid((unsigned)n, (unsigned)((rows + K2B_THREADS - 1) / K2B_THREADS));
  if (any13) {
    k2b_field_rows<13><<<grid, K2B_THREADS, 0, c->stream>>>(c->d_tabG, c->d_tabH, fo, offs, lim, pos, B, 13, lo, skip);
    c->launches++;
  }
  if (any10) {
    k2b_field_rows<10><<<grid, K2B_THREADS, 0, c->stream>>>(c->d_tabG, c->d_tabH, fo, offs, lim, pos, B, 10, lo, skip);
    c->launches++;
  }
}

int ts_magnetic_simulation_batch(ts_ctx* c, int64_t n_trials, const double* kep6, const ts_field_opts* opts,
                                 const int64_t* B_offs, const int64_t* rows_limit, double* B_eci, double* pos, double* vel,
                                 int pointers_are_device) {
  if (!c) return TS_ERR_ARG;
  if (n_trials < 0 || (n_trials > 0 && (!kep6 || !opts || !B_offs || !B_eci)))
    return fail(c, TS_ERR_ARG, "ts_magnetic_simulation_batch: null argument");
  if (n_trials == 0) return TS_OK;
  bool any13 = false, any10 = false;
  int64_t maxN = 0;
  for (int64_t t = 0; t < n_trials; ++t) {
    if (!igrf_date_ok(opts[t].igrf_date))
      return fail(c, TS_ERR_DATE, "trial %lld: IGRF date outside [1900, 2025]", (long long)t);
    if (opts[t].N < 1 || B_offs[t + 1] - B_offs[t] < 2 * opts[t].N)
      return fail(c, TS_ERR_ARG, "trial %lld: N < 1 or B_offs does not leave 2N rows", (long long)t);
    (igrf_nmax_for_date(opts[t].igrf_date) == 13 ? any13 : any10) = true;
    if (opts[t].N > maxN) maxN = opts[t].N;
  }
  TS_CUDA(c, cudaSetDevice(c->device));
  const int64_t total_rows = B_offs[n_trials];
  int rc;
  Staging io(c, pointers_are_device);
  const double* d_kep = io.in(kep6, (size_t)n_trials * 6);
  double* d_B = io.out(B_eci, (size_t)total_rows * 3);
  const size_t pos_count = (size_t)(total_rows + n_trials) * 3;
  double* d_pos = io.out(pos, pos_count);
  if (io.rc) return io.rc;
  if (!pos) {
    void* p = nullptr;
    if ((rc = scratch_reserve(c, SLOT_POSITIONS, pos_count * sizeof(double), &p))) return rc;
    d_pos = (double*)p;
  }
  double* d_vel = io.out(vel, pos_count);
  if (io.rc) return io.rc;
  ts_field_opts_dev* d_opts = nullptr;
  int64_t *d_offs = nullptr, *d_lim = nullptr;
  if ((rc = upload(c, SLOT_ARGS_A, (const ts_field_opts_dev*)opts, (size_t)n_trials, &d_opts))) return rc;
  if ((rc = upload(c, SLOT_ARGS_B, B_offs, (size_t)n_trials + 1, &d_offs))) return rc;
  if (rows_limit && (rc = upload(c, SLOT_ARGS_C, rows_limit, (size_t)n_trials, &d_lim))) return rc;
  io.start();
  k2a_orbit_euler<<<(unsigned)((n_trials + 127) / 128), 128, 0, c->stream>>>(n_trials, d_kep, d_opts, d_offs, d_lim, d_pos, d_vel);
  c->launches++;
  k2b_launch(c, any13, any10, n_trials, 2 * maxN, d_opts, d_offs, d_lim, d_pos, d_B);
  return io.finish();
}

static int gramian_common(ts_ctx* c, int64_t n_trials, const double* B_eci, const int64_t* B_offs, const int64_t* rows,
                          const double* dt, const double* cutoff, double* G, int64_t* tf_index, int pointers_are_device) {
  if (!c) return TS_ERR_ARG;
  if (n_trials < 0 || (n_trials > 0 && (!B_eci || !B_offs || !rows || !dt))) return fail(c, TS_ERR_ARG, "gramian: null argument");
  if (n_trials == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  int64_t total = 0;
  for (int64_t t = 0; t < n_trials; ++t) total = (B_offs[t] + rows[t] > total) ? B_offs[t] + rows[t] : total;
  int rc;
  Staging io(c, pointers_are_device);
  const double* d_B = io.in(B_eci, (size_t)total * 3);
  double* d_G = io.out(G, (size_t)total * 9);
  if (io.rc) return io.rc;
  int64_t *d_offs, *d_rows, *d_idx = nullptr;
  double *d_dt, *d_cut = nullptr;
  if ((rc = upload(c, SLOT_ARGS_A, B_offs, (size_t)n_trials, &d_offs))) return rc;
  if ((rc = upload(c, SLOT_ARGS_B, rows, (size_t)n_trials, &d_rows))) return rc;
  if ((rc = upload(c, SLOT_ARGS_C, dt, (size_t)n_trials, &d_dt))) return rc;
  if (cutoff && (rc = upload(c, SLOT_CUTOFF, cutoff, (size_t)n_trials, &d_cut))) return rc;
  if (tf_index) {
    void* p;
    if ((rc = scratch_reserve(c, SLOT_PER_TRIAL, (size_t)n_trials * sizeof(int64_t), &p))) return rc;
    d_idx = (int64_t*)p;
    io.back(tf_index, d_idx, (size_t)n_trials);
  }
  io.start();
  k2c_gramian_cutoff<<<(unsigned)((n_trials + 127) / 128), 128, 0, c->stream>>>(n_trials, d_B, d_offs, d_rows, d_dt, d_cut, d_G, d_idx);
  c->launches++;
  return io.finish();
}

int ts_magnetic_gramian_batch(ts_ctx* c, int64_t n_trials, const double* B_eci, const int64_t* B_offs, const int64_t* rows,
                              const double* dt, double* G, int pointers_are_device) {
  if (c && !G) return fail(c, TS_ERR_ARG, "ts_magnetic_gramian_batch: G is null");
  return gramian_common(c, n_trials, B_eci, B_offs, rows, dt, nullptr, G, nullptr, pointers_are_device);
}

int ts_condition_cutoff_batch(ts_ctx* c, int64_t n_trials, const double* B_eci, const int64_t* B_offs, const int64_t* rows,
                              const double* dt, const double* cutoff, int64_t* tf_index, int pointers_are_device) {
  if (c && (!cutoff || !tf_index)) return fail(c, TS_ERR_ARG, "ts_condition_cutoff_batch: null argument");
  return gramian_common(c, n_trials, B_eci, B_offs, rows, dt, cutoff, nullptr, tf_index, pointers_are_device);
}

int ts_condition_based_time_batch(ts_ctx* c, int64_t n_trials, const double* G, const int64_t* offs, const int64_t* rows,
                                  const double* cutoff, int64_t* tf_index, int pointers_are_device) {
  if (!c) return TS_ERR_ARG;
  if (n_trials < 0 || (n_trials > 0 && (!G || !offs || !rows || !cutoff || !tf_index)))
    return fail(c, TS_ERR_ARG, "ts_condition_based_time_batch: null argument");
  if (n_trials == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  int64_t total = 0;
  for (int64_t t = 0; t < n_trials; ++t) total = (offs[t] + rows[t] > total) ? offs[t] + rows[t] : total;
  int rc;
  Staging io(c, pointers_are_device);
  const double* d_G = io.in(G, (size_t)total * 9);
  if (io.rc) return io.rc;
  int64_t *d_offs, *d_rows, *d_idx;
  double* d_cut;
  if ((rc = upload(c, SLOT_ARGS_A, offs, (size_t)n_trials, &d_offs))) return rc;
  if ((rc = upload(c, SLOT_ARGS_B, rows, (size_t)n_trials, &d_rows))) return rc;
  if ((rc = upload(c, SLOT_CUTOFF, cutoff, (size_t)n_trials, &d_cut))) return rc;
  void* p;
  if ((rc = scratch_reserve(c, SLOT_PER_TRIAL, (size_t)n_trials * sizeof(int64_t), &p))) return rc;
  d_idx = (int64_t*)p;
  io.back(tf_index, d_idx, (size_t)n_trials);
  io.start();
  k2d_condition_time<<<(unsigned)((n_trials + 127) / 128), 128, 0, c->stream>>>(n_trials, d_G, d_offs, d_rows, d_cut, d_idx);
  c->launches++;
  return io.finish();
}

// ---------------------------------------------------------------------------- K3
static_assert(sizeof(ts_ilqr_opts) == sizeof(ts_ilqr_opts_dev), "ilqr opts layout");
static_assert(sizeof(ts_trial_outcome) == sizeof(ts_trial_outcome_dev) && sizeof(ts_trial_outcome) == 64, "outcome layout");

void ts_ilqr_default_opts(ts_ilqr_opts* o) {
  if (!o) return;
  o->max_outer = 20; o->max_inner = 50; o->max_linesearch = 20; o->dJ_counter_limit = 10;
  o->stage_cost_dt = 0; o->goal_mask = 0x7F;
  o->cost_tol = 1e-4; o->cost_tol_intermediate = 1e-3; o->grad_tol = 1e-5; o->grad_tol_intermediate = 1e-5;
  o->constraint_tol = 1e-3; o->penalty_initial = 1.0; o->penalty_scaling = 10.0; o->penalty_max = 1e8; o->dual_max = 1e8;
  o->ls_lower = 1e-8; o->ls_upper = 10.0; o->bp_reg_increase = 1.6; o->bp_reg_max = 1e8; o->bp_reg_min = 1e-8;
  o->bp_reg_fp = 10.0; o->max_cost_value = 1e8; o->max_state_value = 1e8; o->max_control_value = 1e8;
  o->u_max = 1.0; o->u_min = -1.0;
  o->a2_active_ge = 0; o->a3_grad_over_N = 0; o->a4_no_intermediate = 0; o->a5_dual_active_only = 0;
  o->a6_penalty_conditional = 0; o->a7_carry_cost = 0; o->constraint_decrease_ratio = 0.25;
  o->k3_suspend_after = 150; o->k3_tail_share = 1; o->k3_early_factor = 2.0; o->k3_pair = 2; o->k3_wide_occ = 0; o->quat_error = 0; o->k3_generic_inertia = 0;
}

// slew angle between the initial and the goal attitude (host): the difficulty proxy of the K3 queue order
static double slew_angle(const double* x0, const double* xf) {
  double n0 = 0, nf = 0, d = 0;
  for (int i = 3; i < 7; ++i) { n0 += x0[i] * x0[i]; nf += xf[i] * xf[i]; d += x0[i] * xf[i]; }
  const double c = fabs(d) / sqrt(n0 * nf + 1e-300);
  return 2.0 * acos(c > 1.0 ? 1.0 : c);
}

// Launch K3 on device-resident per-trial arrays (a.* device pointers except where noted): k3_alilqr_kernel (warps
// pull groups of 4 trials, one per 8-lane team) followed by k3_wide_kernel (stragglers handed over to one warp each).
// The launch scheme is controlled by ts_ilqr_opts.k3_* (suspend_after, early_factor, tail_share).  Work is queued on
// the context's stream; nothing here synchronises.
// true when every 3x3 inertia matrix of the (host) array is diagonal: K3 then runs the *_diag_kernel instantiations
static bool all_inertia_diagonal(const double* Jmat, int64_t n) {
  for (int64_t t = 0; t < n; ++t)
    for (int i = 0; i < 9; ++i)
      if (i % 4 != 0 && Jmat[9 * t + i] != 0.0) return false;
  return true;
}

// cont (continuation, ts_alilqr_solve_state_batch with a state): the trials to continue.  They skip the first launch:
// park_import_kernel parks them, and the one-warp-per-trial launch finishes them.
static int k3_launch(ts_ctx* c, K3Args& a, const int64_t* N_i_host, const double* difficulty_host = nullptr, bool diag_inertia = false,
                     const std::vector<int64_t>* cont = nullptr, K3StateIO* sio = nullptr) {
  const int64_t n_trials = a.n_trials;
  // the quaternion-aware variant (opts.quat_error) runs the same two-launch scheme on the QUAT instantiations
  const bool quat = a.opts.quat_error != 0;
  if (quat) {
    const int qm = (a.opts.goal_mask >> 3) & 0xF;
    if (qm != 0 && qm != 0xF)
      return fail(c, TS_ERR_ARG, "quat_error: the goal mask must hold all four quaternion components or none");
  }
  // diagonal inertia matrices (every preset of the reference): instantiations without the products by their zeros
  const bool dj = diag_inertia && !a.opts.k3_generic_inertia;
  // a solve that exports its state runs the exporting instantiations (same results, K3StateIO written at the finish)
  void (*const narrow_kernel)(const K3Args) =
      a.sio ? (quat ? (dj ? k3_alilqr_quat_diag_export_kernel : k3_alilqr_quat_export_kernel)
                    : (dj ? k3_alilqr_diag_export_kernel : k3_alilqr_export_kernel))
            : (quat ? (dj ? k3_alilqr_quat_diag_kernel : k3_alilqr_quat_kernel) : (dj ? k3_alilqr_diag_kernel : k3_alilqr_kernel));
  void (*const wide_kernel)(const K3Args) = quat ? (dj ? k3_wide_quat_diag_kernel : k3_wide_quat_kernel)
                                                 : (dj ? k3_wide_diag_kernel : k3_wide_kernel);
  void (*const pair_kernel)(const K3Args) = dj ? k3_pair_diag_kernel : k3_pair_kernel;
  int64_t Nmax = 0;
  for (int64_t t = 0; t < n_trials; ++t) Nmax = std::max(Nmax, N_i_host[t]);
  int occ = 0;
  TS_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, narrow_kernel, K3_WARPS_PER_BLOCK * 32, K3_SMEM_BYTES));
  if (occ < 1) return fail(c, TS_ERR_CUDA, "k3 kernel does not fit on an SM");
  const int64_t groups = (n_trials + 3) / 4;
  const int64_t max_warps = (int64_t)c->sm_count * occ * K3_WARPS_PER_BLOCK;
  const int64_t warps = std::min(groups, max_warps);
  const int blocks = (int)((warps + K3_WARPS_PER_BLOCK - 1) / K3_WARPS_PER_BLOCK);
  const int64_t slots = (int64_t)blocks * K3_WARPS_PER_BLOCK * 4;
  // the one-warp-per-trial launch uses four slots (36 trajectory buffers) per warp: up to a full wave of warps,
  // never more than there can be parked trials
  int occ_w = 0;
  TS_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_w, wide_kernel, 32, K3_WIDE_SMEM_BYTES));
  if (occ_w < 1) return fail(c, TS_ERR_CUDA, "k3 wide kernel does not fit on an SM");
  int64_t wide_warps = std::min<int64_t>(n_trials, (int64_t)c->sm_count * occ_w);
  // second launch with a producer warp per solver warp (k3_pair_kernel): 1 = always, 0 = never, 2 = when the horizons are
  // ragged (longest >= 2 x mean).  Measured: on the fixed-orbit ensemble (all horizons equal, 2243 stragglers on 1184
  // warps) halving the solver warps costs more than the hidden linearisation gains (6.32 s vs 5.72 s); on the sweep the
  // second launch is the sequential chain of a few very long slews and the producer shortens exactly that chain
  // (13.4 s vs 16.2 s).  (The producer-warp kernel exists for the default solver only.)
  double N_mean = 0.0;
  for (int64_t t = 0; t < n_trials; ++t) N_mean += (double)N_i_host[t];
  N_mean /= (double)std::max<int64_t>(n_trials, 1);
  const bool pair = !quat && (a.opts.k3_pair == 1 || (a.opts.k3_pair == 2 && (double)Nmax >= 2.0 * N_mean));
  int wide_smem = K3_WIDE_SMEM_BYTES;
  if (pair) {
    int occ_p = 0;
    TS_CUDA(c, cudaFuncSetAttribute(pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, K3_PAIR_SMEM_BYTES));
    TS_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_p, pair_kernel, 64 * K3_PAIRS_PER_BLOCK, K3_PAIR_SMEM_BYTES));
    if (occ_p < 1) return fail(c, TS_ERR_CUDA, "k3 pair kernel does not fit on an SM");
    wide_warps = std::min<int64_t>(n_trials, (int64_t)c->sm_count * occ_p * K3_PAIRS_PER_BLOCK);   // solver warps
  } else if (a.opts.k3_wide_occ > 0 && a.opts.k3_wide_occ < occ_w) {
    // fewer blocks per SM: pad the dynamic shared memory so that exactly k3_wide_occ one-warp blocks fit
    wide_smem = std::max(K3_WIDE_SMEM_BYTES, (227 * 1024 / (a.opts.k3_wide_occ + 1) + 1024) & ~15);
    TS_CUDA(c, cudaFuncSetAttribute(wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, wide_smem));
    int occ2 = 0;
    TS_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, wide_kernel, 32, wide_smem));
    wide_warps = std::min<int64_t>(n_trials, (int64_t)c->sm_count * std::max(occ2, 1));
  }
  // Queue order.  (1) sort by horizon (descending): the four teams of a warp get similar trip counts.
  // (2) within a run of (nearly) equal horizons, sort by slew angle and DEAL the trials round-robin over the
  // groups of four, so each warp gets one trial of every difficulty quartile: the makespan of a single-wave
  // ensemble is set by the warp with the most stragglers (non-converging large-angle slews), and dealing
  // them out makes triple clusters (which cannot lend each other lanes) vanishingly rare.
  std::vector<int64_t> order((size_t)n_trials);
  std::iota(order.begin(), order.end(), (int64_t)0);
  std::stable_sort(order.begin(), order.end(), [&](int64_t x, int64_t y) { return N_i_host[x] > N_i_host[y]; });
  const std::vector<int64_t> order_by_N = order;
  if (difficulty_host && n_trials >= 8) {
    size_t lo = 0;
    while (lo < (size_t)n_trials) {
      size_t hi = lo;
      while (hi < (size_t)n_trials && (double)N_i_host[order[hi]] >= 0.97 * (double)N_i_host[order[lo]]) ++hi;
      const size_t len = hi - lo;
      if (len >= 8) {
        std::vector<int64_t> run(order.begin() + lo, order.begin() + hi);
        std::stable_sort(run.begin(), run.end(), [&](int64_t x, int64_t y) { return difficulty_host[x] > difficulty_host[y]; });
        const size_t G = (len + 3) / 4;
        size_t pos = lo;
        for (size_t g = 0; g < G; ++g)
          for (size_t j = 0; j < 4; ++j)
            if (g + j * G < len) order[pos++] = run[g + j * G];
      }
      lo = hi;
    }
  }
  int rc;
  int64_t* d_order = nullptr;
  if ((rc = upload(c, SLOT_PER_TRIAL, order.data(), (size_t)n_trials, &d_order))) return rc;
  void *p_work, *p_q, *p_diag;
  Nmax += (Nmax & 1);  // even: keeps every per-knot record 16-byte aligned for the asynchronous copies
  // ragged arena: warp w's four slots are sized for its static first group (the w-th of the horizon-sorted queue; the
  // dealing above permutes only inside runs of nearly equal horizons, so the group's maximum is taken explicitly)
  const int64_t n_warps = (int64_t)blocks * K3_WARPS_PER_BLOCK;
  std::vector<long long> warp_off((size_t)n_warps);
  std::vector<int> warp_cap((size_t)n_warps);
  long long arena = 0;
  {
    int64_t later_max = 0;   // longest horizon among the trials pulled dynamically (queue positions >= 4 * n_warps)
    for (int64_t q = 4 * n_warps; q < n_trials; ++q) later_max = std::max(later_max, N_i_host[order[(size_t)q]]);
    for (int64_t w = 0; w < n_warps; ++w) {
      int64_t cap = later_max;
      for (int64_t q = 4 * w; q < std::min<int64_t>(4 * w + 4, n_trials); ++q) cap = std::max(cap, N_i_host[order[(size_t)q]]);
      cap = std::max<int64_t>(cap, 2);
      cap += (cap & 1);
      warp_off[(size_t)w] = arena;
      warp_cap[(size_t)w] = (int)cap;
      arena += 4 * cap * K3_SLOT_DOUBLES_PER_KNOT;
    }
  }
  long long* d_woff = nullptr;
  int* d_wcap = nullptr;
  p_work = nullptr;
  if (!cont) {   // a continuation does not run the first launch
    if ((rc = scratch_reserve(c, SLOT_K3_ARENA, (size_t)(arena + 2) * sizeof(double) + 256, &p_work))) return rc;
    if ((rc = upload(c, SLOT_K3_WARP_OFFS, warp_off.data(), (size_t)n_warps, &d_woff))) return rc;
    if ((rc = upload(c, SLOT_K3_WARP_CAPS, warp_cap.data(), (size_t)n_warps, &d_wcap))) return rc;
  }
  if ((rc = scratch_reserve(c, SLOT_K3_COUNTERS, 128, &p_q))) return rc;
  if ((rc = scratch_reserve(c, SLOT_K3_CYCLES, (size_t)n_trials * 3 * sizeof(double) + 64, &p_diag))) return rc;
  {
    unsigned long long h_q[16] = {0};
    h_q[0] = (unsigned long long)(4 * n_warps);   // the dynamic queue starts behind the static first groups
    TS_CUDA(c, cudaMemcpyAsync(p_q, h_q, 128, cudaMemcpyHostToDevice, c->stream));
  }
  TS_CUDA(c, cudaMemsetAsync(p_diag, 0, (size_t)n_trials * 3 * sizeof(double), c->stream));
  a.order = d_order;
  a.Nmax = Nmax;
  a.w_base = (double*)p_work;
  a.warp_off = d_woff;
  a.warp_cap = d_wcap;
  a.n_warps = n_warps;
  a.pool = nullptr;
  a.pool_used = (unsigned long long*)p_q + 10;
  a.pool_cap = 0;
  a.queue = (unsigned long long*)p_q;
  a.diag = (double*)p_diag;
  c->k3_diag_n = n_trials;
  a.tail_share = a.opts.k3_tail_share ? 1 : 0;
  // straggler hand-over (k3_wide_kernel): allowance of the 4-trials-per-warp kernel, in inner iterations of a
  // trial of MEAN horizon; trials are charged in knot-iterations, so a long-horizon trial is handed over sooner
  const int suspend_after = std::max(0, (int)a.opts.k3_suspend_after);
  double N_sum = 0.0;
  for (int64_t t = 0; t < n_trials; ++t) N_sum += (double)N_i_host[t];
  a.park_budget = (long long)((double)suspend_after * N_sum / (double)n_trials);
  if (suspend_after > 0 && a.park_budget < 1) a.park_budget = 1;
  // multi-wave ensembles: a trial that has used early_factor x the allowance is parked even while fresh trials are
  // still queued, so that it stops holding its warp's group back (0 = only once the queue has drained)
  const double early = a.opts.k3_early_factor;
  a.park_budget_early = early > 0.0 ? (long long)(early * (double)a.park_budget) : (long long)4e18;
  a.park_cap = 0;
  a.park_count = (unsigned*)p_q + 8;
  a.park_used = (unsigned long long*)p_q + 5;
  a.queue2 = (unsigned long long*)p_q + 2;
  a.park_state = nullptr;
  a.park_trial = nullptr;
  a.park_off = nullptr;
  a.park_data = nullptr;
  a.park_data_cap = 0;
  a.park_order = nullptr;
  if (cont || suspend_after > 0) {
    // a place for every trial that can be resident when the queue runs dry; array space for the `cap` longest
    // horizons (order[] is sorted by horizon, descending), bounded by 32 GB.  A continuation parks every trial it
    // continues, or fails.
    std::vector<int64_t> cand = cont ? *cont : order_by_N;
    if (cont) std::stable_sort(cand.begin(), cand.end(), [&](int64_t x, int64_t y) { return N_i_host[x] > N_i_host[y]; });
    int64_t cap = cont ? (int64_t)cont->size() : (early > 0.0 ? n_trials : std::min<int64_t>(n_trials, slots));
    // memory of the hand-over: 27 N doubles of parked state per trial + a 261 N region per trial in the worst case
    // (no region is ever re-used); the parking places are limited to what fits 60% of the free device memory
    size_t free_b = 0, total_b = 0;
    TS_CUDA(c, cudaMemGetInfo(&free_b, &total_b));
    const double budget = 0.6 * (double)(free_b + c->scratch_bytes[SLOT_PARK_DATA] + c->scratch_bytes[SLOT_K3_POOL]) / 8.0;
    double need = 0.0, pool_need = 0.0;
    int64_t cap_fit = 0;
    for (int64_t i = 0; i < cap; ++i) {
      const double Ne = (double)(N_i_host[cand[(size_t)i]] + 1);
      const double dpk = (double)k3_wide_doubles_per_knot(a.opts.max_linesearch);
      if (need + pool_need + (27.0 + dpk) * Ne > budget) break;
      need += 27.0 * Ne;
      pool_need += dpk * Ne;
      cap_fit = i + 1;
    }
    if (cont && cap_fit < cap)
      return fail(c, TS_ERR_NOMEM, "continuation: the parked records of %lld trials do not fit in device memory (%lld do)",
                  (long long)cap, (long long)cap_fit);
    cap = cap_fit;
    void *p_ps, *p_pd, *p_pool;
    if ((rc = scratch_reserve(c, SLOT_K3_POOL, (size_t)pool_need * sizeof(double) + 256, &p_pool))) return rc;
    a.pool = (double*)p_pool;
    a.pool_cap = (long long)pool_need;
    if ((rc = scratch_reserve(c, SLOT_PARK_STATE, (size_t)cap * (sizeof(TrialState) + 8 + 8 + 4) + 64, &p_ps))) return rc;
    if ((rc = scratch_reserve(c, SLOT_PARK_DATA, (size_t)need * sizeof(double) + 64, &p_pd))) return rc;
    a.park_cap = (int)cap;
    a.park_state = (TrialState*)p_ps;
    a.park_trial = (int64_t*)((char*)p_ps + (size_t)cap * sizeof(TrialState));
    a.park_off = (long long*)((char*)p_ps + (size_t)cap * (sizeof(TrialState) + 8));
    a.park_order = (int*)((char*)p_ps + (size_t)cap * (sizeof(TrialState) + 16));
    a.park_data = (double*)p_pd;
    a.park_data_cap = (long long)need;
    if (cont && cap > 0) {   // place i = the i-th continuing trial, its record at the host-computed offset
      std::vector<long long> off((size_t)cap);
      unsigned long long used = 0;
      for (int64_t i = 0; i < cap; ++i) {
        const long long N = N_i_host[(*cont)[(size_t)i]];
        off[(size_t)i] = (long long)used;
        used += (unsigned long long)(27 * (N + (N & 1)));
      }
      const unsigned long long h_cnt[2] = {(unsigned long long)cap, used};   // park_count (low word of [4]) | park_used [5]
      TS_CUDA(c, cudaMemcpyAsync(a.park_trial, cont->data(), (size_t)cap * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
      TS_CUDA(c, cudaMemcpyAsync(a.park_off, off.data(), (size_t)cap * sizeof(long long), cudaMemcpyHostToDevice, c->stream));
      TS_CUDA(c, cudaMemcpyAsync((unsigned long long*)p_q + 4, h_cnt, sizeof(h_cnt), cudaMemcpyHostToDevice, c->stream));
      sio->n_import = cap;
    }
  }
  if (sio) {
    TS_CUDA(c, cudaMemcpyAsync((void*)a.sio, sio, sizeof(K3StateIO), cudaMemcpyHostToDevice, c->stream));
    // CS2: every trial's multipliers pass to the output (the continuing trials' rows are then overwritten); queued only
    // now, so that a call that fails above leaves lam_out as it was.  A continuation in place (ts_mc_continue) passes
    // lam_in == lam_out: there is nothing to copy, and an overlapping cudaMemcpyAsync is undefined.
    if (sio->lam_in && sio->lam_in != sio->lam_out)
      TS_CUDA(c, cudaMemcpyAsync(sio->lam_out, sio->lam_in, (size_t)sio->lam_doubles * sizeof(double), cudaMemcpyDeviceToDevice,
                                 c->stream));
  }
  c->k3_timed = true;
  c->d_k3_parked = a.park_count;
  c->k3_park_cap = a.park_cap;
  TS_CUDA(c, cudaEventRecord(c->ev_k3[0], c->stream));
  if (!cont) {
    narrow_kernel<<<blocks, K3_WARPS_PER_BLOCK * 32, K3_SMEM_BYTES, c->stream>>>(a);
    c->launches++;
  }
  TS_CUDA(c, cudaGetLastError());
  TS_CUDA(c, cudaEventRecord(c->ev_k3[1], c->stream));
  TS_CUDA(c, cudaEventRecord(c->ev_k3[2], c->stream));
  if (a.park_cap > 0) {
    // one warp per parked trial; the grid cannot depend on the (device-side) count, idle blocks exit at once
    const int blocks_w = (int)std::max<int64_t>(1, std::min<int64_t>(a.park_cap, wide_warps));
    if (cont) {
      park_import_kernel<<<(unsigned)((sio->n_import + 3) / 4), 32, K3_SMEM_BYTES, c->stream>>>(a);
      c->launches++;
    }
    k3_park_order_kernel<<<1, 1024, 0, c->stream>>>(a);
    if (pair)
      pair_kernel<<<(blocks_w + K3_PAIRS_PER_BLOCK - 1) / K3_PAIRS_PER_BLOCK, 64 * K3_PAIRS_PER_BLOCK, K3_PAIR_SMEM_BYTES, c->stream>>>(a);
    else
      wide_kernel<<<blocks_w, 32, wide_smem, c->stream>>>(a);
    c->launches += 2;
    TS_CUDA(c, cudaGetLastError());
    TS_CUDA(c, cudaEventRecord(c->ev_k3[2], c->stream));
  }
  return TS_OK;
}

static_assert(sizeof(ts_al_state) == 104 && sizeof(ts_al_state) == sizeof(ts_al_state_dev), "ts_al_state layout");

// The option checks of an AL-iLQR solve of n trials with the state weights Qd, Qfd (8 per trial)
static int check_ilqr_opts(ts_ctx* c, const ts_ilqr_opts& o, int64_t n, const double* Qd, const double* Qfd) {
  if (o.max_linesearch < 0 || o.max_linesearch > 63) return fail(c, TS_ERR_ARG, "max_linesearch must be in [0,63]");
  if (o.quat_error)
    for (int64_t t = 0; t < n; ++t)
      for (int i = 4; i < 7; ++i)
        if (Qd[t * 8 + i] != Qd[t * 8 + 3] || Qfd[t * 8 + i] != Qfd[t * 8 + 3])
          return fail(c, TS_ERR_ARG, "quat_error: the four quaternion weights of Q and Qf must be equal (E'QE is then diagonal)");
  return TS_OK;
}

int ts_alilqr_solve_batch(ts_ctx* c, int64_t n_trials, const int64_t* N_i, const int64_t* offs, const double* x0,
                          const double* xf, const double* Jmat, const double* Qd, const double* Qfd, const double* Rd,
                          const double* B_eci, const int64_t* B_offs, const int64_t* B_rows, const double* index_scale,
                          const double* clock_rate, double dt, const double* U0, const ts_ilqr_opts* opts, double* X,
                          double* U, double* K, ts_trial_outcome* out, int pointers_are_device) {
  return ts_alilqr_solve_state_batch(c, n_trials, N_i, offs, x0, xf, Jmat, Qd, Qfd, Rd, B_eci, B_offs, B_rows, index_scale,
                                     clock_rate, dt, U0, opts, X, U, K, out, pointers_are_device, nullptr, nullptr, nullptr, nullptr);
}

int ts_alilqr_solve_state_batch(ts_ctx* c, int64_t n_trials, const int64_t* N_i, const int64_t* offs, const double* x0,
                                const double* xf, const double* Jmat, const double* Qd, const double* Qfd, const double* Rd,
                                const double* B_eci, const int64_t* B_offs, const int64_t* B_rows, const double* index_scale,
                                const double* clock_rate, double dt, const double* U0, const ts_ilqr_opts* opts, double* X,
                                double* U, double* K, ts_trial_outcome* out, int pointers_are_device,
                                const ts_al_state* state_in, const double* lam_in, ts_al_state* state_out, double* lam_out) {
  if (!c) return TS_ERR_ARG;
  if (n_trials < 0 || (n_trials > 0 && (!N_i || !offs || !x0 || !xf || !Jmat || !Qd || !Qfd || !Rd || !B_eci || !B_offs || !B_rows ||
                                        !index_scale || !clock_rate || !X || !U || !out)))
    return fail(c, TS_ERR_ARG, "ts_alilqr_solve_batch: null argument");
  if (state_in && !lam_in) return fail(c, TS_ERR_ARG, "ts_alilqr_solve_state_batch: state_in without lam_in");
  if (state_in)
    for (int64_t t = 0; t < n_trials; ++t)
      if (state_in[t].status < TS_ST_CONVERGED || state_in[t].status > TS_ST_NO_CUTOFF || state_in[t].outer_iters < 1)
        return fail(c, TS_ERR_ARG, "ts_alilqr_solve_state_batch: trial %lld: status %d / outer_iters %d is not an exported state",
                    (long long)t, (int)state_in[t].status, (int)state_in[t].outer_iters);
  if (n_trials == 0) return TS_OK;
  if (!(dt > 0)) return fail(c, TS_ERR_ARG, "ts_alilqr_solve_batch: dt must be > 0");
  ts_ilqr_opts o;
  if (opts) o = *opts; else ts_ilqr_default_opts(&o);
  int rc;
  if ((rc = check_ilqr_opts(c, o, n_trials, Qd, Qfd))) return rc;
  int64_t total_knots = 0, total_rows = 0;
  for (int64_t t = 0; t < n_trials; ++t) {
    if (N_i[t] < 2) return fail(c, TS_ERR_ARG, "trial %lld: N < 2", (long long)t);
    total_knots = std::max(total_knots, offs[t] + N_i[t]);
    total_rows = std::max(total_rows, B_offs[t] + B_rows[t]);
    if (B_rows[t] < 1) return fail(c, TS_ERR_ARG, "trial %lld: empty field table", (long long)t);
  }
  TS_CUDA(c, cudaSetDevice(c->device));
  Staging io(c, pointers_are_device);
  K3Args a = {};
  a.B_eci = io.in(B_eci, (size_t)total_rows * 3);
  a.U0 = io.in(U0, (size_t)total_knots * 3);
  if (state_in) {   // CS2: the rows of the trials that pass through stay as given
    a.X = io.inout(X, (size_t)total_knots * 8);
    a.U = io.inout(U, (size_t)total_knots * 3);
    a.K = io.inout(K, (size_t)total_knots * 24);
    lam_in = io.in(lam_in, (size_t)total_knots * 6);
  } else {
    a.X = io.out(X, (size_t)total_knots * 8);
    a.U = io.out(U, (size_t)total_knots * 3);
    a.K = io.out(K, (size_t)total_knots * 24);
  }
  double* d_lam_out = io.out(lam_out, (size_t)total_knots * 6);
  if (io.rc) return io.rc;
  // per-trial small arrays -> one packed upload
  const size_t T = (size_t)n_trials;
  const size_t n_i64 = 4 * T, n_f64 = (8 + 8 + 9 + 8 + 8 + 3 + 1 + 1) * T;
  std::vector<int64_t> hi(n_i64);
  std::vector<double> hf(n_f64);
  memcpy(&hi[0 * T], N_i, T * 8);
  memcpy(&hi[1 * T], offs, T * 8);
  memcpy(&hi[2 * T], B_offs, T * 8);
  memcpy(&hi[3 * T], B_rows, T * 8);
  size_t fo = 0;
  auto put = [&](const double* src, size_t per) { memcpy(&hf[fo], src, per * T * 8); fo += per * T; return fo - per * T; };
  const size_t o_x0 = put(x0, 8), o_xf = put(xf, 8), o_J = put(Jmat, 9), o_Qd = put(Qd, 8), o_Qfd = put(Qfd, 8), o_Rd = put(Rd, 3),
               o_is = put(index_scale, 1), o_cr = put(clock_rate, 1);
  int64_t* d_i = nullptr;
  double* d_f = nullptr;
  if ((rc = upload(c, SLOT_ARGS_A, hi.data(), n_i64, &d_i))) return rc;
  if ((rc = upload(c, SLOT_ARGS_B, hf.data(), n_f64, &d_f))) return rc;
  void* p_out;
  if ((rc = scratch_reserve(c, SLOT_ARGS_C, T * sizeof(ts_trial_outcome), &p_out))) return rc;
  a.n_trials = n_trials;
  a.N_i = d_i + 0 * T; a.offs = d_i + 1 * T; a.B_offs = d_i + 2 * T; a.B_rows = d_i + 3 * T;
  a.x0 = d_f + o_x0; a.xf = d_f + o_xf; a.Jmat = d_f + o_J; a.Qd = d_f + o_Qd; a.Qfd = d_f + o_Qfd; a.Rd = d_f + o_Rd;
  a.index_scale = d_f + o_is; a.clock_rate = d_f + o_cr;
  a.dt = dt;
  memcpy(&a.opts, &o, sizeof(o));
  a.out = (ts_trial_outcome_dev*)p_out;
  io.back(out, (const ts_trial_outcome*)p_out, T);
  std::vector<int64_t> cont;
  K3StateIO sio = {};
  if (state_out || lam_out || state_in) {
    // device block: states [0, T) imported, [T, 2T) exported | K3StateIO | the multipliers when the caller takes none
    void* p_st;
    const size_t b_st = 2 * T * sizeof(ts_al_state), b_lam = lam_out ? 0 : (size_t)total_knots * 6 * sizeof(double);
    if ((rc = scratch_reserve(c, SLOT_AL_STATES, b_st + 64 + b_lam, &p_st))) return rc;
    ts_al_state_dev* d_in = (ts_al_state_dev*)p_st;
    sio.state_out = d_in + T;
    sio.lam_out = lam_out ? d_lam_out : (double*)((char*)p_st + b_st + 64);
    a.sio = (const K3StateIO*)((char*)p_st + b_st);
    if (state_out) io.back(state_out, (const ts_al_state*)sio.state_out, T);
    if (state_in) {
      // CS2: which trials continue; every other trial's outcome is rebuilt from its state, and its state and multipliers
      // are copied to the outputs (the kernels then overwrite the continuing trials' records)
      std::vector<ts_trial_outcome> oc(T);
      for (size_t t = 0; t < T; ++t) {
        const ts_al_state& st = state_in[t];
        if (st.status == TS_ST_MAX_OUTER && st.outer_iters < o.max_outer) cont.push_back((int64_t)t);
        oc[t] = ts_trial_outcome{st.status, st.outer_iters, st.inner_iters, st.ls_rollouts, N_i[t], st.J, st.c_max, 0.0, 0.0, 0.0};
      }
      TS_CUDA(c, cudaMemcpyAsync(d_in, state_in, T * sizeof(ts_al_state), cudaMemcpyHostToDevice, c->stream));
      TS_CUDA(c, cudaMemcpyAsync(p_out, oc.data(), T * sizeof(ts_trial_outcome), cudaMemcpyHostToDevice, c->stream));
      TS_CUDA(c, cudaMemcpyAsync(sio.state_out, d_in, T * sizeof(ts_al_state), cudaMemcpyDeviceToDevice, c->stream));
      sio.state_in = d_in;
      sio.lam_in = lam_in;
      sio.lam_doubles = total_knots * 6;   // copied to lam_out by k3_launch once the park records are known to fit
    }
  }
  std::vector<double> diff(T);
  for (size_t t = 0; t < T; ++t) diff[t] = slew_angle(x0 + 8 * t, xf + 8 * t);
  io.start();
  if ((rc = k3_launch(c, a, N_i, diff.data(), all_inertia_diagonal(Jmat, n_trials), state_in ? &cont : nullptr, a.sio ? &sio : nullptr)))
    return rc;
  return io.finish();
}

// ---------------------------------------------------------------------------- prep + K4
static_assert(sizeof(ts_tvlqr_opts) == sizeof(ts_tvlqr_opts_dev), "tvlqr opts layout");

// K4's linearisation table: lin_offs (the prefix sum of the n trials' N_i - 1 steps, uploaded) and the records AB
// (54 doubles per step) + clk (one per step)
static int k4_lin_table(ts_ctx* c, const int64_t* N_i, size_t n, K4Args& a) {
  std::vector<int64_t> lin(n + 1, 0);
  for (size_t t = 0; t < n; ++t) lin[t + 1] = lin[t] + (N_i[t] - 1);
  int64_t* d_lin;
  void* p_ab;
  int rc;
  if ((rc = upload(c, SLOT_TABLE, lin.data(), n + 1, &d_lin))) return rc;
  if ((rc = scratch_reserve(c, SLOT_LIN_RECORDS, (size_t)lin[n] * 55 * 8 + 64, &p_ab))) return rc;
  a.AB = (double*)p_ab; a.clk = a.AB + (size_t)lin[n] * 54; a.lin_offs = d_lin; a.lin_total = lin[n];
  return TS_OK;
}

void ts_tvlqr_default_opts(ts_tvlqr_opts* o) {
  if (!o) return;
  memset(o, 0, sizeof(*o));
  o->dt = 0.2; o->t0 = 0.0; o->tf = 0.0;
  for (int i = 0; i < 6; ++i) { o->Qd[i] = 10.0; o->Qfd[i] = 1000.0; }
  for (int i = 0; i < 3; ++i) o->Rd[i] = 7.5e3;
  o->dt_squared = 1; o->noise_mode = 0; o->seed = 0;
  o->w_limit = 0.05; o->ang_limit = 0.08727; o->literal_postproc = 0;
}

int ts_slew_weights_batch(ts_ctx* c, int64_t n, const double* x0, const double* xf, const double* Jmat, const double* t_final,
                          double t0, double dt, double alpha, double beta, int eigen_axis_fix, double* Qd, double* Qfd, double* Rd,
                          const int64_t* goffs, double* w_guess, double* q_guess) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || (n > 0 && (!x0 || !xf || !Jmat || !t_final || !Qd || !Qfd || !Rd))) return fail(c, TS_ERR_ARG, "ts_slew_weights_batch: null argument");
  if ((w_guess || q_guess) && !goffs) return fail(c, TS_ERR_ARG, "ts_slew_weights_batch: guesses need goffs");
  if (n == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  const size_t T = (size_t)n;
  int64_t total = 0;
  if (goffs)
    for (int64_t t = 0; t < n; ++t) total = std::max(total, goffs[t] + (int64_t)range_len(t0, dt, t_final[t]));
  std::vector<double> hf((8 + 8 + 9 + 1) * T);
  memcpy(&hf[0], x0, 8 * T * 8);
  memcpy(&hf[8 * T], xf, 8 * T * 8);
  memcpy(&hf[16 * T], Jmat, 9 * T * 8);
  memcpy(&hf[25 * T], t_final, T * 8);
  double* d_f;
  int64_t* d_g = nullptr;
  int rc;
  if ((rc = upload(c, SLOT_ARGS_A, hf.data(), hf.size(), &d_f))) return rc;
  if (goffs && (rc = upload(c, SLOT_ARGS_B, goffs, T, &d_g))) return rc;
  void *p_o, *p_w = nullptr, *p_q = nullptr;
  if ((rc = scratch_reserve(c, SLOT_ARGS_C, 19 * T * 8, &p_o))) return rc;
  if (w_guess && (rc = scratch_reserve(c, SLOT_ROWS_A, (size_t)total * 3 * 8, &p_w))) return rc;
  if (q_guess && (rc = scratch_reserve(c, SLOT_ROWS_B, (size_t)total * 4 * 8, &p_q))) return rc;
  PrepArgs a;
  a.n_trials = n; a.x0 = d_f; a.xf = d_f + 8 * T; a.Jmat = d_f + 16 * T; a.t_final = d_f + 25 * T;
  a.t0 = t0; a.dt = dt; a.alpha = alpha; a.beta = beta; a.conj_fix = eigen_axis_fix ? 1 : 0;
  a.Qd = (double*)p_o; a.Qfd = a.Qd + 8 * T; a.Rd = a.Qd + 16 * T;
  a.goffs = d_g; a.w_guess = (double*)p_w; a.q_guess = (double*)p_q;
  Staging io(c, 0);
  io.back(Qd, a.Qd, 8 * T);
  io.back(Qfd, a.Qfd, 8 * T);
  io.back(Rd, a.Rd, 3 * T);
  if (w_guess) io.back(w_guess, a.w_guess, (size_t)total * 3);
  if (q_guess) io.back(q_guess, a.q_guess, (size_t)total * 4);
  io.start();
  k_slew_prep<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(a);
  c->launches++;
  return io.finish();
}

int ts_tvlqr_sim_batch(ts_ctx* c, int64_t n, const int64_t* N_i, const int64_t* offs, const double* X_lqr, const double* U_lqr,
                       const double* x0_lqr, const double* Jmat, const double* B_eci, const int64_t* B_offs, const int64_t* B_rows,
                       const double* index_scale, const double* clock_rate, const double* t_final, const double* q_final,
                       const uint32_t* stream_id, const ts_tvlqr_opts* opts, const double* noise, double* X_sim, double* U_sim,
                       double* dX, double* K, int64_t* N_sim, double* slew_time, int pointers_are_device) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || (n > 0 && (!N_i || !offs || !X_lqr || !U_lqr || !x0_lqr || !Jmat || !B_eci || !B_offs || !B_rows || !index_scale ||
                          !clock_rate || !t_final || !q_final)))
    return fail(c, TS_ERR_ARG, "ts_tvlqr_sim_batch: null argument");
  if (n == 0) return TS_OK;
  ts_tvlqr_opts o;
  if (opts) o = *opts; else ts_tvlqr_default_opts(&o);
  if (o.noise_mode == 1 && !noise) return fail(c, TS_ERR_ARG, "ts_tvlqr_sim_batch: noise_mode 1 needs a noise array");
  if (o.literal_postproc && !X_sim) return fail(c, TS_ERR_ARG, "ts_tvlqr_sim_batch: literal_postproc needs X_sim");
  TS_CUDA(c, cudaSetDevice(c->device));
  const size_t T = (size_t)n;
  int64_t knots = 0, rows = 0;
  for (int64_t t = 0; t < n; ++t) {
    if (N_i[t] < 2) return fail(c, TS_ERR_ARG, "trial %lld: N < 2", (long long)t);
    knots = std::max(knots, offs[t] + N_i[t]);
    rows = std::max(rows, B_offs[t] + B_rows[t]);
  }
  int rc;
  Staging io(c, pointers_are_device);
  K4Args a;
  a.X_lqr = io.in(X_lqr, (size_t)knots * 8);
  a.U_lqr = io.in(U_lqr, (size_t)knots * 3);
  a.B_eci = io.in(B_eci, (size_t)rows * 3);
  a.noise = io.in(o.noise_mode == 1 ? noise : nullptr, (size_t)knots * 36);
  a.X_sim = io.out(X_sim, (size_t)knots * 8);
  a.U_sim = io.out(U_sim, (size_t)knots * 3);
  a.dX = io.out(dX, (size_t)knots * 6);
  a.K = io.out(K, (size_t)knots * 18);
  if (io.rc) return io.rc;
  if (!K) {
    void* p;
    if ((rc = scratch_reserve(c, SLOT_K4_GAINS, (size_t)knots * 18 * 8, &p))) return rc;
    a.K = (double*)p;
  }
  std::vector<int64_t> hi(4 * T);
  memcpy(&hi[0], N_i, T * 8); memcpy(&hi[T], offs, T * 8); memcpy(&hi[2 * T], B_offs, T * 8); memcpy(&hi[3 * T], B_rows, T * 8);
  std::vector<double> hf((8 + 9 + 1 + 1 + 1 + 4) * T);
  memcpy(&hf[0], x0_lqr, 8 * T * 8); memcpy(&hf[8 * T], Jmat, 9 * T * 8); memcpy(&hf[17 * T], index_scale, T * 8);
  memcpy(&hf[18 * T], clock_rate, T * 8); memcpy(&hf[19 * T], t_final, T * 8); memcpy(&hf[20 * T], q_final, 4 * T * 8);
  int64_t* d_i; double* d_f; uint32_t* d_s = nullptr;
  if ((rc = upload(c, SLOT_ARGS_A, hi.data(), hi.size(), &d_i))) return rc;
  if ((rc = upload(c, SLOT_ARGS_B, hf.data(), hf.size(), &d_f))) return rc;
  if (stream_id && (rc = upload(c, SLOT_ARGS_C, stream_id, T, &d_s))) return rc;
  void* p_o;
  if ((rc = scratch_reserve(c, SLOT_PER_TRIAL, T * 16, &p_o))) return rc;
  a.n_trials = n; a.N_i = d_i; a.offs = d_i + T; a.B_offs = d_i + 2 * T; a.B_rows = d_i + 3 * T;
  a.x0_lqr = d_f; a.Jmat = d_f + 8 * T;
  a.index_scale = d_f + 17 * T; a.clock_rate = d_f + 18 * T; a.t_final = d_f + 19 * T;
  a.q_final = d_f + 20 * T; a.stream_id = d_s;
  memcpy(&a.opts, &o, sizeof(o));
  a.N_sim = (int64_t*)p_o; a.slew_time = (double*)((int64_t*)p_o + T);
  if (N_sim) io.back(N_sim, a.N_sim, T);
  if (slew_time) io.back(slew_time, a.slew_time, T);
  if ((rc = k4_lin_table(c, N_i, T, a))) return rc;
  io.start();
  k4_launch(c, a);
  return io.finish();
}

// ---------------------------------------------------------------------------- fused Monte-Carlo
// Algorithmic FLOP per unit: AL-iLQR figures COUNTED with an instrumented scalar on the kernels' own math
// (tools/flopcount.cpp -> profiles/flop_counts_r2.json: JVP linearisation 6485 + cost gradients 51 + dense 7-state Riccati
// step 3688 + gradient measure 6 = 10230 per knot-iteration, 607 per line-search rollout knot; 9285 / 535 in the
// diagonal-inertia instantiation; SURVEY 8d's estimate was 6100 / 500);
// IGRF sample 2393 (2243 + rotations) and TVLQR ~7700 per knot are the SURVEY 8d estimates.
static const double FL_FIELD = 2393.0, FL_ITER = 10230.0, FL_ROLL = 607.0, FL_ITER_DIAG = 9285.0, FL_ROLL_DIAG = 535.0, FL_TVLQR = 7700.0;

// The counts and sums of ts_mc_stats over an ensemble's outcome records; flops starts at flops0 and adds every
// record's.  The ms_* fields are left to the caller.
static void mc_stats_of(const ts_trial_outcome* out, int64_t n, bool run_tvlqr, double flops0, ts_mc_stats* stats) {
  memset(stats, 0, sizeof(*stats));
  stats->n_trials = n;
  stats->flops = flops0;
  for (int64_t t = 0; t < n; ++t) {
    const ts_trial_outcome& o = out[t];
    if (o.status >= 0 && o.status < 6) stats->n_status[o.status]++;
    if (o.status == TS_ST_NO_CUTOFF) { stats->n_no_cutoff++; continue; }
    if (o.status == TS_ST_CONVERGED) stats->n_converged++;
    stats->sum_t_final += o.t_final;
    stats->sum_inner_iters += o.inner_iters;
    stats->sum_ls_rollouts += o.ls_rollouts;
    stats->sum_knots += (double)o.N;
    stats->flops += o.flops;
    if (run_tvlqr) {
      if (o.slew_time == o.t_final) stats->n_fail_slew++;
      if (o.slew_time > 0.0) { stats->sum_slew_time += o.slew_time; stats->sum_slew_time_sq += o.slew_time * o.slew_time; }
    }
  }
}

// FLOP of a trial of N knots over `inner` inner iterations and `ls` line-search rollouts (diag: the diagonal-inertia
// instantiation) and, with tvlqr, its replay: a record's flops, or with the counters' increments a continuation's work
static double trial_flops(bool diag, int64_t N, int64_t inner, int64_t ls, bool tvlqr) {
  const double kn = (double)(N - 1);
  return kn * ((double)inner * (diag ? FL_ITER_DIAG : FL_ITER) + (double)ls * (diag ? FL_ROLL_DIAG : FL_ROLL)) + (tvlqr ? kn * FL_TVLQR : 0.0);
}

static int upload_packed(ts_ctx* c, const McPacked& p, Slot si, Slot sf, McPackedView& v) {
  int64_t* d_i;
  double* d_f;
  int rc;
  if ((rc = upload(c, si, p.hi.data(), p.hi.size(), &d_i))) return rc;
  if ((rc = upload(c, sf, p.hf.data(), p.hf.size(), &d_f))) return rc;
  v = {d_i, d_f, p.n};
  return TS_OK;
}

// The fused path's weights block, written by k_slew_prep: Qd (8 per trial) | Qfd (8) | Rd (3) of the n active trials
struct McWeights {
  double *Qd, *Qfd, *Rd;
  McWeights(double* w, size_t n) : Qd(w), Qfd(w + 8 * n), Rd(w + 16 * n) {}
};

// The K3 arguments of the fused path: packed trials v, their weights w, field table B, trajectories X, U, outcome records
static K3Args fused_k3_args(const McPackedView& v, const McWeights& w, const double* B, double* X, double* U, ts_trial_outcome_dev* out,
                            const ts_ilqr_opts& opts, double dt) {
  K3Args a = {};
  a.n_trials = (int64_t)v.n;
  a.N_i = v.col(I_N); a.offs = v.col(I_OFFS); a.B_offs = v.col(I_B_OFFS); a.B_rows = v.col(I_B_ROWS);
  a.x0 = v.col(F_X0); a.xf = v.col(F_XF); a.Jmat = v.col(F_JMAT); a.Qd = w.Qd; a.Qfd = w.Qfd; a.Rd = w.Rd;
  a.index_scale = v.col(F_INDEX_SCALE); a.clock_rate = v.col(F_CLOCK_RATE);
  a.B_eci = B; a.dt = dt; a.U0 = nullptr;
  memcpy(&a.opts, &opts, sizeof(a.opts));
  a.X = X; a.U = U; a.K = nullptr; a.out = out;
  return a;
}

// The run's TVLQR options with the fused path's overrides
static ts_tvlqr_opts_dev fused_tvlqr_opts(const ts_mc_config& cfg) {
  ts_tvlqr_opts_dev o;
  memcpy(&o, &cfg.tvlqr, sizeof(o));
  o.dt = cfg.dt; o.t0 = cfg.t0;
  if (o.noise_mode == 1) o.noise_mode = 2;  // no explicit array in the fused path
  o.literal_postproc = 0;                   // needs X_sim storage; fused path uses the fixed rule (Q12)
  return o;
}

// Completes a (holding k4_lin_table's table) to the K4 arguments of a fused replay of the packed trials v on trajectories
// X, U, field table B, gains K and stream ids sid; X_sim, U_sim, N_sim and slew_time are null until the caller sets them.
static void fused_k4_args(K4Args& a, const McPackedView& v, const double* X, const double* U, const double* B, double* K,
                          const uint32_t* sid, const ts_mc_config& cfg) {
  a.n_trials = (int64_t)v.n; a.N_i = v.col(I_N); a.offs = v.col(I_OFFS); a.B_offs = v.col(I_B_OFFS); a.B_rows = v.col(I_B_ROWS);
  a.X_lqr = X; a.U_lqr = U; a.x0_lqr = v.col(F_X0LQR); a.Jmat = v.col(F_JMAT); a.B_eci = B;
  a.index_scale = v.col(F_INDEX_SCALE); a.clock_rate = v.col(F_CLOCK_RATE); a.t_final = v.col(F_T_FINAL); a.q_final = v.col(F_Q_FINAL);
  a.stream_id = sid;
  a.opts = fused_tvlqr_opts(cfg);
  a.noise = nullptr; a.X_sim = nullptr; a.U_sim = nullptr; a.dX = nullptr; a.K = K;
  a.N_sim = nullptr; a.slew_time = nullptr;
}

int ts_monte_carlo_run(ts_ctx* c, const ts_mc_config* cfg, const double* kep6, const ts_field_opts* fopts, const double* x0,
                       const double* xf, const double* Jmat, const double* q_noise0, const uint32_t* stream_id,
                       ts_trial_outcome* out, ts_mc_stats* stats) {
  if (!c) return TS_ERR_ARG;
  if (!cfg || !kep6 || !fopts || !x0 || !xf || !Jmat || !out) return fail(c, TS_ERR_ARG, "ts_monte_carlo_run: null argument");
  const int64_t n = cfg->n_trials;
  if (n < 0) return fail(c, TS_ERR_ARG, "n_trials < 0");
  if (stats) memset(stats, 0, sizeof(*stats));
  if (n == 0) return TS_OK;
  if (!(cfg->dt > 0) || cfg->N_scope < 1 || !(cfg->tf > cfg->t0)) return fail(c, TS_ERR_ARG, "ts_monte_carlo_run: bad config");
  TS_CUDA(c, cudaSetDevice(c->device));
  const int64_t nf = cfg->shared_orbit ? 1 : n;
  const size_t NF = (size_t)nf;
  int rc;
  Events<7> e;
  ts_ctx::McLast& L = c->mc_last;
  L = {};

  // ---- stage 1: scoping pass (2*N_scope samples per orbit) + gramian cutoff
  std::vector<ts_field_opts> fo(NF);
  std::vector<int64_t> offs_s(NF + 1);
  bool any13 = false, any10 = false;
  for (int64_t f = 0; f < nf; ++f) {
    fo[f] = fopts[f];
    fo[f].t0 = cfg->t0; fo[f].tf = cfg->tf; fo[f].N = cfg->N_scope;
    if (!igrf_date_ok(fo[f].igrf_date)) return fail(c, TS_ERR_DATE, "orbit %lld: IGRF date outside [1900, 2025]", (long long)f);
    (igrf_nmax_for_date(fo[f].igrf_date) == 13 ? any13 : any10) = true;
    offs_s[f] = 2 * cfg->N_scope * f;
  }
  offs_s[nf] = 2 * cfg->N_scope * nf;
  double* d_kep; ts_field_opts_dev* d_fo; int64_t* d_offs_s;
  if ((rc = upload(c, SLOT_ARGS_A, kep6, 6 * NF, &d_kep))) return rc;
  if ((rc = upload(c, SLOT_ARGS_B, (const ts_field_opts_dev*)fo.data(), NF, &d_fo))) return rc;
  if ((rc = upload(c, SLOT_ARGS_C, offs_s.data(), NF + 1, &d_offs_s))) return rc;
  void *p_pos, *p_Bs, *p_sm;
  if ((rc = scratch_reserve(c, SLOT_POSITIONS, (size_t)(offs_s[nf] + nf) * 3 * 8, &p_pos))) return rc;
  if ((rc = scratch_reserve(c, SLOT_ROWS_A, (size_t)offs_s[nf] * 3 * 8, &p_Bs))) return rc;
  if ((rc = scratch_reserve(c, SLOT_ORBIT_BLOCK, NF * 80, &p_sm))) return rc;
  std::vector<int64_t> rows_s(NF, 2 * cfg->N_scope);
  std::vector<double> dts(NF, (cfg->tf - cfg->t0) / (double)cfg->N_scope), cuts(NF, cfg->cutoff);
  int64_t* d_rows_s = (int64_t*)p_sm;
  double* d_dts = (double*)((char*)p_sm + NF * 8);
  double* d_cuts = (double*)((char*)p_sm + NF * 16);
  int64_t* d_idx = (int64_t*)((char*)p_sm + NF * 24);
  double* d_carry = (double*)((char*)p_sm + NF * 32);   // running gramian of an orbit between two sample ranges
  TS_CUDA(c, cudaMemcpyAsync(d_rows_s, rows_s.data(), NF * 8, cudaMemcpyHostToDevice, c->stream));
  TS_CUDA(c, cudaMemcpyAsync(d_dts, dts.data(), NF * 8, cudaMemcpyHostToDevice, c->stream));
  TS_CUDA(c, cudaMemcpyAsync(d_cuts, cuts.data(), NF * 8, cudaMemcpyHostToDevice, c->stream));
  cudaEventRecord(e[0], c->stream);
  k2a_orbit_euler<<<(unsigned)((nf + 127) / 128), 128, 0, c->stream>>>(nf, d_kep, d_fo, d_offs_s, nullptr, (double*)p_pos, nullptr);
  c->launches++;
  // field rows and cutoff search in two sample ranges: most orbits reach the cutoff within the first few thousand
  // samples, and the second range skips those (no host round trip: the kernels look at d_idx themselves)
  TS_CUDA(c, cudaMemsetAsync(d_idx, 0, NF * 8, c->stream));
  {
    const int64_t S2 = 2 * cfg->N_scope, SA = std::min<int64_t>(S2, 4096);
    for (int pass = 0; pass < 2; ++pass) {
      const int64_t lo = pass ? SA : 0, hi = pass ? S2 : SA;
      if (hi <= lo) break;
      k2b_launch(c, any13, any10, nf, hi - lo, d_fo, d_offs_s, nullptr, (double*)p_pos, (double*)p_Bs, lo, pass ? d_idx : nullptr);
      k2c_cutoff_scan<<<(unsigned)nf, K2C_THREADS, 0, c->stream>>>((double*)p_Bs, d_offs_s, d_rows_s, d_dts, d_cuts, lo, hi, d_carry, d_idx);
      c->launches++;
    }
  }
  cudaEventRecord(e[6], c->stream);   // end of the scoping stage on the device (the host sync below is not device time)
  TS_CUDA(c, cudaGetLastError());
  std::vector<int64_t> idx(NF);
  TS_CUDA(c, cudaMemcpyAsync(idx.data(), d_idx, NF * 8, cudaMemcpyDeviceToHost, c->stream));
  TS_CUDA(c, cudaStreamSynchronize(c->stream));

  // ---- host: horizons (TortoiseSat.jl:82-86), fine-pass layout
  std::vector<double> tfin(NF, 0.0);
  std::vector<int64_t> Nf(NF, 0), offs_f(NF + 1, 0), lim(NF, 0);
  std::vector<ts_field_opts> fo2(NF);
  int64_t maxNf = 1;
  double field_samples = 0.0;
  for (int64_t f = 0; f < nf; ++f) {
    fo2[f] = fo[f];
    {  // scoping samples evaluated for this orbit: the first range, and the second one only if the cutoff was not in it
      const int64_t S2 = 2 * cfg->N_scope, SA = std::min<int64_t>(S2, 4096);
      field_samples += (idx[f] > 0 && idx[f] <= SA) ? (double)SA : (double)S2 - 1.0;
    }
    if (idx[f] > 0) {
      tfin[f] = (double)idx[f] * (cfg->tf - cfg->t0) / (double)cfg->N_scope;
      Nf[f] = (int64_t)floor((tfin[f] - cfg->t0) / cfg->dt);
    }
    if (Nf[f] < 2) { Nf[f] = 0; fo2[f].N = 1; fo2[f].tf = cfg->t0 + 1.0; lim[f] = 1; offs_f[f + 1] = offs_f[f] + 2; continue; }
    fo2[f].tf = tfin[f];
    fo2[f].N = Nf[f];
    // rows the solver / replay can index: floor(x8*N + 1), x8 <= N*dt/(tf-t0)   (DerivFunction.jl:28,44)
    const double x8max = (double)(Nf[f] + 1) * cfg->dt / (cfg->tf - cfg->t0);
    int64_t need = (int64_t)floor(x8max * (double)Nf[f] + 1.0) + 4;
    if (need > 2 * Nf[f] - 1) need = 2 * Nf[f] - 1;
    lim[f] = need;
    field_samples += (double)need;
    offs_f[f + 1] = offs_f[f] + 2 * Nf[f];
    maxNf = std::max(maxNf, Nf[f]);
  }
  // active trials
  std::vector<int64_t> act;
  act.reserve((size_t)n);
  for (int64_t t = 0; t < n; ++t) {
    const int64_t f = cfg->shared_orbit ? 0 : t;
    if (Nf[f] >= 2) act.push_back(t);
    else {
      memset(&out[t], 0, sizeof(out[t]));
      out[t].status = TS_ST_NO_CUTOFF;
    }
  }
  const int64_t na = (int64_t)act.size();
  const size_t NA = (size_t)na;
  double ms_field = 0, ms_prep = 0, ms_solve = 0, ms_tvlqr = 0;
  if (na > 0) {
    // ---- stage 2: fine field tables
    ts_field_opts_dev* d_fo2; int64_t *d_offs_f, *d_lim;
    if ((rc = upload(c, SLOT_ARGS_B, (const ts_field_opts_dev*)fo2.data(), NF, &d_fo2))) return rc;
    if ((rc = upload(c, SLOT_ARGS_C, offs_f.data(), NF + 1, &d_offs_f))) return rc;
    if ((rc = upload(c, SLOT_ROW_LIMITS, lim.data(), NF, &d_lim))) return rc;
    void* p_pos2;
    if ((rc = scratch_reserve(c, SLOT_POSITIONS, std::max((size_t)(offs_s[nf] + nf) * 3 * 8, (size_t)(offs_f[nf] + nf) * 3 * 8), &p_pos2))) return rc;
    // per-trial layout
    McPacked P(NA);
    int64_t knots = 0;
    for (int64_t a = 0; a < na; ++a) {
      const int64_t t = act[a], f = cfg->shared_orbit ? 0 : t;
      P.col(I_N)[a] = Nf[f];
      P.col(I_OFFS)[a] = knots;
      P.col(I_B_OFFS)[a] = offs_f[f];
      P.col(I_B_ROWS)[a] = 2 * Nf[f];
      knots += Nf[f];
      memcpy(P.at(F_X0, a), x0 + 8 * t, 64);
      memcpy(P.at(F_XF, a), xf + 8 * t, 64);
      memcpy(P.at(F_JMAT, a), Jmat + 9 * t, 72);
      *P.at(F_T_FINAL, a) = tfin[f];
      *P.at(F_INDEX_SCALE, a) = (double)Nf[f];
      *P.at(F_CLOCK_RATE, a) = 1.0 / (cfg->tf - cfg->t0);
      // x0_lqr (TortoiseSat.jl:227-234): omega from x0, attitude perturbed by q_noise0, clock 0
      tvlqr_x0_lqr(x0 + 8 * t, q_noise0 ? q_noise0 + 3 * t : nullptr, P.at(F_X0LQR, a));
      memcpy(P.at(F_Q_FINAL, a), xf + 8 * t + 3, 32);
      P.sid[a] = stream_id ? stream_id[t] : (uint32_t)t;
    }
    P.hi.back() = knots;
    McPackedView v;
    if ((rc = upload_packed(c, P, SLOT_PACKED_I64, SLOT_PACKED_F64, v))) return rc;
    // device block: fine field tables, weights, X, U, outcomes, slew times
    const size_t b_B = (size_t)offs_f[nf] * 3 * 8, b_w = 19 * NA * 8, b_X = (size_t)knots * 8 * 8, b_U = (size_t)knots * 3 * 8,
                 b_o = NA * sizeof(ts_trial_outcome), b_s = NA * 16;
    void* p_blk;
    if ((rc = scratch_reserve(c, SLOT_KEPT_BLOCK, b_B + b_w + b_X + b_U + b_o + b_s + 512, &p_blk))) return rc;
    char* w = (char*)p_blk;
    double* d_Bf = (double*)w; w += b_B;
    double* d_Qd = (double*)w; w += b_w;
    double* d_X = (double*)w; w += b_X;
    double* d_U = (double*)w; w += b_U;
    ts_trial_outcome_dev* d_out = (ts_trial_outcome_dev*)w; w += b_o;
    int64_t* d_nsim = (int64_t*)w; double* d_slew = (double*)(w + NA * 8);
    cudaEventRecord(e[1], c->stream);  // fine pass starts
    k2a_orbit_euler<<<(unsigned)((nf + 127) / 128), 128, 0, c->stream>>>(nf, d_kep, d_fo2, d_offs_f, d_lim, (double*)p_pos2, nullptr);
    c->launches++;
    {
      int64_t maxlim = 1;
      for (int64_t f = 0; f < nf; ++f) maxlim = std::max(maxlim, 2 * std::max<int64_t>(Nf[f], 1));
      k2b_launch(c, any13, any10, nf, maxlim, d_fo2, d_offs_f, d_lim, (double*)p_pos2, d_Bf);
    }
    cudaEventRecord(e[2], c->stream);
    // ---- stage 3: eigen-axis guess + Bryson weights
    const McWeights wt(d_Qd, NA);
    PrepArgs pa;
    pa.n_trials = na; pa.x0 = v.col(F_X0); pa.xf = v.col(F_XF); pa.Jmat = v.col(F_JMAT); pa.t_final = v.col(F_T_FINAL);
    pa.t0 = cfg->t0; pa.dt = cfg->dt; pa.alpha = cfg->alpha; pa.beta = cfg->beta; pa.conj_fix = cfg->eigen_axis_fix ? 1 : 0;
    pa.Qd = wt.Qd; pa.Qfd = wt.Qfd; pa.Rd = wt.Rd;
    pa.goffs = nullptr; pa.w_guess = nullptr; pa.q_guess = nullptr;
    k_slew_prep<<<(unsigned)((na + 127) / 128), 128, 0, c->stream>>>(pa);
    c->launches++;
    cudaEventRecord(e[3], c->stream);
    // ---- stage 4: AL-iLQR
    K3Args ka = fused_k3_args(v, wt, d_Bf, d_X, d_U, d_out, cfg->ilqr, cfg->dt);
    std::vector<double> diff(NA);
    for (int64_t aa = 0; aa < na; ++aa) diff[aa] = slew_angle(x0 + 8 * act[aa], xf + 8 * act[aa]);
    // keep_trajectories = 2: the solve runs the exporting instantiations, its states and multipliers go to a kept slot
    K3StateIO sio = {};
    void* p_st = nullptr;
    const bool keep_state = cfg->keep_trajectories == 2;
    const size_t b_st = NA * sizeof(ts_al_state);
    if (keep_state) {
      if ((rc = scratch_reserve(c, SLOT_KEPT_STATE, b_st + 64 + (size_t)knots * 6 * 8, &p_st))) return rc;
      sio.state_out = (ts_al_state_dev*)p_st;
      sio.lam_out = (double*)((char*)p_st + b_st + 64);
      ka.sio = (const K3StateIO*)((char*)p_st + b_st);
    }
    // everything stage 5 needs is reserved and uploaded BEFORE the solve is queued: a cudaMalloc between the two would
    // wait for the solve and put its host latency on the device timeline
    void *p_K = nullptr, *p_xs = nullptr, *p_us = nullptr;
    uint32_t* d_sid = nullptr;
    K4Args k4;
    if (cfg->run_tvlqr) {
      if ((rc = scratch_reserve(c, SLOT_K4_GAINS, (size_t)knots * 18 * 8, &p_K))) return rc;
      if ((rc = upload(c, SLOT_STREAM_IDS, P.sid.data(), NA, &d_sid))) return rc;
      if ((rc = k4_lin_table(c, P.col(I_N), NA, k4))) return rc;
      if (cfg->keep_trajectories) {
        if ((rc = scratch_reserve(c, SLOT_KEPT_XSIM, (size_t)knots * 8 * 8 + 64, &p_xs))) return rc;
        if ((rc = scratch_reserve(c, SLOT_KEPT_USIM, (size_t)knots * 3 * 8 + 64, &p_us))) return rc;
      }
    }
    if ((rc = k3_launch(c, ka, P.col(I_N), diff.data(), all_inertia_diagonal(Jmat, n), nullptr, keep_state ? &sio : nullptr))) return rc;
    cudaEventRecord(e[4], c->stream);
    // ---- stage 5: TVLQR replay + slew-time rule
    double *d_Xs_keep = nullptr, *d_Us_keep = nullptr;
    if (cfg->run_tvlqr) {
      fused_k4_args(k4, v, d_X, d_U, d_Bf, (double*)p_K, d_sid, *cfg);
      if (cfg->keep_trajectories) {
        TS_CUDA(c, cudaMemsetAsync(p_xs, 0, (size_t)knots * 8 * 8, c->stream));
        TS_CUDA(c, cudaMemsetAsync(p_us, 0, (size_t)knots * 3 * 8, c->stream));
        k4.X_sim = (double*)p_xs; k4.U_sim = (double*)p_us;
        d_Xs_keep = k4.X_sim; d_Us_keep = k4.U_sim;
      }
      k4.N_sim = d_nsim; k4.slew_time = d_slew;
      k4_launch(c, k4);
    }
    cudaEventRecord(e[5], c->stream);
    TS_CUDA(c, cudaGetLastError());
    std::vector<ts_trial_outcome> oa(NA);
    std::vector<double> slew(NA, 0.0);
    TS_CUDA(c, cudaMemcpyAsync(oa.data(), d_out, b_o, cudaMemcpyDeviceToHost, c->stream));
    if (cfg->run_tvlqr) TS_CUDA(c, cudaMemcpyAsync(slew.data(), d_slew, NA * 8, cudaMemcpyDeviceToHost, c->stream));
    TS_CUDA(c, cudaStreamSynchronize(c->stream));
    ms_field = e.ms(0, 6);
    ms_field += e.ms(1, 2);
    ms_prep = e.ms(2, 3);
    ms_solve = e.ms(3, 4);
    ms_tvlqr = e.ms(4, 5);
    const bool dj = all_inertia_diagonal(Jmat, n) && !cfg->ilqr.k3_generic_inertia;
    for (int64_t a = 0; a < na; ++a) {
      const int64_t t = act[a], f = cfg->shared_orbit ? 0 : t;
      out[t] = oa[a];
      out[t].t_final = tfin[f];
      out[t].slew_time = cfg->run_tvlqr ? slew[a] : 0.0;
      out[t].flops = trial_flops(dj, Nf[f], oa[a].inner_iters, oa[a].ls_rollouts, cfg->run_tvlqr != 0);
    }
    if (cfg->keep_trajectories) {
      L.knots = knots; L.rows = offs_f[nf];
      L.knot_offs.assign((size_t)n + 1, 0);
      L.row_offs.assign((size_t)n + 1, 0);
      for (int64_t t = 0; t < n; ++t) {
        const int64_t f = cfg->shared_orbit ? 0 : t;
        L.knot_offs[t + 1] = L.knot_offs[t] + (Nf[f] >= 2 ? Nf[f] : 0);
        L.row_offs[t] = cfg->shared_orbit ? 0 : offs_f[f];
      }
      L.row_offs[n] = offs_f[nf];
      L.d_X = d_X; L.d_U = d_U; L.d_Xs = d_Xs_keep; L.d_Us = d_Us_keep; L.d_B = d_Bf;
      // the host side of the kept run: what ts_mc_replay_ensemble (and, with keep_trajectories = 2, ts_mc_continue) needs
      L.diag_inertia = all_inertia_diagonal(Jmat, n);
      L.act = act;
      L.in = std::move(P);
    }
    if (keep_state) {
      L.d_in = v; L.d_w = d_Qd;
      L.d_out = (ts_trial_outcome*)d_out;
      L.d_state = (ts_al_state*)p_st;
      L.d_sio = (char*)p_st + b_st;
      L.d_lam = sio.lam_out;
    }
  }
  if (cfg->keep_trajectories) {
    L.cfg = *cfg;
    L.n = n;
    L.out.assign(out, out + n);
  }
  c->last_kernel_ms = ms_field + ms_prep + ms_solve + ms_tvlqr;
  if (stats) {
    mc_stats_of(out, n, cfg->run_tvlqr != 0, field_samples * FL_FIELD, stats);
    stats->ms_field = ms_field; stats->ms_prep = ms_prep; stats->ms_solve = ms_solve; stats->ms_tvlqr = ms_tvlqr;
  }
  return TS_OK;
}

int ts_mc_trajectory_layout(ts_ctx* c, int64_t n_trials, int64_t* knot_offs, int64_t* row_offs) {
  if (!c) return TS_ERR_ARG;
  const ts_ctx::McLast& L = c->mc_last;
  if (!L.cfg.keep_trajectories || L.act.empty()) return fail(c, TS_ERR_ARG, "no Monte-Carlo run with keep_trajectories = 1 on this context");
  if (n_trials != L.n) return fail(c, TS_ERR_ARG, "the kept run had %lld trials", (long long)L.n);
  if (knot_offs) memcpy(knot_offs, L.knot_offs.data(), (size_t)(L.n + 1) * 8);
  if (row_offs) memcpy(row_offs, L.row_offs.data(), (size_t)(L.n + 1) * 8);
  return TS_OK;
}

int ts_mc_fetch_trajectories(ts_ctx* c, double* X, double* U, double* X_sim, double* U_sim, double* B_eci) {
  if (!c) return TS_ERR_ARG;
  const ts_ctx::McLast& L = c->mc_last;
  if (!L.cfg.keep_trajectories || L.act.empty()) return fail(c, TS_ERR_ARG, "no Monte-Carlo run with keep_trajectories = 1 on this context");
  if ((X_sim || U_sim) && !L.d_Xs) return fail(c, TS_ERR_ARG, "the kept run had run_tvlqr = 0: no X_sim / U_sim");
  TS_CUDA(c, cudaSetDevice(c->device));
  const size_t K = (size_t)L.knots;
  if (X) TS_CUDA(c, cudaMemcpyAsync(X, L.d_X, K * 8 * 8, cudaMemcpyDeviceToHost, c->stream));
  if (U) TS_CUDA(c, cudaMemcpyAsync(U, L.d_U, K * 3 * 8, cudaMemcpyDeviceToHost, c->stream));
  if (X_sim) TS_CUDA(c, cudaMemcpyAsync(X_sim, L.d_Xs, K * 8 * 8, cudaMemcpyDeviceToHost, c->stream));
  if (U_sim) TS_CUDA(c, cudaMemcpyAsync(U_sim, L.d_Us, K * 3 * 8, cudaMemcpyDeviceToHost, c->stream));
  if (B_eci) TS_CUDA(c, cudaMemcpyAsync(B_eci, L.d_B, (size_t)L.rows * 3 * 8, cudaMemcpyDeviceToHost, c->stream));
  TS_CUDA(c, cudaStreamSynchronize(c->stream));
  return TS_OK;
}

int ts_mc_fetch_state(ts_ctx* c, ts_al_state* state, double* lam) {
  if (!c) return TS_ERR_ARG;
  const ts_ctx::McLast& L = c->mc_last;
  if (L.cfg.keep_trajectories != 2) return fail(c, TS_ERR_ARG, "no Monte-Carlo run with keep_trajectories = 2 on this context");
  TS_CUDA(c, cudaSetDevice(c->device));
  const size_t NA = L.act.size();
  std::vector<ts_al_state> st(NA);
  if (state && NA) TS_CUDA(c, cudaMemcpyAsync(st.data(), L.d_state, NA * sizeof(ts_al_state), cudaMemcpyDeviceToHost, c->stream));
  if (lam && L.knots) TS_CUDA(c, cudaMemcpyAsync(lam, L.d_lam, (size_t)L.knots * 6 * 8, cudaMemcpyDeviceToHost, c->stream));
  TS_CUDA(c, cudaStreamSynchronize(c->stream));
  if (state) {
    memset(state, 0, (size_t)L.n * sizeof(ts_al_state));
    for (int64_t t = 0; t < L.n; ++t) state[t].status = TS_ST_NO_CUTOFF;
    for (size_t a = 0; a < NA; ++a) state[L.act[a]] = st[a];
  }
  return TS_OK;
}

// MC1-MC3 (DESIGN.md section 4, K3).  The continuing trials are solved on the kept block in place, exactly as
// ts_alilqr_solve_state_batch continues them over the run's active trials, and replayed on their own.
int ts_mc_continue(ts_ctx* c, int64_t n_trials, const ts_ilqr_opts* opts, ts_trial_outcome* out, ts_mc_stats* stats) {
  if (!c) return TS_ERR_ARG;
  ts_ctx::McLast& L = c->mc_last;
  if (L.cfg.keep_trajectories != 2) return fail(c, TS_ERR_ARG, "ts_mc_continue: no Monte-Carlo run with keep_trajectories = 2 on this context");
  if (n_trials != L.n) return fail(c, TS_ERR_ARG, "ts_mc_continue: the kept run had %lld trials", (long long)L.n);
  if (!opts || !out) return fail(c, TS_ERR_ARG, "ts_mc_continue: null argument");
  const ts_ilqr_opts& o = *opts;
  const int64_t na = (int64_t)L.act.size();
  const size_t NA = (size_t)na;
  const ts_mc_config& cfg = L.cfg;
  TS_CUDA(c, cudaSetDevice(c->device));
  int rc;
  // the option checks of ts_alilqr_solve_state_batch; quat_error's reads the run's weights back
  const size_t nw = o.quat_error ? NA : 0;
  std::vector<double> w(16 * nw);
  if (nw) TS_CUDA(c, cudaMemcpy(w.data(), L.d_w, w.size() * 8, cudaMemcpyDeviceToHost));
  const McWeights hw(w.data(), nw);
  if ((rc = check_ilqr_opts(c, o, (int64_t)nw, hw.Qd, hw.Qfd))) return rc;
  // MC1: CS2 on the kept states (their status and outer count are the kept records')
  std::vector<int64_t> cont;
  for (int64_t a = 0; a < na; ++a) {
    const ts_trial_outcome& r = L.out[(size_t)L.act[(size_t)a]];
    if (r.status == TS_ST_MAX_OUTER && r.outer_iters < o.max_outer) cont.push_back(a);
  }
  const size_t NC = cont.size();
  double ms_solve = 0.0, ms_tvlqr = 0.0, flops = 0.0;
  std::vector<ts_trial_outcome> rec = L.out;
  if (NC == 0) c->k3_timed = false;   // no solve: ts_k3_last_split / ts_k3_last_parked report nothing
  if (NC > 0) {
    // MC3: the replay's per-trial arrays, compacted to the continuing trials
    const McPacked P = L.in.compact(cont);
    McPackedView v;
    void *p_q = nullptr, *p_K = nullptr;
    K4Args k4;
    if (cfg.run_tvlqr) {
      if ((rc = upload_packed(c, P, SLOT_ARGS_A, SLOT_ARGS_B, v))) return rc;
      if ((rc = scratch_reserve(c, SLOT_ARGS_C, NC * 20 + 64, &p_q))) return rc;
      TS_CUDA(c, cudaMemcpyAsync(p_q, P.sid.data(), NC * 4, cudaMemcpyHostToDevice, c->stream));
      if ((rc = scratch_reserve(c, SLOT_K4_GAINS, (size_t)L.knots * 18 * 8, &p_K))) return rc;
      if ((rc = k4_lin_table(c, P.col(I_N), NC, k4))) return rc;
    }
    // MC2: the K3 arguments of the run, on the kept block; the states and multipliers are read and written in place
    K3Args ka = fused_k3_args(L.d_in, McWeights(L.d_w, NA), L.d_B, L.d_X, L.d_U, (ts_trial_outcome_dev*)L.d_out, o, cfg.dt);
    ka.sio = (const K3StateIO*)L.d_sio;
    K3StateIO sio = {};
    sio.state_in = sio.state_out = (ts_al_state_dev*)L.d_state;
    sio.lam_in = sio.lam_out = L.d_lam;
    sio.lam_doubles = L.knots * 6;
    std::vector<double> diff(NA);
    for (size_t a = 0; a < NA; ++a) diff[a] = slew_angle(L.in.at(F_X0, a), L.in.at(F_XF, a));
    Events<3> e;
    cudaEventRecord(e[0], c->stream);
    // X, U, the states and lam are input and output of the same call.  That is safe because park_import_kernel, the
    // first kernel k3_launch queues for a continuation, reads every imported row (X, U, lam_in, state_in) before the
    // straggler kernel that follows it on the stream writes any.  k3_launch fails before it queues anything that writes
    // kept storage (TS_ERR_NOMEM when the parked records do not fit), so the kept run stays continuable.
    if ((rc = k3_launch(c, ka, L.in.col(I_N), diff.data(), L.diag_inertia, &cont, &sio))) return rc;
    cudaEventRecord(e[1], c->stream);
    if (cfg.run_tvlqr) {
      k4_clear_rows_kernel<<<(unsigned)NC, 256, 0, c->stream>>>((int64_t)NC, v.col(I_N), v.col(I_OFFS), L.d_Xs, L.d_Us);
      c->launches++;
      fused_k4_args(k4, v, L.d_X, L.d_U, L.d_B, (double*)p_K, (const uint32_t*)p_q, cfg);
      k4.X_sim = L.d_Xs; k4.U_sim = L.d_Us;
      k4.N_sim = (int64_t*)((char*)p_q + ((NC * 4 + 15) & ~(size_t)15));
      k4.slew_time = (double*)(k4.N_sim + NC);
      k4_launch(c, k4);
    }
    cudaEventRecord(e[2], c->stream);
    TS_CUDA(c, cudaGetLastError());
    std::vector<ts_trial_outcome> oa(NA);
    std::vector<double> slew(NC, 0.0);
    TS_CUDA(c, cudaMemcpyAsync(oa.data(), L.d_out, NA * sizeof(ts_trial_outcome), cudaMemcpyDeviceToHost, c->stream));
    if (cfg.run_tvlqr) TS_CUDA(c, cudaMemcpyAsync(slew.data(), k4.slew_time, NC * 8, cudaMemcpyDeviceToHost, c->stream));
    TS_CUDA(c, cudaStreamSynchronize(c->stream));
    ms_solve = e.ms(0, 1);
    if (cfg.run_tvlqr) ms_tvlqr = e.ms(1, 2);
    const bool dj = L.diag_inertia && !o.k3_generic_inertia, tv = cfg.run_tvlqr != 0;
    for (size_t k = 0; k < NC; ++k) {
      const int64_t t = L.act[(size_t)cont[k]];
      const ts_trial_outcome& prev = L.out[(size_t)t];
      ts_trial_outcome r = oa[(size_t)cont[k]];
      r.N = prev.N;
      r.t_final = prev.t_final;
      r.slew_time = cfg.run_tvlqr ? slew[k] : 0.0;
      r.flops = trial_flops(dj, prev.N, r.inner_iters, r.ls_rollouts, tv);
      flops += trial_flops(dj, prev.N, r.inner_iters - prev.inner_iters, r.ls_rollouts - prev.ls_rollouts, tv);
      rec[(size_t)t] = r;
    }
    L.out = rec;
  }
  c->last_kernel_ms = ms_solve + ms_tvlqr;
  memcpy(out, rec.data(), (size_t)L.n * sizeof(ts_trial_outcome));
  if (stats) {
    mc_stats_of(out, L.n, cfg.run_tvlqr != 0, 0.0, stats);
    stats->flops = flops;
    stats->ms_solve = ms_solve; stats->ms_tvlqr = ms_tvlqr;
  }
  return TS_OK;
}

// RE1-RE5 (DESIGN.md section 4, K4): the kept run's slews replayed under n_real disturbance draws each.  The gains of
// the selected trials come from the unchanged K4a + K4b on host-compacted arrays (as ts_mc_continue replays), then K4e
// replays every (trial, realisation) pair.  Only per-call slots are written: the kept run stays as it was (RE5).
int ts_mc_replay_ensemble(ts_ctx* c, int64_t n_trials, const ts_replay_ensemble_opts* opts, int64_t n_sel, const int64_t* trials,
                          double* slew_time, double* x_final) {
  if (!c) return TS_ERR_ARG;
  const ts_ctx::McLast& L = c->mc_last;
  if (L.cfg.keep_trajectories < 1) return fail(c, TS_ERR_ARG, "ts_mc_replay_ensemble: no Monte-Carlo run with keep_trajectories >= 1 on this context");
  if (n_trials != L.n) return fail(c, TS_ERR_ARG, "ts_mc_replay_ensemble: the kept run had %lld trials", (long long)L.n);
  if (!opts || !slew_time) return fail(c, TS_ERR_ARG, "ts_mc_replay_ensemble: null argument");
  const int64_t R = opts->n_real, r0 = opts->r_first;
  if (R < 1 || r0 < 0 || r0 + R > ((int64_t)1 << 30))
    return fail(c, TS_ERR_ARG, "ts_mc_replay_ensemble: need n_real >= 1, r_first >= 0, r_first + n_real <= 2^30");
  if (trials ? n_sel < 0 : n_sel != n_trials)
    return fail(c, TS_ERR_ARG, "ts_mc_replay_ensemble: n_sel must be >= 0 (= n_trials without a trial list)");
  for (int64_t p = 0; trials && p < n_sel; ++p)
    if (trials[p] < 0 || trials[p] >= n_trials) return fail(c, TS_ERR_ARG, "ts_mc_replay_ensemble: trial %lld out of range", (long long)trials[p]);
  // selected active trials, longest horizon first (stable: repeats and the caller's order decide nothing about a row, RE4)
  std::vector<int64_t> act_of((size_t)n_trials, -1);
  for (size_t a = 0; a < L.act.size(); ++a) act_of[(size_t)L.act[a]] = (int64_t)a;
  std::vector<int64_t> pos;   // caller rows with an active trial
  for (int64_t p = 0; p < n_sel; ++p)
    if (act_of[(size_t)(trials ? trials[p] : p)] >= 0) pos.push_back(p);
  auto act_at = [&](int64_t p) { return act_of[(size_t)(trials ? trials[p] : p)]; };
  std::stable_sort(pos.begin(), pos.end(), [&](int64_t u, int64_t v) { return L.in.col(I_N)[act_at(u)] > L.in.col(I_N)[act_at(v)]; });
  const size_t NC = pos.size(), RR = (size_t)R;
  const size_t per = x_final ? 9 : 1;   // doubles per (trial, realisation) row
  std::vector<double> hs(NC * RR), hx(x_final ? NC * RR * 8 : 0);
  c->ens_ms[0] = c->ens_ms[1] = 0.0;
  c->last_kernel_ms = 0.0;
  if (NC > 0) {
    TS_CUDA(c, cudaSetDevice(c->device));
    std::vector<int64_t> sel(NC);
    for (size_t k = 0; k < NC; ++k) sel[k] = act_at(pos[k]);
    const McPacked P = L.in.compact(sel);
    int rc;
    void *p_out, *p_K;
    if ((rc = scratch_reserve(c, SLOT_ENSEMBLE_OUT, NC * RR * per * 8 + 64, &p_out))) return rc;
    if ((rc = scratch_reserve(c, SLOT_K4_GAINS, (size_t)L.knots * 18 * 8, &p_K))) return rc;
    McPackedView v;
    uint32_t* d_sid;
    if ((rc = upload_packed(c, P, SLOT_ARGS_A, SLOT_ARGS_B, v))) return rc;
    if ((rc = upload(c, SLOT_ARGS_C, P.sid.data(), NC, &d_sid))) return rc;
    K4Args k4;
    if ((rc = k4_lin_table(c, P.col(I_N), NC, k4))) return rc;
    fused_k4_args(k4, v, L.d_X, L.d_U, L.d_B, (double*)p_K, d_sid, L.cfg);   // RE2: the run's options with the overrides
    k4.opts.noise_mode = 2;                                                  // realisations always draw
    K4eArgs e = k4e_args(k4, v.col(F_X0));
    e.n_real = R; e.r_first = r0; e.n_blk = (R + 31) / 32;
    e.q_noise_scale = opts->q_noise_scale;
    e.slew_time = (double*)p_out;
    e.x_final = x_final ? e.slew_time + NC * RR : nullptr;
    Events<3> ev;
    cudaEventRecord(ev[0], c->stream);
    k4_gains_launch(c, k4);
    cudaEventRecord(ev[1], c->stream);
    const int64_t warps = (int64_t)NC * e.n_blk;
    k4e_ensemble_replay_kernel<<<(unsigned)((warps + K4E_WARPS - 1) / K4E_WARPS), 32 * K4E_WARPS, 0, c->stream>>>(e);
    c->launches++;
    cudaEventRecord(ev[2], c->stream);
    TS_CUDA(c, cudaGetLastError());
    TS_CUDA(c, cudaMemcpyAsync(hs.data(), e.slew_time, NC * RR * 8, cudaMemcpyDeviceToHost, c->stream));
    if (x_final) TS_CUDA(c, cudaMemcpyAsync(hx.data(), e.x_final, NC * RR * 64, cudaMemcpyDeviceToHost, c->stream));
    TS_CUDA(c, cudaStreamSynchronize(c->stream));
    c->ens_ms[0] = ev.ms(0, 1);
    c->ens_ms[1] = ev.ms(1, 2);
    c->last_kernel_ms = c->ens_ms[0] + c->ens_ms[1];
  }
  // rows in the caller's order; a NO_CUTOFF trial gets NaN rows
  std::vector<char> done((size_t)n_sel, 0);
  for (size_t k = 0; k < NC; ++k) {
    const size_t p = (size_t)pos[k];
    done[p] = 1;
    memcpy(slew_time + p * RR, &hs[k * RR], RR * 8);
    if (x_final) memcpy(x_final + p * RR * 8, &hx[k * RR * 8], RR * 64);
  }
  for (int64_t p = 0; p < n_sel; ++p)
    if (!done[(size_t)p]) {
      for (size_t i = 0; i < RR; ++i) slew_time[(size_t)p * RR + i] = NAN;
      if (x_final)
        for (size_t i = 0; i < RR * 8; ++i) x_final[(size_t)p * RR * 8 + i] = NAN;
    }
  return TS_OK;
}

int ts_mc_replay_ensemble_last_split(ts_ctx* c, double* gains_ms, double* replay_ms) {
  if (!c) return TS_ERR_ARG;
  if (gains_ms) *gains_ms = c->ens_ms[0];
  if (replay_ms) *replay_ms = c->ens_ms[1];
  return TS_OK;
}

// ---------------------------------------------------------------------------- K5 element-wise ops
int ts_kep_eci_batch(ts_ctx* c, int64_t n, const double* kep6, const double* t0, double GM, double* rv6) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || (n > 0 && (!kep6 || !rv6))) return fail(c, TS_ERR_ARG, "ts_kep_eci_batch: null argument");
  if (n == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  Staging io(c, 0);
  const double* dk = io.in(kep6, (size_t)n * 6);
  const double* dt0 = io.in(t0, (size_t)n);
  double* dr = io.out(rv6, (size_t)n * 6);
  if (io.rc) return io.rc;
  io.start();
  k5_kep_eci<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(n, dk, dt0, GM, dr);
  c->launches++;
  return io.finish();
}

int ts_orbit_rhs_batch(ts_ctx* c, int64_t n, const double* x6, double* dx6) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || (n > 0 && (!x6 || !dx6))) return fail(c, TS_ERR_ARG, "ts_orbit_rhs_batch: null argument");
  if (n == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  Staging io(c, 0);
  const double* dx = io.in(x6, (size_t)n * 6);
  double* dd = io.out(dx6, (size_t)n * 6);
  if (io.rc) return io.rc;
  io.start();
  k5_orbit_rhs<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(n, dx, dd);
  c->launches++;
  return io.finish();
}

int ts_legendre_schmidt_batch(ts_ctx* c, int64_t n, const double* theta, int n_max, double* P, double* dP) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || (n > 0 && (!theta || !P))) return fail(c, TS_ERR_ARG, "ts_legendre_schmidt_batch: null argument");
  if (n_max < 1 || n_max > 13) return fail(c, TS_ERR_ARG, "n_max must be in [1, 13]");
  if (n == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  Staging io(c, 0);
  const size_t d2 = (size_t)(n_max + 1) * (n_max + 1);
  const double* dth = io.in(theta, (size_t)n);
  double* dPd = io.out(P, (size_t)n * d2);
  double* ddP = io.out(dP, (size_t)n * d2);
  if (io.rc) return io.rc;
  io.start();
  k5_legendre<<<(unsigned)((n + 63) / 64), 64, 0, c->stream>>>(n, dth, n_max, dPd, ddP);
  c->launches++;
  return io.finish();
}

int ts_dynamics_batch(ts_ctx* c, int mode, int64_t n, const double* x, const double* u, const double* B, int64_t B_rows,
                      double index_scale, double clock_rate, const double* Jmat, double* dx) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || mode < 0 || mode > 2 || (n > 0 && (!x || !u || !B || !Jmat || !dx))) return fail(c, TS_ERR_ARG, "ts_dynamics_batch: bad argument");
  if (mode != 2 && B_rows < 1) return fail(c, TS_ERR_ARG, "ts_dynamics_batch: empty field table");
  if (n == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  Staging io(c, 0);
  const int nx = (mode == 2) ? 7 : 8;
  const double* dxs = io.in(x, (size_t)n * nx);
  const double* du = io.in(u, (size_t)n * 3);
  const double* dB = io.in(B, (mode == 2) ? (size_t)n * 3 : (size_t)B_rows * 3);
  const double* dJ = io.in(Jmat, 9);
  double* dd = io.out(dx, (size_t)n * nx);
  if (io.rc) return io.rc;
  io.start();
  k5_dynamics<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(mode, n, dxs, du, dB, B_rows, index_scale, clock_rate, dJ, dd);
  c->launches++;
  return io.finish();
}

int ts_rk3_step_batch(ts_ctx* c, int64_t n, const double* x, const double* u, const double* B, int64_t B_rows, double index_scale,
                      double clock_rate, const double* Jmat, double dt, double* xn) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || B_rows < 1 || (n > 0 && (!x || !u || !B || !Jmat || !xn))) return fail(c, TS_ERR_ARG, "ts_rk3_step_batch: bad argument");
  if (n == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  Staging io(c, 0);
  const double* dxs = io.in(x, (size_t)n * 8);
  const double* du = io.in(u, (size_t)n * 3);
  const double* dB = io.in(B, (size_t)B_rows * 3);
  const double* dJ = io.in(Jmat, 9);
  double* dd = io.out(xn, (size_t)n * 8);
  if (io.rc) return io.rc;
  io.start();
  k5_rk3_step<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(n, dxs, du, dB, B_rows, index_scale, clock_rate, dJ, dt, dd);
  c->launches++;
  return io.finish();
}

// ---------------------------------------------------------------------------- K7 comparison controller
int ts_psiaki_pd_batch(ts_ctx* c, int64_t n_trials, const int64_t* N_i, const int64_t* offs, const double* x0, const double* w_guess,
                       const double* q_guess, const double* B_eci, const double* Jmat, double dt, double C_1, double C_2, double* X,
                       double* M, double* q_err) {
  if (!c) return TS_ERR_ARG;
  if (n_trials < 0 || (n_trials > 0 && (!N_i || !offs || !x0 || !w_guess || !q_guess || !B_eci || !Jmat || !X)))
    return fail(c, TS_ERR_ARG, "ts_psiaki_pd_batch: null argument");
  if (n_trials == 0) return TS_OK;
  if (!(dt > 0)) return fail(c, TS_ERR_ARG, "ts_psiaki_pd_batch: dt must be > 0");
  int64_t knots = 0;
  for (int64_t t = 0; t < n_trials; ++t) {
    if (N_i[t] < 1) return fail(c, TS_ERR_ARG, "trial %lld: N < 1", (long long)t);
    knots = std::max(knots, offs[t] + N_i[t]);
  }
  TS_CUDA(c, cudaSetDevice(c->device));
  Staging io(c, 0);
  K7Args a;
  a.n_trials = n_trials;
  a.N_i = io.in(N_i, (size_t)n_trials);
  a.offs = io.in(offs, (size_t)n_trials);
  a.x0 = io.in(x0, (size_t)n_trials * 7);
  a.w_guess = io.in(w_guess, (size_t)knots * 3);
  a.q_guess = io.in(q_guess, (size_t)knots * 4);
  a.B_eci = io.in(B_eci, (size_t)knots * 3);
  a.Jmat = io.in(Jmat, (size_t)n_trials * 9);
  a.dt = dt; a.C1 = C_1; a.C2 = C_2;
  a.X = io.out(X, (size_t)knots * 7);
  a.M = io.out(M, (size_t)knots * 3);
  a.Qe = io.out(q_err, (size_t)knots * 4);
  if (io.rc) return io.rc;
  io.start();
  k7_psiaki_pd_kernel<<<(unsigned)((n_trials + 63) / 64), 64, 0, c->stream>>>(a);
  c->launches++;
  return io.finish();
}

int ts_attitude_dynamics_linear_batch(ts_ctx* c, int64_t n, const double* x, const double* u, const double* x_linear, const double* B_B,
                                      const double* Jmat, double* dx) {
  if (!c) return TS_ERR_ARG;
  if (n < 0 || (n > 0 && (!x || !u || !x_linear || !B_B || !Jmat || !dx))) return fail(c, TS_ERR_ARG, "ts_attitude_dynamics_linear_batch: null argument");
  if (n == 0) return TS_OK;
  TS_CUDA(c, cudaSetDevice(c->device));
  Staging io(c, 0);
  const double* dxs = io.in(x, (size_t)n * 7);
  const double* du = io.in(u, (size_t)n * 3);
  const double* dl = io.in(x_linear, (size_t)n * 7);
  const double* dB = io.in(B_B, (size_t)n * 3);
  const double* dJ = io.in(Jmat, 9);
  double* dd = io.out(dx, (size_t)n * 7);
  if (io.rc) return io.rc;
  io.start();
  k7_attitude_dynamics_linear<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(n, dxs, du, dl, dB, dJ, dd);
  c->launches++;
  return io.finish();
}

}  // extern "C"

#include "multi.cuh"
