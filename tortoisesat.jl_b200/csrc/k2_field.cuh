// K2 -- per-trial orbit propagation, ECI field table, magnetic gramian and
// condition-number cutoff.  Replaces, batched over trials,
//   kep_ECI(kep,t0,GM)                         reference src/kep_ECI.jl:1-49
//   OrbitPlotter + solve(Euler(), dt)          src/OrbitPlotter.jl:1-52, src/magnetic_toolbox.jl:51-56
//   magnetic_simulation(p,t0,tf,N,mag_field)   src/magnetic_toolbox.jl:33-106
//   magnetic_gramian(B_N,dt)                   src/magnetic_toolbox.jl:1-12
//   condition_based_time(B_gram,cutoff)        src/magnetic_toolbox.jl:14-31
//
// Kernels:
//   k2a_orbit_euler   one thread per trial, strictly sequential explicit Euler (2N steps, ~45 instructions each:
//                     orbit_rhs_fast), positions/velocities streamed to HBM;
//   k2b_field_rows    one thread per (trial, sample): GMST -> ECEF -> lat/long ->
//                     IGRF-12 (igrf_device.cuh, coefficients of the trial's date
//                     staged in shared memory per block) -> NED->ENU->ECEF->ECI;
//   k2c_cutoff_scan   one block per trial: block-wide prefix scan of the gramian terms, cond() of every prefix in
//                     parallel, first sample below the cutoff by ballot (the fused Monte-Carlo path: two sample ranges,
//                     the second one only for the orbits that did not reach the cutoff in the first);
//   k2c_gramian_cutoff one thread per trial: running gramian in the reference's summation order + 3x3 symmetric Jacobi
//                     eigenvalues (the stand-alone magnetic_gramian / condition_based_time entry points).
// Roofline: k2b is FP64-pipe bound (IGRF, ~2.4 kFLOP/sample, 48 B/sample); k2a is a latency-bound sequential chain.
// Measured on the 8192-orbit sweep (round 2): field stage 80 ms -> 15.7 ms (10.1 ms for 4096 orbits).
#pragma once
#include "common.cuh"
#include "igrf_device.cuh"

// Per-trial options of the field pass (mirrors the reference's globals p.GM, p.MJD, alt, R_E).
struct ts_field_opts_dev {
  double GM, mjd, igrf_date, field_radius_m, t0, tf;
  int64_t N;
};

namespace ts {

// Julia sind/cosd: exact argument reduction in degrees (cosd(90) == 0).
__device__ __forceinline__ double sind_dev(double x) {
  const double rx = copysign(fmod(x, 360.0), x);
  const double arx = fabs(rx);
  if (rx == 0.0) return rx;
  if (arx < 45.0) return sinpi(rx / 180.0);
  if (arx <= 135.0) return copysign(cospi((90.0 - arx) / 180.0), rx);
  if (arx == 180.0) return copysign(0.0, rx);
  if (arx < 225.0) return sinpi(((180.0 - arx) * (rx < 0 ? -1.0 : 1.0)) / 180.0);
  if (arx <= 315.0) return -copysign(cospi((270.0 - arx) / 180.0), rx);
  return sinpi((rx - copysign(360.0, rx)) / 180.0);
}
__device__ __forceinline__ double cosd_dev(double x) {
  const double rx = fabs(fmod(x, 360.0));
  if (rx <= 45.0) return cospi(rx / 180.0);
  if (rx < 135.0) return sinpi((90.0 - rx) / 180.0);
  if (rx <= 225.0) return -cospi((180.0 - rx) / 180.0);
  if (rx < 315.0) return sinpi((rx - 270.0) / 180.0);
  return cospi((360.0 - rx) / 180.0);
}

__device__ __forceinline__ void mat3_mul(const double A[9], const double B[9], double C[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) C[i * 3 + j] = A[i * 3 + 0] * B[0 * 3 + j] + A[i * 3 + 1] * B[1 * 3 + j] + A[i * 3 + 2] * B[2 * 3 + j];
}
__device__ __forceinline__ void mat3_vec(const double A[9], const double v[3], double o[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) o[i] = A[i * 3 + 0] * v[0] + A[i * 3 + 1] * v[1] + A[i * 3 + 2] * v[2];
}

// kep_ECI.jl:1-35 (the reference mutates kep[6]; the batch API leaves inputs untouched)
__device__ inline void kep_eci_dev(const double* kep, double t0, double GM, double u[6]) {
  const double PI = 3.141592653589793;
  const double e = kep[0], a = kep[1];
  const double M = fmod(kep[5] + t0 * sqrt(GM / (a * a * a)), 360.0);
  double E = M / 180 * PI;
  for (int i = 0; i < 100; ++i) E = E - (E - e * sin(E) - M / 180 * PI) / (1 - e * cos(E));
  const double nu = 2 * (atan2(sqrt(1 + e) * sin(E / 2), sqrt(1 - e) * cos(E / 2)) * (180.0 / PI));
  const double r_c = a * (1 - e * cos(E));
  const double o[3] = {r_c * cosd_dev(nu), r_c * sind_dev(nu), r_c * 0.0};
  const double f = sqrt(GM * a) / r_c;
  const double od[3] = {f * -sin(E), f * (sqrt(1 - e * e) * cos(E)), f * 0.0};
  const double an = -kep[3], ai = -kep[2], aw = -kep[4];
  const double Rz1[9] = {cosd_dev(an), sind_dev(an), 0, -sind_dev(an), cosd_dev(an), 0, 0, 0, 1};
  const double Rx[9] = {1, 0, 0, 0, cosd_dev(ai), sind_dev(ai), 0, -sind_dev(ai), cosd_dev(ai)};
  const double Rz2[9] = {cosd_dev(aw), sind_dev(aw), 0, -sind_dev(aw), cosd_dev(aw), 0, 0, 0, 1};
  double T[9], R[9];
  mat3_mul(Rz1, Rx, T);
  mat3_mul(T, Rz2, R);
  mat3_vec(R, o, u);
  mat3_vec(R, od, u + 3);
}

// OrbitPlotter.jl:1-52: two-body + the literal "J2" expression (:40-42, 6*r[3] not squared)
__device__ __forceinline__ void orbit_rhs_dev(const double x[6], double dx[6]) {
  const double GM = 3.986004418E14 * ((1.0 / 1000) * (1.0 / 1000) * (1.0 / 1000));
  const double nr = sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
  const double J2 = 0.0010826359;
  const double nr2 = nr * nr, nr7 = nr2 * nr2 * nr2 * nr;  // |r|^7 (the term is ~1e-19 km/s^2)
  const double rxy = x[0] * x[0] + x[1] * x[1];
  const double g = GM / nr2;
  const double c01 = 6 * x[2] - 1.5 * rxy, c2 = 3 * x[2] - 4.5 * rxy;
  dx[0] = x[3];
  dx[1] = x[4];
  dx[2] = x[5];
  dx[3] = (g * -x[0] / nr) + J2 * x[0] / nr7 * c01;
  dx[4] = (g * -x[1] / nr) + J2 * x[1] / nr7 * c01;
  dx[5] = (g * -x[2] / nr) + J2 * x[2] / nr7 * c2;
}

// The same right-hand side for the sequential Euler integration of k2a (up to 47 000 dependent steps per orbit): one
// reciprocal square root (hardware seed + one third-order step) and products instead of a square root and seven
// divisions -- ~45 instead of ~235 instructions per step.  Each quotient of the literal form above is reproduced to
// <= 1 ulp; positions after 10^4 steps agree with the oracle to < 1e-13 relative (tests: 1e-12).
__device__ __forceinline__ void orbit_rhs_fast(const double x[6], double dx[6]) {
  const double GM = 3.986004418E14 * ((1.0 / 1000) * (1.0 / 1000) * (1.0 / 1000));
  const double J2 = 0.0010826359;
  const double s = x[0] * x[0] + x[1] * x[1] + x[2] * x[2];
  double y0;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(s));
  const double e = fma(-s, y0 * y0, 1.0);
  const double inv = fma(fma(e, 0.375, 0.5), e * y0, y0);   // 1 / |r|
  const double inv2 = inv * inv, inv3 = inv2 * inv, inv7 = inv3 * inv2 * inv2;
  const double rxy = x[0] * x[0] + x[1] * x[1];
  const double c01 = 6 * x[2] - 1.5 * rxy, c2 = 3 * x[2] - 4.5 * rxy;
  const double a = -(GM * inv3), j = J2 * inv7;
  dx[0] = x[3];
  dx[1] = x[4];
  dx[2] = x[5];
  dx[3] = a * x[0] + (j * x[0]) * c01;
  dx[4] = a * x[1] + (j * x[1]) * c01;
  dx[5] = a * x[2] + (j * x[2]) * c2;
}

// pos/vel: per trial (2N+1) x 3 rows starting at row B_offs[t] + t.  vel may be null.
__global__ void __launch_bounds__(128)
k2a_orbit_euler(int64_t n_trials, const double* __restrict__ kep6, const ts_field_opts_dev* __restrict__ opts,
                const int64_t* __restrict__ B_offs, const int64_t* __restrict__ rows_limit, double* __restrict__ pos,
                double* __restrict__ vel) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_trials) return;
  const ts_field_opts_dev o = opts[t];
  double u[6];
  kep_eci_dev(kep6 + t * 6, o.t0, o.GM, u);
  const double dt = (o.tf - o.t0) / (double)o.N;
  int64_t steps = 2 * o.N;
  if (rows_limit && rows_limit[t] > 0 && rows_limit[t] < steps) steps = rows_limit[t];
  double* p = pos + (B_offs[t] + t) * 3;
  double* v = vel ? vel + (B_offs[t] + t) * 3 : nullptr;
  for (int64_t i = 0; i <= steps; ++i) {
    p[i * 3 + 0] = u[0];
    p[i * 3 + 1] = u[1];
    p[i * 3 + 2] = u[2];
    if (v) {
      v[i * 3 + 0] = u[3];
      v[i * 3 + 1] = u[4];
      v[i * 3 + 2] = u[5];
    }
    double du[6];
    orbit_rhs_fast(u, du);
#pragma unroll
    for (int c = 0; c < 6; ++c) u[c] = u[c] + dt * du[c];
  }
}

constexpr int K2B_THREADS = 128;

// grid.x = trial, grid.y = chunk of K2B_THREADS samples.  Rows >= 2N-1 (and rows
// beyond rows_limit) are zero-filled, like the reference's untouched last row.
template <int NMAX>
__global__ void __launch_bounds__(K2B_THREADS)
k2b_field_rows(const double* __restrict__ tabG, const double* __restrict__ tabH, const ts_field_opts_dev* __restrict__ opts,
               const int64_t* __restrict__ B_offs, const int64_t* __restrict__ rows_limit, const double* __restrict__ pos,
               double* __restrict__ B_eci, int nmax_select, int64_t i_lo = 0, const int64_t* __restrict__ skip_found = nullptr) {
  __shared__ double2 s_gh[2 * IGRF_NCOEF];
  const int64_t t = blockIdx.x;
  if (skip_found && skip_found[t] != 0) return;   // scoping pass, later sample ranges: this orbit already has its cutoff
  const ts_field_opts_dev o = opts[t];
  if (igrf_nmax_for_date(o.igrf_date) != nmax_select) return;  // handled by the other instantiation
  const int64_t rows = 2 * o.N;
  int64_t live = rows - 1;
  if (rows_limit && rows_limit[t] > 0 && rows_limit[t] < live) live = rows_limit[t];
  const int64_t i0 = i_lo + (int64_t)blockIdx.y * K2B_THREADS;
  if (i0 >= rows) return;
  igrf_stage_coeffs(s_gh, tabG, tabH, o.igrf_date);
  __syncthreads();
  const int64_t i = i0 + threadIdx.x;
  if (i >= rows) return;
  double* out = B_eci + (B_offs[t] + i) * 3;
  if (i >= live) {
    out[0] = out[1] = out[2] = 0.0;
    return;
  }
  const double PI = 3.141592653589793;
  const double dt = (o.tf - o.t0) / (double)o.N;
  // t_i = t0 + i*dt ; GMST in the reference's literal operation order (quirk Q5), no FMA
  const double ti = __dadd_rn(o.t0, __dmul_rn((double)i, dt));
  double g = __ddiv_rn(__ddiv_rn(__ddiv_rn(ti, 24.0), 60.0), 60.0);
  g = __dadd_rn(g, o.mjd);
  g = __dmul_rn(360.9856473, g);
  g = __dadd_rn(280.4606, g);
  g = __dsub_rn(g, 51544.5);
  g = __ddiv_rn(g, 180.0);
  const double GMST = __dmul_rn(g, PI);
  double sg, cg;
  sincos(GMST, &sg, &cg);
  const double* p = pos + (B_offs[t] + t + i) * 3;
  const double ROT[9] = {cg, sg, 0, -sg, cg, 0, 0, 0, 1};
  const double pv[3] = {p[0], p[1], p[2]};
  double pe[3];
  mat3_vec(ROT, pv, pe);
  const double lat = asin(pe[2] / sqrt(pe[0] * pe[0] + pe[1] * pe[1] + pe[2] * pe[2]));
  const double lon = atan2(pe[1], pe[0]);
  double bn, be, bd;
  igrf12_point<NMAX>(s_gh, o.field_radius_m, lat, lon, bn, be, bd);
  const double b[3] = {bn / 1.e9, be / 1.e9, bd / 1.e9};
  double slo, clo, sla, cla;
  sincos(lon, &slo, &clo);
  sincos(lat, &sla, &cla);
  const double RT[9] = {cg, -sg, 0, sg, cg, 0, 0, 0, 1};  // Rz(GMST)'
  const double RE[9] = {-slo, -sla * clo, cla * clo, clo, -sla * slo, cla * slo, 0, cla, sla};
  double M1[9];
  mat3_mul(RT, RE, M1);
  // (.)*NED_to_ENU = [0 1 0;1 0 0;0 0 -1]: swap columns 0/1, negate column 2
  const double M2[9] = {M1[1], M1[0], -M1[2], M1[4], M1[3], -M1[5], M1[7], M1[6], -M1[8]};
  double r3[3];
  mat3_vec(M2, b, r3);
  out[0] = r3[0];
  out[1] = r3[1];
  out[2] = r3[2];
}

// |eig| ratio of a symmetric 3x3 (cyclic Jacobi) == Julia cond() of the gramian.
__device__ inline double cond_sym3_dev(const double Gs[6] /*xx,xy,xz,yy,yz,zz*/) {
  double A[3][3] = {{Gs[0], Gs[1], Gs[2]}, {Gs[1], Gs[3], Gs[4]}, {Gs[2], Gs[4], Gs[5]}};
  for (int sweep = 0; sweep < 30; ++sweep) {
    const double off = A[0][1] * A[0][1] + A[0][2] * A[0][2] + A[1][2] * A[1][2];
    const double dia = A[0][0] * A[0][0] + A[1][1] * A[1][1] + A[2][2] * A[2][2];
    if (off <= 1e-36 * dia || off == 0.0) break;
#pragma unroll
    for (int p = 0; p < 2; ++p)
#pragma unroll
      for (int q = p + 1; q < 3; ++q) {
        if (A[p][q] == 0.0) continue;
        const double th = (A[q][q] - A[p][p]) / (2 * A[p][q]);
        const double tt = (th >= 0 ? 1.0 : -1.0) / (fabs(th) + sqrt(th * th + 1));
        const double c = 1 / sqrt(tt * tt + 1), s = tt * c;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double akp = A[k][p], akq = A[k][q];
          A[k][p] = c * akp - s * akq;
          A[k][q] = s * akp + c * akq;
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const double apk = A[p][k], aqk = A[q][k];
          A[p][k] = c * apk - s * aqk;
          A[q][k] = s * apk + c * aqk;
        }
      }
  }
  const double e0 = fabs(A[0][0]), e1 = fabs(A[1][1]), e2 = fabs(A[2][2]);
  const double mx = fmax(e0, fmax(e1, e2)), mn = fmin(e0, fmin(e1, e2));
  if (mn == 0.0) return INFINITY;
  return mx / mn;
}

__device__ __forceinline__ void hat_hatT_dev(const double* b, double h[6]) {
  // hat(b)*hat(b)' = |b|^2 I - b b', written as the reference's matrix product (row i . row j of hat)
  const double x = b[0], y = b[1], z = b[2];
  h[0] = (-z) * (-z) + y * y;      // (0,0)
  h[1] = y * (-x);                 // (0,1): 0*z + (-z)*0 + y*(-x)
  h[2] = (-z) * x;                 // (0,2)
  h[3] = z * z + (-x) * (-x);      // (1,1)
  h[4] = z * (-y);                 // (1,2): z*(-y) + 0 + (-x)*0
  h[5] = (-y) * (-y) + x * x;      // (2,2)
}

// One thread per trial.  Optional G output (rows x 9 per trial at B_offs[t]*3 doubles... see host).
__global__ void __launch_bounds__(128)
k2c_gramian_cutoff(int64_t n_trials, const double* __restrict__ B_eci, const int64_t* __restrict__ B_offs,
                   const int64_t* __restrict__ rows, const double* __restrict__ dts, const double* __restrict__ cutoffs,
                   double* __restrict__ G_out, int64_t* __restrict__ tf_index) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_trials) return;
  const double* B = B_eci + B_offs[t] * 3;
  const int64_t R = rows[t];
  const double dt = dts[t];
  const double cutoff = cutoffs ? cutoffs[t] : -1.0;
  double acc[6], h[6];
  int64_t found = 0;
  for (int64_t i = 0; i < R; ++i) {
    hat_hatT_dev(B + i * 3, h);
    if (i == 0) {
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[k] = h[k];  // first term has no dt (quirk Q9)
    } else {
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[k] = acc[k] + h[k] * dt;
    }
    if (G_out) {
      double* g = G_out + (B_offs[t] + i) * 9;
      g[0] = acc[0]; g[1] = acc[1]; g[2] = acc[2];
      g[3] = acc[1]; g[4] = acc[3]; g[5] = acc[4];
      g[6] = acc[2]; g[7] = acc[4]; g[8] = acc[5];
    }
    if (cutoff >= 0 && !found) {
      if (cond_sym3_dev(acc) < cutoff) {
        found = i + 1;
        if (!G_out) break;
      }
    }
  }
  if (tf_index) tf_index[t] = found;
}

// The cutoff search of the fused Monte-Carlo path, one BLOCK per orbit (k2c_gramian_cutoff above walks the samples with
// one thread per orbit: up to 10^4 dependent Jacobi eigen-solves, 34 ms for an 8192-orbit sweep).  Samples [i_lo, i_hi)
// in chunks of one per thread: h_i*dt -> block-wide inclusive scan of the six gramian entries (+ the carry of the
// previous chunks / of an earlier call, `carry` 6 doubles per orbit) -> cond() of every prefix in parallel -> the first
// sample below the cutoff by ballot.  The prefix sums are formed pairwise instead of left to right, i.e. they differ from
// the sequential gramian in the last bits (relative 1e-16) -- far below the ~1e-4 by which cond() moves per sample, so
// the index is the same (tests/test_gpu_scoping.py: hits on chunk and range edges, the benchmark sweep's second-range
// orbits).  tf_index[t] != 0 on entry: nothing to do.
constexpr int K2C_THREADS = 128;
__global__ void __launch_bounds__(K2C_THREADS)
k2c_cutoff_scan(const double* __restrict__ B_eci, const int64_t* __restrict__ B_offs, const int64_t* __restrict__ rows,
                const double* __restrict__ dts, const double* __restrict__ cutoffs, int64_t i_lo, int64_t i_hi,
                double* __restrict__ carry, int64_t* __restrict__ tf_index) {
  __shared__ double s_tot[K2C_THREADS / 32][6];
  __shared__ int s_first[K2C_THREADS / 32];
  const int64_t t = blockIdx.x;
  if (tf_index[t] != 0) return;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const double* B = B_eci + B_offs[t] * 3;
  int64_t R = rows[t];
  if (R > i_hi) R = i_hi;
  const double dt = dts[t], cutoff = cutoffs[t];
  double car[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) car[k] = (i_lo > 0) ? carry[t * 6 + k] : 0.0;
  for (int64_t base = i_lo; base < R; base += K2C_THREADS) {
    const int64_t i = base + tid;
    double v[6];
    if (i < R) {
      hat_hatT_dev(B + i * 3, v);
      if (i != 0) {   // the first term has no dt (quirk Q9)
#pragma unroll
        for (int k = 0; k < 6; ++k) v[k] = v[k] * dt;
      }
    } else {
#pragma unroll
      for (int k = 0; k < 6; ++k) v[k] = 0.0;
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {   // inclusive scan inside the warp
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double u = __shfl_up_sync(0xffffffffu, v[k], o);
        if (lane >= o) v[k] += u;
      }
    }
    if (lane == 31) {
#pragma unroll
      for (int k = 0; k < 6; ++k) s_tot[wid][k] = v[k];
    }
    __syncthreads();
    double acc[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      double pre = car[k];
      for (int w = 0; w < wid; ++w) pre += s_tot[w][k];
      acc[k] = pre + v[k];
    }
    const bool hit = (i < R) && (cond_sym3_dev(acc) < cutoff);
    const unsigned bal = __ballot_sync(0xffffffffu, hit);
    if (lane == 0) s_first[wid] = bal ? (wid * 32 + __ffs(bal) - 1) : K2C_THREADS;
#pragma unroll
    for (int k = 0; k < 6; ++k) {   // carry for the next chunk: everything up to the block's last sample
      double tot = car[k];
      for (int w = 0; w < K2C_THREADS / 32; ++w) tot += s_tot[w][k];
      car[k] = tot;
    }
    __syncthreads();
    int first = K2C_THREADS;
    for (int w = 0; w < K2C_THREADS / 32; ++w) first = min(first, s_first[w]);
    if (first < K2C_THREADS) {
      if (tid == 0) tf_index[t] = base + first + 1;
      return;
    }
    __syncthreads();   // s_tot / s_first are rewritten by the next chunk
  }
  if (tid == 0) {
#pragma unroll
    for (int k = 0; k < 6; ++k) carry[t * 6 + k] = car[k];
  }
}

// condition_based_time on caller-supplied gramians (rows x 9 per trial).
__global__ void __launch_bounds__(128)
k2d_condition_time(int64_t n_trials, const double* __restrict__ G, const int64_t* __restrict__ offs, const int64_t* __restrict__ rows,
                   const double* __restrict__ cutoffs, int64_t* __restrict__ tf_index) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_trials) return;
  int64_t found = 0;
  for (int64_t i = 0; i < rows[t]; ++i) {
    const double* g = G + (offs[t] + i) * 9;
    const double s[6] = {0.5 * (g[0] + g[0]), 0.5 * (g[1] + g[3]), 0.5 * (g[2] + g[6]), 0.5 * (g[4] + g[4]), 0.5 * (g[5] + g[7]),
                         0.5 * (g[8] + g[8])};
    if (cond_sym3_dev(s) < cutoffs[t]) {
      found = i + 1;
      break;
    }
  }
  tf_index[t] = found;
}

}  // namespace ts
