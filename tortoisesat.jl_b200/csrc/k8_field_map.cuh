// K8 -- the cubic B-spline interpolant of the igrf_data field map [src/magnetic_toolbox.jl:124-125]:
//   extrapolate(interpolate(A, BSpline(Cubic(Reflect(OnCell())))), Periodic())   (Interpolations v0.12.5)
// Rules FM1..FM4 are frozen in DESIGN.md section 4 (K8); the kernels below implement FM1 (prefilter), FM2 + FM3
// (evaluation with periodic wrap).  FM4 (integer component index, period 3) is a host-side rule: every evaluation
// returns all three components.
//
// Layouts: the data grid is n0 x n1 x 3 row-major (component fastest); the coefficients C are (n0+2) x (n1+2) x 3,
// padded by one coefficient on each side of both spatial axes (C[p][q] holds c_{p,q}, p = 0..n0+1, q = 0..n1+1).
#pragma once
#include "common.cuh"

namespace ts {

// largest axis length: keeps the transpose grid (one block row per 32 grid rows) inside gridDim.y <= 65535
constexpr int64_t K8_MAX_AXIS = 1 << 20;

// ---------------------------------------------------------------------------------------------------- prefilter
// FM1 on one axis of length m (6 x the system): rows 1 and m read [5 1], interior rows [1 4 1], right-hand side 6 a_k
// (c_0 = c_1 and c_{m+1} = c_m folded into the first and last row).  With the off-diagonal equal to 1 the Thomas
// factors reduce to one sequence inv_k = 1 / (b_k - inv_{k-1}) (inv_0 = 0), shared by every line of the axis:
//   forward  d_k = (6 a_k - d_{k-1}) inv_k,   back  c_m = d_m,  c_k = d_k - inv_k c_{k+1}.
inline void k8_thomas_factors(int64_t m, double* inv) {
  double prev = 0.0;
  for (int64_t k = 0; k < m; ++k) {
    const double b = (k == 0 || k == m - 1) ? 5.0 : 4.0;
    inv[k] = 1.0 / (b - prev);
    prev = inv[k];
  }
}

// In-place solve of w independent lines laid out as the columns of buf ((m+2) rows x w, row stride w): rows 1..m hold
// the data on entry; on exit rows 0..m+1 hold c_0..c_{m+1}.  One thread per column: consecutive threads touch
// consecutive doubles of every row, so both sweeps read and write coalesced.  The forward sweep parks d_k in row k,
// where the back sweep reads it.  Each sweep is one dependent FMA per row (6 a_k inv_k is off the chain).
__global__ void __launch_bounds__(128) k8_prefilter_cols(double* __restrict__ buf, int64_t m, int64_t w,
                                                         const double* __restrict__ inv) {
  const int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= w) return;
  double* p = buf + col;
  double d = 0.0;
  for (int64_t k = 0; k < m; ++k) {
    const double f = inv[k];
    d = fma(-d, f, 6.0 * f * p[(k + 1) * w]);
    p[(k + 1) * w] = d;
  }
  double x = d;  // c_m = d_m (already in row m)
  p[(m + 1) * w] = x;
  for (int64_t k = m - 2; k >= 0; --k) {
    x = fma(-inv[k], x, p[(k + 1) * w]);
    p[(k + 1) * w] = x;
  }
  p[0] = x;  // c_0 = c_1
}

// out[s][r][:] = in[r][s][:] for an R x S array of 3-vectors; out has row stride out_stride doubles.  32 x 32 tiles
// staged in shared memory: each warp reads and writes rows of 96 contiguous doubles.
constexpr int K8_TILE = 32;
__global__ void __launch_bounds__(256) k8_transpose3(const double* __restrict__ in, int64_t R, int64_t S, double* __restrict__ out,
                                                     int64_t out_stride) {
  __shared__ double tile[K8_TILE][3 * K8_TILE + 1];
  const int64_t r0 = (int64_t)blockIdx.y * K8_TILE, s0 = (int64_t)blockIdx.x * K8_TILE;
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int64_t ns = S - s0 < K8_TILE ? S - s0 : K8_TILE, nr = R - r0 < K8_TILE ? R - r0 : K8_TILE;
  for (int rl = ty; rl < nr; rl += blockDim.y) {
    const double* row = in + ((r0 + rl) * S + s0) * 3;
    for (int e = tx; e < 3 * ns; e += K8_TILE) tile[rl][e] = row[e];
  }
  __syncthreads();
  for (int sl = ty; sl < ns; sl += blockDim.y) {
    double* row = out + (s0 + sl) * out_stride + r0 * 3;
    for (int e = tx; e < 3 * nr; e += K8_TILE) row[e] = tile[e / 3][3 * sl + e % 3];
  }
}

// --------------------------------------------------------------------------------------------------- evaluation
// FM3: x <- mod(x - 1/2, n) + 1/2 (Julia's floored mod: fmod is exact, a negative remainder gets n added).
__device__ __forceinline__ double k8_wrap(double x, double n) {
  double r = fmod(x - 0.5, n);
  if (r < 0.0) r += n;
  return r + 0.5;
}

// FM2: segment k = clamp(floor(x), 1, n-1) (1-based), delta = x - k in [-1/2, 3/2], weights of C[k-1 .. k+2].
__device__ __forceinline__ int64_t k8_weights(double x, int64_t n, double w[4]) {
  double kf = floor(x);
  kf = kf < 1.0 ? 1.0 : (kf > (double)(n - 1) ? (double)(n - 1) : kf);
  const double d = x - kf, e = 1.0 - d;
  const double d2 = d * d, e2 = e * e;
  w[0] = e2 * e * (1.0 / 6.0);
  w[1] = 2.0 / 3.0 - d2 + 0.5 * d2 * d;
  w[2] = 2.0 / 3.0 - e2 + 0.5 * e2 * e;
  w[3] = d2 * d * (1.0 / 6.0);
  return (int64_t)kf;
}

// C with each 24-byte node padded to 32 bytes (fourth double 0), so that every tap is one aligned 256-bit load.
__global__ void __launch_bounds__(256) k8_pad4(const double* __restrict__ C3, int64_t nodes, double* __restrict__ C4) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nodes) return;
  C4[4 * i] = C3[3 * i];
  C4[4 * i + 1] = C3[3 * i + 1];
  C4[4 * i + 2] = C3[3 * i + 2];
  C4[4 * i + 3] = 0.0;
}

__device__ __forceinline__ void k8_ld256(const double* p, double& a, double& b, double& c) {
  double pad;
  asm("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(pad) : "l"(p));
}

// One point per thread: SoA indices in (1-based, any real), n x 3 row-major out.  16 taps per point, four rows of 128
// contiguous, 32-byte-aligned bytes of the padded C4 (one 256-bit load per tap: 16 load instructions per point instead
// of 48 scalar ones); C4 of a 1000^2 map is 32 MB and stays in L2 across the batch.
// A non-finite index gives NaN in all three components of its row and raises *bad_flag.
// ptxas (sm_100a, CUDA 12.9): 64 registers, 0 spill bytes, no local memory (launch bounds 256 x 4 = 32 warps per SM;
// 256 x 6 at 40 registers timed the same on a B200).  Measured against 48 scalar loads from the unpadded C: 6.61 ms
// instead of 8.40 ms for 10^8 points (tools/field_map_bench.py; the 32 MB copy is made inside the call).
constexpr int K8_THREADS = 256;
__global__ void __launch_bounds__(K8_THREADS, 4)
k8_field_map_eval(const double* __restrict__ C4, int64_t n0, int64_t n1, int64_t n, const double* __restrict__ x0,
                  const double* __restrict__ x1, double* __restrict__ out, int* __restrict__ bad_flag) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double a = x0[i], b = x1[i];
  double r0 = nan(""), r1 = r0, r2 = r0;
  if (isfinite(a) && isfinite(b)) {
    double w0[4], w1[4];
    const int64_t k0 = k8_weights(k8_wrap(a, (double)n0), n0, w0);
    const int64_t k1 = k8_weights(k8_wrap(b, (double)n1), n1, w1);
    const int64_t ld = (n1 + 2) * 4;
    // 1-based segment k -> taps at padded indices k-1 .. k+2
    const double* base = C4 + (k0 - 1) * ld + (k1 - 1) * 4;
    r0 = r1 = r2 = 0.0;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const double* row = base + m * ld;
      double s0 = 0.0, s1 = 0.0, s2 = 0.0;
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        double c0, c1, c2;
        k8_ld256(row + 4 * l, c0, c1, c2);
        s0 = fma(w1[l], c0, s0);
        s1 = fma(w1[l], c1, s1);
        s2 = fma(w1[l], c2, s2);
      }
      r0 = fma(w0[m], s0, r0);
      r1 = fma(w0[m], s1, r1);
      r2 = fma(w0[m], s2, r2);
    }
  } else {
    *bad_flag = 1;
  }
  out[3 * i] = r0;
  out[3 * i + 1] = r1;
  out[3 * i + 2] = r2;
}

}  // namespace ts
