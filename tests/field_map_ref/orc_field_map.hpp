// CPU restatement of the field-map interpolant (rules FM1..FM4 of DESIGN.md section 4, K8):
//   extrapolate(interpolate(A, BSpline(Cubic(Reflect(OnCell())))), Periodic())   [src/magnetic_toolbox.jl:124-125]
// Written from the rules, not from the kernels: FM1 solves the full (n+2)-row system, boundary rows included, with a
// textbook Thomas elimination; FM2 sums the 16 taps in the order the formula is written.  Compiled without FMA
// contraction (-ffp-contract=off), so the operation order below is what executes.
#pragma once
#include <cmath>
#include <cstdint>
#include <vector>

namespace orc_fm {

// FM1 on one line: data a[0..n-1] (a_1..a_n) at stride `sa`, coefficients c[0..n+1] (c_0..c_{n+1}) at stride `sc`.
//   row 0:      c_0 - c_1 = 0
//   row k:      c_{k-1}/6 + 2 c_k/3 + c_{k+1}/6 = a_k      (k = 1..n)
//   row n+1:    c_{n+1} - c_n = 0
inline void prefilter_line(int64_t n, const double* a, int64_t sa, double* c, int64_t sc) {
  const int64_t m = n + 2;
  std::vector<double> lo(m), di(m), up(m), rhs(m);
  lo[0] = 0.0, di[0] = 1.0, up[0] = -1.0, rhs[0] = 0.0;
  for (int64_t k = 1; k <= n; ++k) lo[k] = 1.0 / 6.0, di[k] = 2.0 / 3.0, up[k] = 1.0 / 6.0, rhs[k] = a[(k - 1) * sa];
  lo[m - 1] = -1.0, di[m - 1] = 1.0, up[m - 1] = 0.0, rhs[m - 1] = 0.0;
  std::vector<double> cp(m), dp(m);
  cp[0] = up[0] / di[0];
  dp[0] = rhs[0] / di[0];
  for (int64_t k = 1; k < m; ++k) {
    const double den = di[k] - lo[k] * cp[k - 1];
    cp[k] = up[k] / den;
    dp[k] = (rhs[k] - lo[k] * dp[k - 1]) / den;
  }
  c[(m - 1) * sc] = dp[m - 1];
  for (int64_t k = m - 2; k >= 0; --k) c[k * sc] = dp[k] - cp[k] * c[(k + 1) * sc];
}

// FM1 in 2-D: grid n0 x n1 x 3 -> C (n0+2) x (n1+2) x 3.  Axis 1 (j) for every data row, then axis 0 (i) for every one
// of the n1+2 resulting columns; each component on its own.
inline void prefilter(int64_t n0, int64_t n1, const double* grid, double* C) {
  const int64_t ld = (n1 + 2) * 3;
  std::vector<double> T((size_t)(n0 * ld));
  for (int64_t i = 0; i < n0; ++i)
    for (int c = 0; c < 3; ++c) prefilter_line(n1, grid + i * n1 * 3 + c, 3, T.data() + i * ld + c, 3);
  for (int64_t q = 0; q < n1 + 2; ++q)
    for (int c = 0; c < 3; ++c) prefilter_line(n0, T.data() + q * 3 + c, ld, C + q * 3 + c, ld);
}

// FM3: x <- mod(x - 1/2, n) + 1/2 with Julia's floored mod (mod(x, y) = r = rem(x, y); r + y when r and y differ in sign)
inline double wrap(double x, int64_t n) {
  const double y = (double)n;
  double r = std::fmod(x - 0.5, y);
  if (r != 0.0 && r < 0.0) r = r + y;
  return r + 0.5;
}

// FM2 weights of C[k-1], C[k], C[k+1], C[k+2] (1-based segment k = clamp(floor(x), 1, n-1), delta = x - k)
inline int64_t segment(double x, int64_t n, double w[4]) {
  int64_t k = (int64_t)std::floor(x);
  if (k < 1) k = 1;
  if (k > n - 1) k = n - 1;
  const double d = x - (double)k;
  w[0] = (1.0 - d) * (1.0 - d) * (1.0 - d) / 6.0;
  w[1] = 2.0 / 3.0 - d * d + d * d * d / 2.0;
  w[2] = 2.0 / 3.0 - (1.0 - d) * (1.0 - d) + (1.0 - d) * (1.0 - d) * (1.0 - d) / 2.0;
  w[3] = d * d * d / 6.0;
  return k;
}

// FM2 + FM3 at one point, all three components.  Returns false (and NaN) for a non-finite index.
inline bool eval(int64_t n0, int64_t n1, const double* C, double x0, double x1, double out[3]) {
  if (!std::isfinite(x0) || !std::isfinite(x1)) {
    out[0] = out[1] = out[2] = std::nan("");
    return false;
  }
  double w0[4], w1[4];
  const int64_t k0 = segment(wrap(x0, n0), n0, w0), k1 = segment(wrap(x1, n1), n1, w1);
  const int64_t ld = (n1 + 2) * 3;
  for (int c = 0; c < 3; ++c) {
    double s = 0.0;
    for (int m = -1; m <= 2; ++m)
      for (int l = -1; l <= 2; ++l) s += w0[m + 1] * w1[l + 1] * C[(k0 + m) * ld + (k1 + l) * 3 + c];
    out[c] = s;
  }
  return true;
}

// FM4: the component index must be an integer; it wraps with period 3 (1-based).  Returns false for a fractional c.
inline bool call(int64_t n0, int64_t n1, const double* C, double i, double j, double c, double* value) {
  if (!(std::floor(c) == c)) return false;
  double o[3];
  eval(n0, n1, C, i, j, o);
  int64_t k = ((int64_t)c - 1) % 3;
  if (k < 0) k += 3;
  *value = o[k];
  return true;
}

}  // namespace orc_fm
