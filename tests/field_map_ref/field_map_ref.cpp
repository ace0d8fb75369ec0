// C entry points of the CPU field-map restatement (orc_field_map.hpp), loaded by tests/field_map_oracle.py.
#include "orc_field_map.hpp"

extern "C" {

void orc_field_map_prefilter(int64_t n0, int64_t n1, const double* grid, double* coefs) {
  orc_fm::prefilter(n0, n1, grid, coefs);
}

// returns the number of points with a non-finite index (their rows are NaN)
int64_t orc_field_map_eval(int64_t n0, int64_t n1, const double* coefs, int64_t n, const double* x0, const double* x1, double* out) {
  int64_t bad = 0;
  for (int64_t p = 0; p < n; ++p) bad += orc_fm::eval(n0, n1, coefs, x0[p], x1[p], out + 3 * p) ? 0 : 1;
  return bad;
}

// returns 0, or -2 for a fractional component index
int orc_field_map_call(int64_t n0, int64_t n1, const double* coefs, double i, double j, double c, double* value) {
  return orc_fm::call(n0, n1, coefs, i, j, c, value) ? 0 : -2;
}
}
