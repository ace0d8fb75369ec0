// Philox4x32-10 counter-based generator (Salmon, Moraes, Dror, Shaw, SC'11) and the
// noise layout of the TVLQR replay.  The reference draws randn/rand from Julia's
// MersenneTwister inside every dynamics call (src/simulator.jl:5,10,22); that stream
// cannot be reproduced outside Julia, so the engine freezes a counter-based one:
// counter = (trial, step, stage, block), key = seed.  Any trial is reproducible from
// (seed, trial) on any GPU, independent of sharding.
#pragma once
#include <math.h>
#include <stdint.h>

#include "ilqr_math.cuh"

namespace ts {

TS_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0;
  out[1] = c1;
  out[2] = c2;
  out[3] = c3;
}

TS_HD double u01_from_u32(uint32_t x) { return ((double)x + 0.5) * (1.0 / 4294967296.0); }

TS_HD void box_muller(uint32_t a, uint32_t b, double& z0, double& z1) {
  const double rad = sqrt(-2.0 * log(u01_from_u32(a)));
  const double ang = 2.0 * 3.14159265358979323846 * u01_from_u32(b);
  z0 = rad * cos(ang);
  z1 = rad * sin(ang);
}

// a product rounded on its own: the caller may add it to something, and nvcc must not contract the two into one FMA
TS_HD double mul_rn(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}

// 9 scaled perturbations of one simulator() call:
//  [0:3) randn(3)*(.38*pi/180)^2 (simulator.jl:5), [3:6) randn(3)*(pi/180)^2 (:10), [6:9) rand(3)*(1e-5)^2 (:22)
// Realisation `real` of a disturbance ensemble (ts_mc_replay_ensemble, RE2) draws counter blocks 4 real + {0, 1, 2};
// realisation 0 is the stream every single replay draws.  The rate and attitude products are rounded before they are
// used: K4n stores them to memory and the replay adds them to omega later, so a replay that draws inline (K4e) must not
// let them fuse into that addition (RE3).
TS_HD void tvlqr_noise(uint64_t seed, uint32_t trial, uint32_t step, uint32_t stage, double out[9], uint32_t real = 0) {
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const uint32_t b = 4u * real;
  uint32_t r0[4], r1[4], r2[4];
  philox4x32_10(trial, step, stage, b, k0, k1, r0);
  philox4x32_10(trial, step, stage, b + 1u, k0, k1, r1);
  philox4x32_10(trial, step, stage, b + 2u, k0, k1, r2);
  double n[6];
  box_muller(r0[0], r0[1], n[0], n[1]);
  box_muller(r0[2], r0[3], n[2], n[3]);
  box_muller(r1[0], r1[1], n[4], n[5]);
  const double PI = 3.14159265358979323846;
  const double s_w = (.38 * PI / 180) * (.38 * PI / 180);
  const double s_q = (1 * PI / 180) * (1 * PI / 180);
  const double s_b = (1E-5) * (1E-5);
  for (int i = 0; i < 3; ++i) out[i] = mul_rn(n[i], s_w);
  for (int i = 0; i < 3; ++i) out[3 + i] = mul_rn(n[3 + i], s_q);
  out[6] = u01_from_u32(r1[2]) * s_b;
  out[7] = u01_from_u32(r1[3]) * s_b;
  out[8] = u01_from_u32(r2[0]) * s_b;
}

// The initial attitude perturbation of realisation real >= 1 of a disturbance ensemble (RE2): step word 0xFFFFFFFF (no
// replay step reaches it), counter block 4 real; q_noise = scale * (z0, z1, z2) with (z0, z1) = box_muller(o0, o1) and
// z2 the first of box_muller(o2, o3).
TS_HD void tvlqr_initial_qnoise(uint64_t seed, uint32_t trial, uint32_t real, double scale, double qn[3]) {
  uint32_t o[4];
  philox4x32_10(trial, 0xFFFFFFFFu, 0u, 4u * real, (uint32_t)seed, (uint32_t)(seed >> 32), o);
  double z0, z1, z2, z3;
  box_muller(o[0], o[1], z0, z1);
  box_muller(o[2], o[3], z2, z3);
  qn[0] = scale * z0;
  qn[1] = scale * z1;
  qn[2] = scale * z2;
}

}  // namespace ts
