"""The draws of a disturbance-ensemble realisation restated in numpy (rule RE2 of DESIGN.md section 4, K4), and the host
build of the K4 source's ensemble entry points (tests/hostsim/hostsim_ensemble.cpp), compiled with g++ on first use
into a temporary directory keyed by the source hash, so the tests write nothing into the tree."""
import ctypes as C
import os

import numpy as np

import alilqr_state as AS

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
MASK = np.uint64(0xFFFFFFFF)
PI = 3.14159265358979323846
S_W, S_Q, S_B = (.38 * PI / 180) * (.38 * PI / 180), (1 * PI / 180) * (1 * PI / 180), 1e-5 * 1e-5


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on uint32 counter words (arrays broadcast together) and a 2-word key."""
    c = [np.asarray(x, dtype=np.uint64) & MASK for x in (c0, c1, c2, c3)]
    c0, c1, c2, c3 = np.broadcast_arrays(*c)
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        n0 = (p1 >> np.uint64(32)) ^ c1 ^ k0
        n2 = (p0 >> np.uint64(32)) ^ c3 ^ k1
        c1, c3, c0, c2 = p1 & MASK, p0 & MASK, n0, n2
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & MASK, (k1 + np.uint64(0xBB67AE85)) & MASK
    return c0, c1, c2, c3


def u01(x):
    return (np.asarray(x, dtype=np.float64) + 0.5) * (1.0 / 4294967296.0)


def box_muller(a, b):
    rad = np.sqrt(-2.0 * np.log(u01(a)))
    ang = 2.0 * PI * u01(b)
    return rad * np.cos(ang), rad * np.sin(ang)


def tvlqr_noise(seed, stream, step, stage, r):
    """(..., 9) stage draws of realisation r: counter (stream, step, stage, block + 4r), key = seed."""
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    b = 4 * int(r)
    r0 = philox4x32_10(stream, step, stage, b, k0, k1)
    r1 = philox4x32_10(stream, step, stage, b + 1, k0, k1)
    r2 = philox4x32_10(stream, step, stage, b + 2, k0, k1)
    n0, n1 = box_muller(r0[0], r0[1])
    n2, n3 = box_muller(r0[2], r0[3])
    n4, n5 = box_muller(r1[0], r1[1])
    return np.stack([n0 * S_W, n1 * S_W, n2 * S_W, n3 * S_Q, n4 * S_Q, n5 * S_Q, u01(r1[2]) * S_B, u01(r1[3]) * S_B,
                     u01(r2[0]) * S_B], axis=-1)


def initial_qnoise(seed, stream, r, scale):
    """q_noise of realisation r >= 1: counter (stream, 0xFFFFFFFF, 0, 4r)."""
    o = philox4x32_10(stream, 0xFFFFFFFF, 0, 4 * int(r), seed & 0xFFFFFFFF, seed >> 32)
    z0, z1 = box_muller(o[0], o[1])
    z2, _ = box_muller(o[2], o[3])
    return scale * np.array([float(z0), float(z1), float(z2)])


def qmult(a, b):
    s1, v1, s2, v2 = a[0], np.asarray(a[1:]), b[0], np.asarray(b[1:])
    return np.concatenate([[s1 * s2 - v1 @ v2], s1 * v2 + s2 * v1 + np.cross(v1, v2)])


def x0_lqr(x0, qn):
    """ts_monte_carlo_run's x0_lqr: omega from x0, attitude rotated by q_noise (zero row: none), clock 0."""
    x = np.array(x0, dtype=float).copy()
    th = float(np.linalg.norm(qn))
    if th > 1e-300:
        x[3:7] = qmult(x[3:7], np.concatenate([[np.cos(th / 2)], np.asarray(qn) / th * np.sin(th / 2)]))
    x[7] = 0.0
    return x


def noise_array(seed, stream, N, r):
    """The explicit (N, 4, 9) noise array (mode 1 layout; the last step unused) that realisation r draws."""
    k = np.arange(N)[:, None]
    s = np.arange(4)[None, :]
    return tvlqr_noise(seed, stream, k, s, r)


def hostsim_ensemble():
    d = os.path.join(HERE, "hostsim")
    csrc = os.path.join(ROOT, "tortoisesat.jl_b200", "csrc")
    deps = [os.path.join(csrc, f) for f in ("ilqr_solver.cuh", "ilqr_math.cuh", "tvlqr_solver.cuh", "philox.cuh")]
    L = AS._build("hostsim_ensemble", os.path.join(d, "hostsim_ensemble.cpp"), deps, ["-O2", "-std=c++20"])
    L.hse_tvlqr_noise.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
    L.hse_initial_qnoise.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_double, C.c_void_p]
    L.hse_x0_lqr.argtypes = [C.c_void_p] * 3
    L.hse_tvlqr_real.argtypes = [C.c_int64] + [C.c_void_p] * 5 + [C.c_int64, C.c_double, C.c_double, C.c_double, C.c_void_p,
                                                                  C.c_uint32, C.c_uint32] + [C.c_void_p] * 5
    L.hse_tvlqr_real.restype = C.c_int64
    return L
