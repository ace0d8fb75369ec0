"""The truth-model parameters of a dispersion-ensemble realisation restated in numpy (rule DE2 of DESIGN.md section 4,
K4), the host build of the K4 source's dispersion entry points (tests/hostsim/hostsim_dispersion.cpp) and the oracle's
truth-model replay (tests/dispersion_ref/dispersion_ref.cpp), both compiled with g++ on first use into a temporary
directory keyed by the source hash, so the tests write nothing into the tree."""
import ctypes as C
import os

import numpy as np

import alilqr_state as AS
import replay_ensemble_ref as RE
from oracle import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def dispersion_params(seed, stream, r, sigmas):
    """The ten parameters d0 d1 d2 g0 g1 g2 s_B phi0 phi1 phi2 of realisation r for sigmas = (sigma_inertia,
    sigma_torquer, sigma_field_scale, sigma_field_angle): normals z0..z9 from counters (stream, 0xFFFFFFFE, 0, 4r + b),
    b = 0, 1, 2, key = seed."""
    p = np.array([1.0] * 7 + [0.0] * 3)
    if r == 0:
        return p
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    o = [[int(v) for v in RE.philox4x32_10(stream, 0xFFFFFFFE, 0, 4 * int(r) + b, k0, k1)] for b in range(3)]
    z = []
    for a, b in ((o[0][0], o[0][1]), (o[0][2], o[0][3]), (o[1][0], o[1][1]), (o[1][2], o[1][3]), (o[2][0], o[2][1])):
        z += [float(v) for v in RE.box_muller(a, b)]
    si, st, ss, sa = sigmas
    if si > 0:
        p[0:3] = np.exp(si * np.array(z[0:3]) / 2)
    if st > 0:
        p[3:6] = np.exp(st * np.array(z[3:6]))
    if ss > 0:
        p[6] = np.exp(ss * z[6])
    if sa > 0:
        p[7:10] = sa * np.array(z[7:10])
    return p


def hostsim_dispersion():
    d = os.path.join(HERE, "hostsim")
    csrc = os.path.join(ROOT, "tortoisesat.jl_b200", "csrc")
    deps = [os.path.join(csrc, f) for f in ("ilqr_solver.cuh", "ilqr_math.cuh", "tvlqr_solver.cuh", "philox.cuh")]
    L = AS._build("hostsim_dispersion", os.path.join(d, "hostsim_dispersion.cpp"), deps, ["-O2", "-std=c++20"])
    L.hsd_dispersion_params.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    L.hsd_tvlqr_disp_real.argtypes = [C.c_int64] + [C.c_void_p] * 5 + [C.c_int64, C.c_double, C.c_double, C.c_double, C.c_void_p,
                                                                       C.c_uint32, C.c_uint32] + [C.c_void_p] * 6
    L.hsd_tvlqr_disp_real.restype = C.c_int64
    return L


def host_params(seed, stream, r, sigmas):
    p = np.zeros(10)
    hostsim_dispersion().hsd_dispersion_params(seed, stream, r, orc.P(orc.f64(sigmas)), orc.P(p))
    return p


def host_disp_real(s, X, U, x0, g, stream, r, prm):
    """One dispersed realisation through the host build of the kernel source: (X_sim[:ns], ns, slew, x_last)."""
    L = hostsim_dispersion()
    N = s.N
    Xs, K, xl, slew = np.zeros((N, 8)), np.zeros((N, 18)), np.zeros(8), np.zeros(1)
    Up = np.zeros((N, 3))
    Up[:N - 1] = U
    B = np.ascontiguousarray(s.B)
    ns = L.hsd_tvlqr_disp_real(N, orc.P(orc.f64(X)), orc.P(Up), orc.P(orc.f64(x0)), orc.P(orc.f64(s.J.reshape(-1))), orc.P(B), B.shape[0],
                               s.index_scale, s.clock_rate, s.t_final, orc.P(orc.f64(s.xf[3:7])), stream, r, orc.P(orc.f64(prm)),
                               C.addressof(g), orc.P(Xs), orc.P(K), orc.P(xl), orc.P(slew))
    return Xs[:ns], ns, slew[0], xl


def oracle_lib():
    d = os.path.join(HERE, "dispersion_ref")
    odir = os.path.join(ROOT, "oracle")
    deps = [os.path.join(odir, f) for f in sorted(os.listdir(odir)) if f.endswith(".hpp")]
    L = AS._build("dispersion_ref", os.path.join(d, "dispersion_ref.cpp"), deps, ["-O2", "-std=c++17"])
    L.dre_attitude_simulation_truth.argtypes = [C.POINTER(orc.Dyn), C.POINTER(orc.TvlqrOpts), C.c_int64] + [C.c_void_p] * 7
    L.dre_attitude_simulation_truth.restype = C.c_int64
    return L


def oracle_truth(s, X, U, x0, o, prm, noise):
    """The oracle's truth-model replay of one slew (nominal gains) fed the parameters prm and the explicit stage draws
    noise ((N, 4, 9)): (X_sim[:ns], ns, slew_time by the oracle's mc_slew_time)."""
    L = oracle_lib()
    d = orc.make_dyn(s.B, s.index_scale, s.clock_rate, s.J)
    o.tf = s.t_final
    N = s.N
    Xs, K = np.zeros((N, 8)), np.zeros((N - 1, 18))
    ns = L.dre_attitude_simulation_truth(C.byref(d), C.byref(o), N, orc.P(orc.f64(X)), orc.P(orc.f64(U)), orc.P(orc.f64(x0)),
                                         orc.P(orc.f64(noise)), orc.P(orc.f64(prm)), orc.P(Xs), orc.P(K))
    slew = orc.lib().orc_mc_slew_time(orc.P(Xs), ns, orc.P(orc.f64(s.xf[3:7])), s.t_final, o.dt, 0.05, 0.08727, 0, 1)
    return Xs[:ns], ns, slew
