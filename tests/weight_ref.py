"""The weight-sweep ensemble's references (rules WE2 and WE4 of DESIGN.md section 4, K4): the host build of the K4 source's
replay under a given weighting and torquer limit (tests/hostsim/hostsim_weight.cpp) and the oracle's truth-model replay
with the limit (wre_attitude_simulation_truth_limited, tests/weight_ref/weight_ref.cpp), compiled with g++ on first
use into a temporary directory keyed by the source hash, so the tests write nothing into the tree."""
import ctypes as C
import os

import numpy as np

import alilqr_state as AS
from oracle import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def run_weights(cfg_tvlqr):
    """The (15,) weighting Qd 6 | Qfd 6 | Rd 3 of a TvlqrOpts."""
    return np.array(list(cfg_tvlqr.Qd) + list(cfg_tvlqr.Qfd) + list(cfg_tvlqr.Rd), dtype=np.float64)


def scaled(w, q=1.0, r=1.0, qf_equals_q=False):
    """w with Q (and Qf) scaled by q and R by r; qf_equals_q: Qf = the scaled Q."""
    w = np.array(w, dtype=np.float64)
    w[0:6] *= q
    w[6:12] = w[0:6] if qf_equals_q else w[6:12] * q
    w[12:15] *= r
    return w


def hostsim_weight():
    d = os.path.join(HERE, "hostsim")
    csrc = os.path.join(ROOT, "tortoisesat.jl_b200", "csrc")
    deps = [os.path.join(csrc, f) for f in ("ilqr_solver.cuh", "ilqr_math.cuh", "tvlqr_solver.cuh", "philox.cuh")]
    L = AS._build("hostsim_weight", os.path.join(d, "hostsim_weight.cpp"), deps, ["-O2", "-std=c++20"])
    L.hsw_tvlqr_weight_real.argtypes = [C.c_int64] + [C.c_void_p] * 5 + [C.c_int64, C.c_double, C.c_double, C.c_double, C.c_void_p,
                                                                         C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                                                         C.c_double] + [C.c_void_p] * 4
    L.hsw_tvlqr_weight_real.restype = C.c_int64
    return L


def host_weight_real(s, X, U, x0, g, stream, r, prm, w15, u_limit):
    """One realisation through the host build of the kernel source under weighting w15 and limit u_limit: (X_sim[:ns],
    ns, slew, x_last)."""
    L = hostsim_weight()
    N = s.N
    Xs, K, xl, slew = np.zeros((N, 8)), np.zeros((N, 18)), np.zeros(8), np.zeros(1)
    Up = np.zeros((N, 3))
    Up[:N - 1] = U
    B = np.ascontiguousarray(s.B)
    ns = L.hsw_tvlqr_weight_real(N, orc.P(orc.f64(X)), orc.P(Up), orc.P(orc.f64(x0)), orc.P(orc.f64(s.J.reshape(-1))), orc.P(B), B.shape[0],
                                 s.index_scale, s.clock_rate, s.t_final, orc.P(orc.f64(s.xf[3:7])), stream, r, orc.P(orc.f64(prm)),
                                 C.addressof(g), orc.P(orc.f64(w15)), float(u_limit), orc.P(Xs), orc.P(K), orc.P(xl), orc.P(slew))
    return Xs[:ns], ns, slew[0], xl


def oracle_lib():
    d = os.path.join(HERE, "weight_ref")
    odir = os.path.join(ROOT, "oracle")
    deps = [os.path.join(odir, f) for f in sorted(os.listdir(odir)) if f.endswith(".hpp")]
    deps.append(os.path.join(HERE, "dispersion_ref", "dispersion_ref.cpp"))
    L = AS._build("weight_ref", os.path.join(d, "weight_ref.cpp"), deps, ["-O2", "-std=c++17"])
    L.wre_attitude_simulation_truth_limited.argtypes = [C.POINTER(orc.Dyn), C.POINTER(orc.TvlqrOpts), C.c_int64] + [C.c_void_p] * 7 + [C.c_double]
    L.wre_attitude_simulation_truth_limited.restype = C.c_int64
    return L


def oracle_truth_weighted(s, X, U, x0, o, prm, noise, w15, u_limit):
    """The oracle's truth-model replay (DR.oracle_truth) with the gains of weighting w15 and the torquer limit u_limit
    (0: none): (X_sim[:ns], ns, slew_time)."""
    L = oracle_lib()
    for i in range(6):
        o.Qd[i], o.Qfd[i] = float(w15[i]), float(w15[6 + i])
    for i in range(3):
        o.Rd[i] = float(w15[12 + i])
    d = orc.make_dyn(s.B, s.index_scale, s.clock_rate, s.J)
    o.tf = s.t_final
    N = s.N
    Xs, K = np.zeros((N, 8)), np.zeros((N - 1, 18))
    ns = L.wre_attitude_simulation_truth_limited(C.byref(d), C.byref(o), N, orc.P(orc.f64(X)), orc.P(orc.f64(U)), orc.P(orc.f64(x0)),
                                                 orc.P(orc.f64(noise)), orc.P(orc.f64(prm)), orc.P(Xs), orc.P(K), float(u_limit))
    slew = orc.lib().orc_mc_slew_time(orc.P(Xs), ns, orc.P(orc.f64(s.xf[3:7])), s.t_final, o.dt, 0.05, 0.08727, 0, 1)
    return Xs[:ns], ns, slew
