"""Continuation of the AL-iLQR solve on the CPU (test infrastructure): the oracle with the solver state in and out
(tests/alilqr_state_ref) and the export / import pair of the lane emulator (tests/hostsim/hostsim_state.cpp).

Both libraries are compiled with g++ on first use into a temporary directory (keyed by the source hash), so the tests
write nothing into the tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
AL_STATE_DTYPE = np.dtype([("mu", "<f8"), ("lam_goal", "<f8", (8,)), ("J", "<f8"), ("c_max", "<f8"), ("status", "<i4"),
                           ("outer_iters", "<i4"), ("inner_iters", "<i4"), ("ls_rollouts", "<i4")])
_LIBS = {}


def _build(name, main, deps, flags):
    if name not in _LIBS:
        srcs = [main] + deps
        h = hashlib.sha256(b"".join(open(s, "rb").read() for s in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "ts_%s_%d_%s.so" % (name, os.getuid(), h))
        if not os.path.exists(so):
            tmp = so + ".%d" % os.getpid()
            r = subprocess.run(["/usr/bin/g++"] + flags + ["-fPIC", "-shared", "-ffp-contract=off", "-o", tmp, main],
                               capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("%s build failed:\n%s" % (name, r.stderr))
            os.replace(tmp, so)
        _LIBS[name] = C.CDLL(so)
    return _LIBS[name]


def oracle_lib():
    d = os.path.join(HERE, "alilqr_state_ref")
    odir = os.path.join(ROOT, "oracle")
    deps = [os.path.join(d, "orc_alilqr_state.hpp")] + [os.path.join(odir, f) for f in sorted(os.listdir(odir))
                                                         if f.endswith((".cpp", ".hpp", ".inc"))]
    L = _build("alilqr_state_ref", os.path.join(d, "alilqr_state_ref.cpp"), deps, ["-O2", "-std=c++17", "-fopenmp"])
    L.orc_alilqr_solve_state_batch.argtypes = [C.c_int64] + [C.c_void_p] * 13 + [C.c_double, C.c_void_p, C.POINTER(orc.IlqrOpts)] + \
        [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 4
    return L


def hostsim_lib():
    d = os.path.join(HERE, "hostsim")
    csrc = os.path.join(ROOT, "tortoisesat.jl_b200", "csrc")
    deps = [os.path.join(d, "hostsim.cpp")] + [os.path.join(csrc, f) for f in ("ilqr_solver.cuh", "ilqr_math.cuh", "tvlqr_solver.cuh")]
    L = _build("hostsim_state", os.path.join(d, "hostsim_state.cpp"), deps, ["-O2", "-std=c++20", "-pthread"])
    L.hs_alilqr_solve_state_w.argtypes = [C.c_int, C.c_int64] + [C.c_void_p] * 7 + [C.c_int64, C.c_double, C.c_double, C.c_double] + \
        [C.c_void_p] * 10
    return L


def pack(slews):
    """The per-trial arrays of a list of slew_setup.Slew objects, as ts_alilqr_solve_batch takes them."""
    T = len(slews)
    p = {}
    p["N_i"] = np.array([s.N for s in slews], dtype=np.int64)
    p["offs"] = np.concatenate([[0], np.cumsum(p["N_i"])]).astype(np.int64)
    rows = np.array([s.B.shape[0] for s in slews], dtype=np.int64)
    p["B_rows"] = rows
    p["B_offs"] = np.concatenate([[0], np.cumsum(rows)])[:-1].astype(np.int64)
    p["B_eci"] = np.ascontiguousarray(np.concatenate([s.B for s in slews]))
    for name, w in (("x0", 8), ("xf", 8), ("J", 9), ("Qd", 8), ("Qfd", 8), ("Rd", 3)):
        p[name] = np.ascontiguousarray(np.stack([getattr(s, name).reshape(-1) for s in slews])).reshape(T, w)
    p["index_scale"] = np.array([s.index_scale for s in slews])
    p["clock_rate"] = np.array([s.clock_rate for s in slews])
    p["dt"] = slews[0].dt
    return p


def oracle_state_solve(slews, opts, state=None, lam=None, X=None, U=None, K=None, nthreads=4):
    """The oracle's continuation solve -> (X, U, K, out, state, lam) in the ragged layout of the C ABI."""
    p = pack(slews)
    T, tot = len(slews), int(p["offs"][-1])
    X = np.zeros((tot, 8)) if X is None else np.array(X, dtype=np.float64)
    U = np.zeros((tot, 3)) if U is None else np.array(U, dtype=np.float64)
    K = np.zeros((tot, 24)) if K is None else np.array(K, dtype=np.float64).reshape(tot, 24)
    out = np.zeros(T, dtype=orc.OUTCOME_DTYPE)
    so = np.zeros(T, dtype=AL_STATE_DTYPE)
    lo = np.zeros((tot, 6))
    si = None if state is None else np.ascontiguousarray(state, dtype=AL_STATE_DTYPE)
    li = None if lam is None else np.ascontiguousarray(lam, dtype=np.float64)
    P = orc.P
    oracle_lib().orc_alilqr_solve_state_batch(
        T, P(p["N_i"]), P(p["offs"]), P(p["x0"]), P(p["xf"]), P(p["J"]), P(p["Qd"]), P(p["Qfd"]), P(p["Rd"]), P(p["B_eci"]),
        P(p["B_offs"]), P(p["B_rows"]), P(p["index_scale"]), P(p["clock_rate"]), p["dt"], None, C.byref(opts), P(X), P(U), P(K),
        out.ctypes.data, nthreads, None if si is None else si.ctypes.data, P(li), so.ctypes.data, P(lo))
    return X, U, K.reshape(tot, 3, 8), out, so, lo


def hostsim_state_solve(s, opts, width=8, state=None, lam=None, X=None, U=None):
    """One trial through the lane emulator's export / import pair -> (X, U (N x 3), K, outcome, state, lam)."""
    N = s.N
    X = np.zeros((N, 8)) if X is None else np.array(X, dtype=np.float64)
    U = np.zeros((N, 3)) if U is None else np.array(U, dtype=np.float64)
    K = np.zeros((N, 24))
    out = np.zeros(1, dtype=orc.OUTCOME_DTYPE)
    so = np.zeros(1, dtype=AL_STATE_DTYPE)
    lo = np.zeros((N, 6))
    si = None if state is None else np.ascontiguousarray(np.atleast_1d(state), dtype=AL_STATE_DTYPE)
    li = None if lam is None else np.ascontiguousarray(lam, dtype=np.float64)
    B = np.ascontiguousarray(s.B)
    f = orc.f64
    hostsim_lib().hs_alilqr_solve_state_w(
        width, N, orc.P(f(s.x0)), orc.P(f(s.xf)), orc.P(f(s.J.reshape(-1))), orc.P(f(s.Qd)), orc.P(f(s.Qfd)), orc.P(f(s.Rd)), orc.P(B),
        B.shape[0], s.index_scale, s.clock_rate, s.dt, None, C.addressof(opts), orc.P(X), orc.P(U), orc.P(K), out.ctypes.data,
        None if si is None else si.ctypes.data, orc.P(li), so.ctypes.data, orc.P(lo))
    return X, U, K.reshape(N, 3, 8), out[0], so[0], lo
