"""CPU restatement of the field-map interpolant (FM1..FM4, tests/field_map_ref/orc_field_map.hpp): test infrastructure.

The library is compiled with g++ on first use into a temporary directory (keyed by the source hash), so the tests
write nothing into the tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "field_map_ref")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        srcs = [os.path.join(_DIR, f) for f in ("field_map_ref.cpp", "orc_field_map.hpp")]
        h = hashlib.sha256(b"".join(open(s, "rb").read() for s in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "ts_field_map_ref_%d_%s.so" % (os.getuid(), h))
        if not os.path.exists(so):
            tmp = so + ".%d" % os.getpid()
            r = subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", tmp, srcs[0]],
                               capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("field-map reference build failed:\n" + r.stderr)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.orc_field_map_prefilter.argtypes = [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
        L.orc_field_map_prefilter.restype = None
        L.orc_field_map_eval.argtypes = [C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_field_map_eval.restype = C.c_int64
        L.orc_field_map_call.argtypes = [C.c_int64, C.c_int64, C.c_void_p, C.c_double, C.c_double, C.c_double,
                                         C.POINTER(C.c_double)]
        L.orc_field_map_call.restype = C.c_int
        _LIB = L
    return _LIB


def prefilter(grid):
    """FM1: n0 x n1 x 3 grid -> (n0+2) x (n1+2) x 3 coefficients."""
    grid = np.ascontiguousarray(grid, dtype=np.float64)
    n0, n1, _ = grid.shape
    coefs = np.empty((n0 + 2, n1 + 2, 3))
    lib().orc_field_map_prefilter(n0, n1, grid.ctypes.data, coefs.ctypes.data)
    return coefs


def evaluate(coefs, x0, x1):
    """FM2 + FM3 at the points (x0[p], x1[p]) -> (n x 3, number of non-finite points)."""
    coefs = np.ascontiguousarray(coefs, dtype=np.float64)
    x0, x1 = np.ascontiguousarray(x0, dtype=np.float64), np.ascontiguousarray(x1, dtype=np.float64)
    out = np.empty((x0.shape[0], 3))
    bad = lib().orc_field_map_eval(coefs.shape[0] - 2, coefs.shape[1] - 2, coefs.ctypes.data, x0.shape[0], x0.ctypes.data,
                                   x1.ctypes.data, out.ctypes.data)
    return out, int(bad)


def call(coefs, i, j, c):
    """FM1..FM4: mag_field(i, j, c); raises ValueError for a fractional component index."""
    coefs = np.ascontiguousarray(coefs, dtype=np.float64)
    v = C.c_double()
    if lib().orc_field_map_call(coefs.shape[0] - 2, coefs.shape[1] - 2, coefs.ctypes.data, i, j, c, C.byref(v)):
        raise ValueError("fractional component index %r" % c)
    return v.value
