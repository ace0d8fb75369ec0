"""CPU: the field-map interpolant of igrf_data (magnetic_toolbox.jl:124-125) -- the restatement of rules FM1..FM4
(DESIGN section 4, K8; tests/field_map_ref/orc_field_map.hpp) against an independent numpy transcription of the same
rules (scipy.linalg.solve_banded for FM1), the properties FM1 + FM2 imply, and the exports of the C ABI."""
import ctypes
import os
import re

import numpy as np
import pytest
from scipy.linalg import solve_banded

import field_map_oracle as fmo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [(2, 2), (2, 5), (5, 2), (3, 7), (13, 29), (40, 17)]


# ------------------------------------------------------------------ numpy transcription of FM1..FM3
def np_prefilter_axis(a, axis):
    """FM1 along `axis`: the (n+2)-row system c0 - c1 = 0, c_{k-1}/6 + 2c_k/3 + c_{k+1}/6 = a_k, c_{n+1} - c_n = 0."""
    a = np.moveaxis(a, axis, 0)
    n = a.shape[0]
    ab = np.zeros((3, n + 2))
    ab[0, 1] = -1.0
    ab[0, 2:] = 1.0 / 6.0
    ab[1, :] = 2.0 / 3.0
    ab[1, 0] = ab[1, -1] = 1.0
    ab[2, :n] = 1.0 / 6.0
    ab[2, n] = -1.0
    rhs = np.zeros((n + 2,) + a.shape[1:])
    rhs[1:-1] = a
    c = solve_banded((1, 1), ab, rhs.reshape(n + 2, -1)).reshape(rhs.shape)
    return np.moveaxis(c, 0, axis)


def np_prefilter(grid):
    return np_prefilter_axis(np_prefilter_axis(grid, 1), 0)


def np_weights(x, n):
    k = np.clip(np.floor(x), 1, n - 1)
    d = x - k
    w = np.stack([(1 - d) ** 3 / 6, 2 / 3 - d ** 2 + d ** 3 / 2, 2 / 3 - (1 - d) ** 2 + (1 - d) ** 3 / 2, d ** 3 / 6], -1)
    return k.astype(np.int64), w


def np_eval(C, x0, x1):
    n0, n1 = C.shape[0] - 2, C.shape[1] - 2
    x0 = np.mod(x0 - 0.5, n0) + 0.5          # FM3
    x1 = np.mod(x1 - 0.5, n1) + 0.5
    k0, w0 = np_weights(x0, n0)
    k1, w1 = np_weights(x1, n1)
    out = np.zeros((x0.shape[0], 3))
    for m in range(4):
        for l in range(4):
            out += (w0[:, m] * w1[:, l])[:, None] * C[k0 - 1 + m, k1 - 1 + l]
    return out


def sample_points(n0, n1, rng, count=4000):
    """Random points over several periods, the outer half cells, nodes, and dyadic points that hit cell edges."""
    x0 = np.concatenate([rng.uniform(-3 * n0, 4 * n0, count), rng.uniform(0.5, 1.0, 50), rng.uniform(n0, n0 + 0.5, 50),
                         np.arange(1, n0 + 1, dtype=float), [0.5, n0 + 0.5 - 2 ** -40, -1e6 + 0.25, 1e6 + 0.75]])
    x1 = np.concatenate([rng.uniform(-3 * n1, 4 * n1, count), rng.uniform(n1, n1 + 0.5, 50), rng.uniform(0.5, 1.0, 50),
                         np.arange(1, n1 + 1, dtype=float)[np.arange(n0) % n1], [n1 + 0.5 - 2 ** -40, 0.5, 7.5, -33.125]])
    return x0, x1


@pytest.mark.parametrize("shape", SHAPES)
def test_reference_matches_numpy_transcription(shape):
    n0, n1 = shape
    rng = np.random.default_rng(n0 * 100 + n1)
    grid = rng.normal(size=(n0, n1, 3)) * np.array([2e-5, 5e-6, 4e-5])
    scale = np.abs(grid).max()
    C = fmo.prefilter(grid)
    assert C.shape == (n0 + 2, n1 + 2, 3)
    assert np.abs(C - np_prefilter(grid)).max() <= 1e-13 * scale
    x0, x1 = sample_points(n0, n1, rng)
    got, bad = fmo.evaluate(C, x0, x1)
    assert bad == 0
    assert np.abs(got - np_eval(np_prefilter(grid), x0, x1)).max() <= 1e-13 * scale


@pytest.mark.parametrize("shape", SHAPES)
def test_nodes_reproduce_the_data(shape):
    """FM1 + FM2: at every integer node S equals the data, nodes 1 and n included."""
    n0, n1 = shape
    rng = np.random.default_rng(7)
    grid = rng.normal(size=(n0, n1, 3))
    C = fmo.prefilter(grid)
    I, J = np.meshgrid(np.arange(1, n0 + 1, dtype=float), np.arange(1, n1 + 1, dtype=float), indexing="ij")
    got, _ = fmo.evaluate(C, I.ravel(), J.ravel())
    assert np.abs(got - grid.reshape(-1, 3)).max() <= 1e-13 * np.abs(grid).max()


def test_constant_map_is_reproduced():
    """A constant map gives that constant everywhere (exact in real arithmetic; here up to a few rounding errors)."""
    v = np.array([1.5e-5, -3.25e-6, 4.0e-5])
    grid = np.broadcast_to(v, (9, 6, 3)).copy()
    C = fmo.prefilter(grid)
    rng = np.random.default_rng(3)
    got, _ = fmo.evaluate(C, rng.uniform(-20, 30, 2000), rng.uniform(-20, 30, 2000))
    assert np.abs(got - v).max() <= 8 * np.finfo(float).eps * np.abs(v).max()


@pytest.mark.parametrize("axis", [0, 1])
def test_value_and_slope_are_continuous_across_an_interior_knot(axis):
    """The cubic B-spline is C2; value and first derivative (one-sided finite differences) must match across the
    knot x = 4 between the segments k = 3 and k = 4.  A slope jump would show up as an O(1) difference."""
    rng = np.random.default_rng(11)
    grid = rng.normal(size=(8, 9, 3))
    C = fmo.prefilter(grid)
    h, knot, other = 1e-4, 4.0, 5.3

    def S(x):
        x = np.atleast_1d(np.asarray(x, dtype=float))
        o = np.full_like(x, other)
        return fmo.evaluate(C, *((x, o) if axis == 0 else (o, x)))[0]

    left, mid, right = S(knot - h), S(knot), S(knot + h)
    # second-order one-sided differences: each side sees only its own segment's polynomial
    slope_l = (3 * mid - 4 * left + S(knot - 2 * h)) / (2 * h)
    slope_r = (-3 * mid + 4 * right - S(knot + 2 * h)) / (2 * h)
    scale = np.abs(grid).max()
    assert np.abs(right - left).max() <= 1e-3 * scale
    assert np.abs(slope_r - slope_l).max() <= 1e-5 * scale
    # the same differences straddling a point of one segment as a control of the tolerance's size
    inner_l = (3 * S(4.5) - 4 * S(4.5 - h) + S(4.5 - 2 * h)) / (2 * h)
    inner_r = (-3 * S(4.5) + 4 * S(4.5 + h) - S(4.5 + 2 * h)) / (2 * h)
    assert np.abs(inner_r - inner_l).max() <= 1e-5 * scale


def test_periodic_wrap_identities():
    """FM3: S(x0 + p n0, x1 + q n1) = S(x0, x1) (bit-identical on dyadic points, where every step of the wrap is exact),
    and the component index wraps with period 3 (FM4)."""
    n0, n1 = 11, 6
    rng = np.random.default_rng(5)
    C = fmo.prefilter(rng.normal(size=(n0, n1, 3)))
    x0 = np.round(rng.uniform(0.5, n0 + 0.5, 500) * 1024) / 1024
    x1 = np.round(rng.uniform(0.5, n1 + 0.5, 500) * 1024) / 1024
    base, _ = fmo.evaluate(C, x0, x1)
    for p, q in [(1, 0), (0, 1), (-1, -1), (3, -5), (-40, 17)]:
        got, _ = fmo.evaluate(C, x0 + p * n0, x1 + q * n1)
        assert np.array_equal(got, base), (p, q)
    for c in (1, 2, 3):
        v = fmo.call(C, 2.25, 3.5, c)
        assert v == fmo.evaluate(C, [2.25], [3.5])[0][0, c - 1]
        assert fmo.call(C, 2.25, 3.5, c + 3) == v == fmo.call(C, 2.25, 3.5, c - 3)
        assert fmo.call(C, 2.25 + n0, 3.5 - n1, c) == v
    assert fmo.call(C, 2.25, 3.5, 0) == fmo.call(C, 2.25, 3.5, 3)


def test_fractional_component_is_rejected_and_nan_index_gives_nan_row():
    C = fmo.prefilter(np.ones((4, 4, 3)))
    with pytest.raises(ValueError):
        fmo.call(C, 2.0, 2.0, 1.5)
    out, bad = fmo.evaluate(C, np.array([1.5, np.nan, 2.0, 1.0]), np.array([1.5, 2.0, np.inf, 3.0]))
    assert bad == 2
    assert np.all(np.isnan(out[1:3])) and np.all(np.isfinite(out[[0, 3]]))


# ------------------------------------------------------------------ C ABI (no compute without a GPU)
def test_field_map_entry_points_exported_and_version():
    import __graft_entry__ as g
    g.build()
    import tortoisesat.jl_b200 as tb
    lib = ctypes.CDLL(tb.lib_path())
    for s in ("ts_field_map_prefilter", "ts_field_map_eval_batch"):
        assert hasattr(lib, s), s
    assert lib.ts_version() >= 101
    hdr = open(os.path.join(ROOT, "include", "tortoise_b200.h")).read()
    assert re.search(r"int ts_field_map_prefilter\(ts_ctx\* ctx, int64_t n0, int64_t n1, const double\* grid, double\* coefs, "
                     r"int pointers_are_device\);", hdr)
    assert "src/magnetic_toolbox.jl:124-125" in hdr


def test_k8_kernels_use_no_local_memory():
    """Static check of the shipped library (cuobjdump, no GPU): the K8 kernels are compiled for sm_100a with no spill
    or local-memory traffic."""
    import shutil
    import subprocess
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import __graft_entry__ as g
    g.build()
    import tortoisesat.jl_b200 as tb
    sass = subprocess.run([exe, "-sass", tb.lib_path()], capture_output=True, text=True, check=True).stdout
    bodies = re.split(r"\n\s*Function : ", sass)
    k8 = [b for b in bodies if re.match(r"\S*k8_", b)]
    assert len(k8) == 4, [b.split("\n", 1)[0] for b in k8]
    for b in k8:
        assert not re.search(r"\b(LDL|STL)\b", b), b.split("\n", 1)[0]


def test_host_rejects_bad_shapes_before_the_library():
    from tortoisesat.jl_b200 import host
    with pytest.raises(ValueError):
        host._field_map_grid_dims((1, 5, 3))
    with pytest.raises(ValueError):
        host._field_map_grid_dims((4, 5, 2))
    with pytest.raises(ValueError):
        host._field_map_coef_dims((3, 6, 3))
    assert host._field_map_coef_dims((1002, 1002, 3)) == (1000, 1000)
