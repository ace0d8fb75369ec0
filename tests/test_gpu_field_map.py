"""GPU: K8, the cubic B-spline interpolant of the igrf_data map (magnetic_toolbox.jl:124-125, rules FM1..FM4 of DESIGN
section 4), through the C ABI against the CPU restatement (tests/field_map_ref/orc_field_map.hpp)."""
import math

import numpy as np
import pytest

import field_map_oracle as fmo

pytestmark = pytest.mark.gpu


def random_grid(n0, n1, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(size=(n0, n1, 3)) * np.array([2e-5, 5e-6, 4e-5])


def eval_points(n0, n1, count, seed):
    """Random points over several periods, the outer half cells, negative and far-out indices, and every node."""
    rng = np.random.default_rng(seed)
    m = count - n0 * n1 - 400
    x0 = np.concatenate([rng.uniform(-2 * n0, 3 * n0, m), rng.uniform(0.5, 1.0, 100), rng.uniform(n0, n0 + 0.5, 100),
                         rng.uniform(-1e7, -1e6, 100), rng.uniform(1e6, 1e9, 100)])
    x1 = np.concatenate([rng.uniform(-2 * n1, 3 * n1, m), rng.uniform(n1, n1 + 0.5, 100), rng.uniform(0.5, 1.0, 100),
                         rng.uniform(1e6, 1e9, 100), rng.uniform(-1e7, -1e6, 100)])
    I, J = np.meshgrid(np.arange(1, n0 + 1, dtype=float), np.arange(1, n1 + 1, dtype=float), indexing="ij")
    return np.concatenate([x0, I.ravel()]), np.concatenate([x1, J.ravel()])


@pytest.mark.parametrize("shape", [(2, 2), (2, 9), (7, 3), (61, 45), (1000, 1000)])
def test_prefilter_vs_reference(engine, shape):
    grid = random_grid(*shape, seed=shape[0] + 7 * shape[1])
    got = engine.field_map_prefilter(grid)
    ref = fmo.prefilter(grid)
    assert got.shape == ref.shape
    assert np.abs(got - ref).max() <= 1e-13 * np.abs(grid).max()


@pytest.mark.parametrize("shape", [(2, 3), (61, 45), (200, 333)])
def test_eval_vs_reference_1e5_points(engine, shape):
    n0, n1 = shape
    grid = random_grid(n0, n1, seed=3)
    coefs = fmo.prefilter(grid)
    x0, x1 = eval_points(n0, n1, 100_000, seed=n0)
    got = engine.field_map_eval_batch(coefs, x0, x1)
    ref, bad = fmo.evaluate(coefs, x0, x1)
    assert bad == 0
    assert np.abs(got - ref).max() <= 1e-13 * np.abs(grid).max()
    nodes = got[-n0 * n1:]
    assert np.abs(nodes - grid.reshape(-1, 3)).max() <= 1e-13 * np.abs(grid).max()   # FM1 + FM2: S = data at every node


def test_host_and_device_paths_bit_identical(engine):
    import torch
    n0, n1 = 129, 77
    grid = random_grid(n0, n1, seed=5)
    x0, x1 = eval_points(n0, n1, 200_000, seed=9)
    c_host = engine.field_map_prefilter(grid)
    c_dev = engine.field_map_prefilter(torch.from_numpy(grid).cuda())
    assert np.array_equal(c_host, c_dev.cpu().numpy())
    o_host = engine.field_map_eval_batch(c_host, x0, x1)
    o_dev = engine.field_map_eval_batch(c_dev, torch.from_numpy(x0).cuda(), torch.from_numpy(x1).cuda())
    assert np.array_equal(o_host, o_dev.cpu().numpy())
    assert engine.last_kernel_ms() > 0.0


def test_nonfinite_index_gives_domain_error_and_nan_row_only(engine):
    import tortoisesat.jl_b200 as tb
    grid = random_grid(10, 12, seed=1)
    coefs = engine.field_map_prefilter(grid)
    x0 = np.array([1.5, 2.25, np.nan, 4.0, 9.75])
    x1 = np.array([3.5, np.inf, 1.0, 7.0, -2.0])
    out = np.zeros((5, 3))
    with pytest.raises(tb.TortoiseError) as ei:
        engine.field_map_eval_batch(coefs, x0, x1, out=out)
    assert ei.value.code == tb.host.TS_ERR_DOMAIN
    assert np.all(np.isnan(out[1:3]))
    ok = [0, 3, 4]
    assert not np.any(np.isnan(out[ok]))
    assert np.array_equal(out[ok], engine.field_map_eval_batch(coefs, x0[ok], x1[ok]))


def test_argument_errors(engine):
    lib = engine.lib
    g = np.zeros((4, 4, 3))
    c = np.zeros((6, 6, 3))
    x = np.zeros(4)
    o = np.zeros((4, 3))
    TS_ERR_ARG = -2
    assert lib.ts_field_map_prefilter(engine.h, 1, 4, g.ctypes.data, c.ctypes.data, 0) == TS_ERR_ARG
    assert lib.ts_field_map_prefilter(engine.h, 4, -4, g.ctypes.data, c.ctypes.data, 0) == TS_ERR_ARG
    assert lib.ts_field_map_prefilter(engine.h, 4, 4, None, c.ctypes.data, 0) == TS_ERR_ARG
    assert lib.ts_field_map_eval_batch(engine.h, 4, 4, c.ctypes.data, -1, x.ctypes.data, x.ctypes.data, o.ctypes.data, 0) == TS_ERR_ARG
    assert lib.ts_field_map_eval_batch(engine.h, 4, 4, c.ctypes.data, 4, x.ctypes.data, None, o.ctypes.data, 0) == TS_ERR_ARG
    assert lib.ts_field_map_eval_batch(engine.h, 4, 1, c.ctypes.data, 4, x.ctypes.data, x.ctypes.data, o.ctypes.data, 0) == TS_ERR_ARG
    assert lib.ts_field_map_eval_batch(engine.h, 4, 4, c.ctypes.data, 0, None, None, None, 0) == 0
    assert engine.field_map_eval_batch(c, np.zeros(0), np.zeros(0)).shape == (0, 3)


def test_interpolant_call_shape(engine):
    """MagFieldMap.interpolant(): real i, j with periodic wrap, integer c with period 3 (FM4); a fractional c is
    rejected; the map's own __call__ still takes integer nodes only."""
    import tortoisesat.jl_b200 as tb
    grid = random_grid(20, 31, seed=2)
    mf = tb.host.MagFieldMap(grid)
    s = mf.interpolant(engine)
    coefs = fmo.prefilter(grid)
    scale = np.abs(grid).max()
    for (i, j) in [(1.0, 1.0), (20.0, 31.0), (3.25, 17.5), (0.6, 31.4), (-7.125, 100.75)]:
        for c in (1, 2, 3):
            assert abs(s(i, j, c) - fmo.call(coefs, i, j, c)) <= 1e-13 * scale
    assert abs(s(5, 7, 2) - mf(5, 7, 2)) <= 1e-13 * scale
    assert s(3.25, 17.5, 4) == s(3.25, 17.5, 1) == s(3.25 + 20, 17.5 - 31, 1)
    assert s(3.25, 17.5, 0) == s(3.25, 17.5, 3)
    with pytest.raises(ValueError):
        s(3.25, 17.5, 1.5)
    with pytest.raises(ValueError):
        mf(1.5, 2, 1)
    got = s.eval(np.array([3.25, 4.0]), np.array([17.5, 2.0]))
    assert got.shape == (2, 3) and isinstance(got, np.ndarray)
    assert np.array_equal(got[0], [s(3.25, 17.5, c) for c in (1, 2, 3)])


# The spline of the 1000 x 1000 map between its nodes against the field itself: sanity bounds, not tuned tolerances.
# Relative errors (norm of the difference / norm of the field) printed on a B200 at the 999^2 cell centres:
#  - 1.36e-1 at worst, in the cells next to the south-pole row: there the map's east component is -0 at every
#    longitude (the s == 0 branch of igrf.jl at theta = pi), not the limit of its neighbours, and the spline passes
#    through that row; the error falls by 2 + sqrt(3) per cell away from it;
#  - 1.5e-4 next to the first and last longitude columns: Reflect(OnCell()) gives the spline zero slope at the map's
#    edges (the map is not treated as periodic in longitude, FM3), decaying the same way;
#  - 1.7e-10 at least 20 cells from every edge (grid spacing 0.18 deg in lat, 0.36 deg in long).
IGRF_ALL_BOUND = 0.2
IGRF_INTERIOR_BOUND = 1e-9


def test_igrf_interpolant_at_cell_centres_vs_k1(engine):
    import tortoisesat.jl_b200 as tb
    n = 1000
    mf = tb.host.igrf_data(400, 2019, n=n)
    s = mf.interpolant(engine)
    c = np.arange(1, n, dtype=float) + 0.5
    I, J = np.meshgrid(c, c, indexing="ij")
    got = s.eval(I.ravel(), J.ravel())
    lat = -math.pi / 2 + (I.ravel() - 1) * math.pi / (n - 1)
    lon = -math.pi + (J.ravel() - 1) * 2 * math.pi / (n - 1)
    ref = np.stack(engine.igrf12_batch(2019.0, np.full(lat.size, (400 + 6378) * 1000.0), lat, lon), -1) / 1e9
    err = (np.linalg.norm(got - ref, axis=1) / np.linalg.norm(ref, axis=1)).reshape(n - 1, n - 1)
    inner = err[20:-20, 20:-20]
    print("igrf interpolant at cell centres: max rel err %.3e (row next to the south pole %.3e, next to the first "
          "longitude column %.3e), >= 20 cells from every edge %.3e"
          % (err.max(), err[0].max(), err[20:-20, 0].max(), inner.max()))
    assert err.max() <= IGRF_ALL_BOUND
    assert inner.max() <= IGRF_INTERIOR_BOUND
