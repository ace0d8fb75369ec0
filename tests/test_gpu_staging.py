"""GPU: how the C ABI moves a call's arguments and keeps state between calls.

- Every entry with `pointers_are_device` gives bit-identical results for host arrays and for device arrays (torch CUDA
  tensors), so the two ways of staging a call cannot drift apart.
- The K3 hand-over counters that ts_k3_last_split / ts_k3_last_parked read after a solve survive later K2 calls.
- The element-wise (K5) entries set ts_last_kernel_ms like every other kernel call."""
import ctypes as C

import numpy as np
import pytest

import slew_setup as S

pytestmark = pytest.mark.gpu


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _p(a):
    """numpy array or torch CUDA tensor -> raw address; anything else is passed as it is"""
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr() if hasattr(a, "data_ptr") else a


def _call_device(engine, fn, *args):
    """engine.lib.<fn>(ctx, *args, pointers_are_device = 1) after torch's queued copies have finished (the library runs
    on its own stream)."""
    import torch
    torch.cuda.synchronize()
    engine._check(getattr(engine.lib, fn)(engine.h, *[_p(a) for a in args], 1))


def _same(host, dev):
    assert np.array_equal(host, dev.cpu().numpy().reshape(host.shape))


def _field_inputs(tb, T=5, seed=2):
    rng = np.random.default_rng(seed)
    kep = np.zeros((T, 6))
    o = np.zeros(T, dtype=tb.host.FIELD_OPTS_DTYPE)
    for t in range(T):
        alt = rng.uniform(350, 800)
        kep[t] = [0.002 * t, alt + 6371.0, rng.uniform(0, 98), rng.uniform(0, 360), 0.0, rng.uniform(0, 360)]
        o[t] = (S.GM, rng.uniform(58155, 58520), 1988.4 if t == 1 else 2015 + 5 * rng.random(), (alt + 6371.0) * 1000.0, 0.0,
                rng.uniform(300, 900), int(rng.integers(40, 300)))
    return kep, o


def test_magnetic_simulation_device_path(engine):
    import tortoisesat.jl_b200 as tb
    kep, o = _field_inputs(tb)
    B, offs, pos, vel = engine.magnetic_simulation_batch(kep, o, want_pos=True)
    dB, dpos, dvel = _dev(np.zeros_like(B)), _dev(np.zeros_like(pos)), _dev(np.zeros_like(vel))
    _call_device(engine, "ts_magnetic_simulation_batch", len(o), _dev(kep), o, offs, None, dB, dpos, dvel)
    for h, d in ((B, dB), (pos, dpos), (vel, dvel)):
        _same(h, d)


def test_gramian_and_cutoff_device_paths(engine):
    import tortoisesat.jl_b200 as tb
    kep, o = _field_inputs(tb, seed=4)
    B, offs = engine.magnetic_simulation_batch(kep, o)
    T = len(o)
    rows = (offs[1:] - offs[:-1]).astype(np.int64)
    boffs = np.ascontiguousarray(offs[:-1])
    dts = (o["tf"] - o["t0"]) / o["N"]
    cut = np.linspace(20.0, 400.0, T)
    G = engine.magnetic_gramian_batch(B, boffs, rows, dts)
    dG = _dev(np.zeros_like(G))
    _call_device(engine, "ts_magnetic_gramian_batch", T, _dev(B), boffs, rows, dts, dG)
    _same(G, dG)
    idx = engine.condition_cutoff_batch(B, boffs, rows, dts, cut)
    assert np.any(idx > 0)
    idx_d = np.zeros(T, dtype=np.int64)
    _call_device(engine, "ts_condition_cutoff_batch", T, _dev(B), boffs, rows, dts, cut, idx_d)
    assert np.array_equal(idx, idx_d)
    idx2 = engine.condition_based_time_batch(G, boffs, rows, cut)
    assert np.array_equal(idx2, idx)
    idx2_d = np.zeros(T, dtype=np.int64)
    _call_device(engine, "ts_condition_based_time_batch", T, _dev(G), boffs, rows, cut, idx2_d)
    assert np.array_equal(idx2, idx2_d)


@pytest.fixture(scope="module")
def slews():
    qf = np.array([1.0, 0, 0, 0])
    return [S.build_slew([0, 6578, 96, 0, 0, 90], S.J_1P, S.quat_axis_angle([1, 0, 1], 8.0), qf, t_final=24.0),
            S.build_slew([0, 6871, 51.6, 30, 0, 10], S.J_3U, S.quat_axis_angle([0, 1, 0], 3.0), qf, t_final=31.0),
            S.build_slew([0, 6771, 96.6, 100, 0, 200], S.J_1U, S.quat_axis_angle([0, 0, 1], 12.0), qf, t_final=20.0)]


def _solver_inputs(sl):
    T = len(sl)
    N_i = np.array([s.N for s in sl], dtype=np.int64)
    offs = np.concatenate([[0], np.cumsum(N_i)]).astype(np.int64)
    rows = np.array([s.B.shape[0] for s in sl], dtype=np.int64)
    B_offs = np.concatenate([[0], np.cumsum(rows)])[:-1].astype(np.int64)
    pk = lambda name, w: np.ascontiguousarray(np.stack([getattr(s, name).reshape(-1) for s in sl]).reshape(T, w))
    return dict(N_i=N_i, offs=offs, x0=pk("x0", 8), xf=pk("xf", 8), Jmat=pk("J", 9), Qd=pk("Qd", 8), Qfd=pk("Qfd", 8),
                Rd=pk("Rd", 3), B_eci=np.ascontiguousarray(np.concatenate([s.B for s in sl])), B_offs=B_offs, B_rows=rows,
                index_scale=np.array([s.index_scale for s in sl]), clock_rate=np.array([s.clock_rate for s in sl]))


def test_alilqr_solve_device_path(engine, slews):
    import tortoisesat.jl_b200 as tb
    a = _solver_inputs(slews)
    T, tot = len(slews), int(a["offs"][-1])
    U0 = np.random.default_rng(8).normal(size=(tot, 3)) * 1e-3
    o = tb.host.default_ilqr_opts()
    X, U, K, out, offs = engine.alilqr_solve_batch(a["N_i"], a["x0"], a["xf"], a["Jmat"], a["Qd"], a["Qfd"], a["Rd"], a["B_eci"],
                                                   a["B_offs"], a["B_rows"], a["index_scale"], a["clock_rate"], slews[0].dt,
                                                   U0=U0, opts=o)
    dX, dU, dK = _dev(np.zeros((tot, 8))), _dev(np.zeros((tot, 3))), _dev(np.zeros((tot, 3, 8)))
    out_d = np.zeros(T, dtype=tb.host.OUTCOME_DTYPE)
    _call_device(engine, "ts_alilqr_solve_batch", T, a["N_i"], a["offs"], a["x0"], a["xf"], a["Jmat"], a["Qd"],
                 a["Qfd"], a["Rd"], _dev(a["B_eci"]), a["B_offs"], a["B_rows"], a["index_scale"], a["clock_rate"],
                 float(slews[0].dt), _dev(U0), C.pointer(o), dX, dU, dK, out_d)
    assert out_d.tobytes() == out.tobytes()
    _same(X, dX)
    # U and K have N-1 rows per trial; the last row of each trial is not an output
    ctl = np.concatenate([np.arange(offs[t], offs[t + 1] - 1) for t in range(T)])
    assert np.array_equal(U[ctl], dU.cpu().numpy()[ctl]) and np.array_equal(K[ctl], dK.cpu().numpy()[ctl])


def test_tvlqr_sim_device_path(engine, slews):
    import tortoisesat.jl_b200 as tb
    a = _solver_inputs(slews)
    T = len(slews)
    X, U, _, _, offs = engine.alilqr_solve_batch(a["N_i"], a["x0"], a["xf"], a["Jmat"], a["Qd"], a["Qfd"], a["Rd"], a["B_eci"],
                                                 a["B_offs"], a["B_rows"], a["index_scale"], a["clock_rate"], slews[0].dt)
    tot = int(offs[-1])
    U[offs[1:] - 1] = 0.0                    # not a solver output
    rng = np.random.default_rng(12)
    noise = rng.normal(size=(tot, 4, 9)) * np.array([1e-5] * 3 + [3e-4] * 3 + [1e-10] * 3)
    x0l = a["x0"].copy()
    x0l[:, 7] = 0
    tfin = np.array([s.t_final for s in slews])
    qfin = np.ascontiguousarray(a["xf"][:, 3:7])
    sid = np.array([5, 9, 2], dtype=np.uint32)
    _, g = S.tvlqr_opts_pair(noise_mode=1, seed=3)
    Xs, Us, dX, K, nsim, slew, _ = engine.tvlqr_sim_batch(a["N_i"], X, U, x0l, a["Jmat"], a["B_eci"], a["B_offs"], a["B_rows"],
                                                          a["index_scale"], a["clock_rate"], tfin, qfin, opts=g, noise=noise,
                                                          stream_id=sid)
    dXs, dUs, ddX, dK = (_dev(np.zeros((tot, w))) for w in (8, 3, 6, 18))
    nsim_d, slew_d = np.zeros(T, dtype=np.int64), np.zeros(T)
    _call_device(engine, "ts_tvlqr_sim_batch", T, a["N_i"], offs, _dev(X), _dev(U), x0l, a["Jmat"], _dev(a["B_eci"]),
                 a["B_offs"], a["B_rows"], a["index_scale"], a["clock_rate"], tfin, qfin, sid, C.pointer(g), _dev(noise),
                 dXs, dUs, ddX, dK, nsim_d, slew_d)
    assert np.array_equal(nsim, nsim_d) and np.array_equal(slew, slew_d)
    sim = np.concatenate([np.arange(offs[t], offs[t] + nsim[t]) for t in range(T)])     # rows the replay reached
    ctl = np.concatenate([np.arange(offs[t], offs[t + 1] - 1) for t in range(T)])
    for h, d, r in ((Xs, dXs, sim), (Us, dUs, sim), (dX, ddX, sim), (K.reshape(tot, 18), dK, ctl)):
        assert np.array_equal(h[r], d.cpu().numpy()[r])


def test_igrf12syn_device_path(engine):
    rng = np.random.default_rng(6)
    n = 5000
    alt, colat, elong = rng.uniform(300, 900, n), rng.uniform(0.5, 179.5, n), rng.uniform(-180, 360, n)
    for isv, date, itype in ((0, 2019.0, 1), (1, 1994.0, 2)):
        ref = engine.igrf12syn_batch(isv, date, itype, alt, colat, elong)
        outs = [_dev(np.zeros(n)) for _ in range(4)]
        _call_device(engine, "ts_igrf12syn_batch", isv, date, itype, n, _dev(alt), _dev(colat), _dev(elong), *outs)
        for h, d in zip(ref, outs):
            _same(h, d)


def test_park_counter_survives_k2_calls(engine):
    """The hand-over count and the parked trials reported after a solve stay those of the solve when a K2 call follows."""
    import tortoisesat.jl_b200 as tb
    rng = np.random.default_rng(5)
    sl = [S.build_slew([0, 6578, 96, 0, 0, 90], S.J_1P, S.quat_axis_angle(rng.normal(size=3), rng.uniform(3, 25)),
                       np.array([1.0, 0, 0, 0]), t_final=float(rng.integers(20, 50))) for _ in range(12)]
    a = _solver_inputs(sl)
    o = tb.host.default_ilqr_opts()
    o.k3_suspend_after = 10
    engine.alilqr_solve_batch(a["N_i"], a["x0"], a["xf"], a["Jmat"], a["Qd"], a["Qfd"], a["Rd"], a["B_eci"], a["B_offs"],
                              a["B_rows"], a["index_scale"], a["clock_rate"], sl[0].dt, opts=o)
    n_parked = engine.k3_last_split()[2]
    parked = engine.k3_last_parked(64)
    assert n_parked > 0
    T = 8
    B = np.random.default_rng(1).normal(size=(T * 60, 3)) * 2e-5
    engine.condition_cutoff_batch(B, 60 * np.arange(T), np.full(T, 60), np.full(T, 1.0), np.full(T, 30.0))
    assert engine.k3_last_split()[2] == n_parked
    for before, after in zip(parked, engine.k3_last_parked(64)):
        assert np.array_equal(before, after)


def test_elementwise_calls_set_last_kernel_ms(engine):
    rng = np.random.default_rng(0)
    engine.igrf12_batch(2019.0, 6.8e6 + rng.random(1000), rng.uniform(-1.5, 1.5, 1000), rng.uniform(-3, 3, 1000))
    after_igrf = engine.last_kernel_ms()
    n = 1_000_000
    kep = np.column_stack([np.full(n, 0.001), rng.uniform(6700, 7200, n), rng.uniform(0, 98, n), rng.uniform(0, 360, n),
                           rng.uniform(0, 360, n), rng.uniform(0, 360, n)])
    engine.kep_eci_batch(kep)
    assert engine.last_kernel_ms() > 0.0
    assert engine.last_kernel_ms() != after_igrf
