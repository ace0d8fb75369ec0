"""GPU: weight-sweep ensembles of a kept Monte-Carlo run (ts_mc_weight_ensemble, ts_multi_mc_weight_ensemble; rules
WE1-WE7 of DESIGN.md section 4, K4) against the dispersion and disturbance ensembles, the CPU oracle's truth-model
replay under the set's weighting and torquer limit, other call shapes, later calls and the error cases."""
import ctypes as C
import math
import types

import numpy as np
import pytest

import replay_ensemble_ref as RE
import slew_setup as S
import weight_ref as WR
from test_gpu_dispersion_ensemble import ALL
from test_gpu_mc_continue import J_GEN, cont_opts, run, shared_ensemble, snapshot, sweep_ensemble

pytestmark = pytest.mark.gpu
QS = (math.pi / 180) ** 2


def four_sets(cfg):
    """Four weightings, the run's own second: R x 0.01, the run's, Q x 10, Qf = Q."""
    w = WR.run_weights(cfg.tvlqr)
    return np.stack([WR.scaled(w, r=0.01), w, WR.scaled(w, q=10.0), WR.scaled(w, qf_equals_q=True)])


def assert_we3(engine, e, out, n, n_real=40):
    """The run's weighting (set 1) with u_limit 0: rows bit-equal to mc_dispersion_ensemble with every group on and to
    mc_replay_ensemble with a null dispersion; a NO_CUTOFF trial gets NaN rows in every set."""
    sets = four_sets(e["cfg"])
    s, x = engine.mc_weight_ensemble(n, n_real, sets, 0.0, ALL, want_x_final=True)
    assert s.shape == (n, 4, n_real) and x.shape == (n, 4, n_real, 8)
    sd, xd, _ = engine.mc_dispersion_ensemble(n, n_real, want_x_final=True, **ALL)
    assert s[:, 1].tobytes() == sd.tobytes() and x[:, 1].tobytes() == xd.tobytes()
    s0, x0 = engine.mc_weight_ensemble(n, n_real, sets, 0.0, None, want_x_final=True)
    se, xe = engine.mc_replay_ensemble(n, n_real, want_x_final=True)
    assert s0[:, 1].tobytes() == se.tobytes() and x0[:, 1].tobytes() == xe.tobytes()
    g, r = engine.mc_replay_ensemble_split()
    assert g > 0 and r > 0 and engine.last_kernel_ms() > 0
    for t in range(n):
        nc = out["status"][t] == 5
        for a in (s[t], x[t], s0[t], x0[t]):
            assert np.all(np.isnan(a)) == nc and (nc or not np.any(np.isnan(a))), t
        if not nc:   # the weightings change the rows
            for w in (0, 2, 3):
                assert np.any(x[t, w] != x[t, 1]), (t, w)


@pytest.mark.parametrize("quat,J", [(0, "diag"), (1, "diag"), (0, "general")])
def test_we3_fixed_orbit(engine, quat, J):
    e = shared_ensemble(J=S.J_1U if J == "diag" else J_GEN)
    n = len(e["x0"])
    out, _ = run(engine, e, 5, keep=1, quat=quat)
    assert_we3(engine, e, out, n)


def test_we3_sweep(engine):
    """The sweep: ragged horizons, one NO_CUTOFF trial."""
    e = sweep_ensemble()
    n = len(e["x0"])
    out, _ = run(engine, e, 8, keep=1)
    assert (out["status"] == 5).sum() == 1
    assert_we3(engine, e, out, n)


def test_oracle_with_and_without_the_limit(engine):
    """The longest sweep slew and r = 2^30 - 1, each non-default set with u_limit 0 and 1, every group on: the oracle's
    truth-model replay fed the returned draws' parameters, the restatement's noise and the set's weights matches x_final
    to 1e-10 with the same slew time; the limit binds in at least one case."""
    import dispersion_ref as DR
    e = sweep_ensemble()
    n = len(e["x0"])
    cfg = e["cfg"]
    out, _ = run(engine, e, 8, keep=1)
    tr = engine.mc_trajectories(n)
    ko, ro = tr["knot_offs"], tr["row_offs"]
    act = np.nonzero(out["status"] != 5)[0]
    longest = act[np.argmax(out["N"][act])]
    seed = int(cfg.tvlqr.seed)
    sets = four_sets(cfg)[[0, 2, 3]]
    o, _ = S.tvlqr_opts_pair(noise_mode=1, seed=seed, R=float(cfg.tvlqr.Rd[0]))
    bound = 0
    for t, r in ((longest, 1), (act[0], 2**30 - 1)):
        _, _, p = engine.mc_dispersion_ensemble(n, 1, r_first=r, trials=[t], want_params=True, **ALL)
        sid = int(e["sid"][t])
        N = int(out["N"][t])
        s = types.SimpleNamespace(B=np.ascontiguousarray(tr["B_eci"][ro[t]:ro[t] + 2 * N]), index_scale=float(N),
                                  clock_rate=1.0 / (cfg.tf - cfg.t0), J=e["J"], t_final=float(out["t_final"][t]), N=N, xf=e["xf"][t])
        x0 = RE.x0_lqr(e["x0"][t], RE.initial_qnoise(seed, sid, r, QS))
        nz = RE.noise_array(seed, sid, N, r)
        rows = {}
        for u in (0.0, 1.0):
            slew, xf = engine.mc_weight_ensemble(n, 1, sets, u, ALL, r_first=r, trials=[t], want_x_final=True)
            rows[u] = xf
            for w in range(len(sets)):
                a, ns, slew_a = WR.oracle_truth_weighted(s, tr["X"][ko[t]:ko[t + 1]], tr["U"][ko[t]:ko[t + 1] - 1], x0, o, p[0, 0], nz,
                                                         sets[w], u)
                assert np.max(np.abs(xf[0, w, 0] - a[ns - 1])) <= 1e-10, (t, r, w, u)
                assert slew[0, w, 0] == slew_a, (t, r, w, u, slew[0, w, 0], slew_a)
        bound += int(np.sum(np.any(rows[0.0] != rows[1.0], axis=-1)))
    assert bound >= 1


def test_we5_call_shape(engine):
    """Rows are bit-equal under a permutation of the sets, a subset of them, chunking by r_first, and repeated,
    reordered trials; with and without the limit."""
    e = sweep_ensemble()
    n = len(e["x0"])
    run(engine, e, 8, keep=1)
    sets = four_sets(e["cfg"])
    for u in (0.0, 1.0):
        s, x = engine.mc_weight_ensemble(n, 64, sets, u, ALL, want_x_final=True)
        perm = [3, 1, 0, 2]
        sp, xp = engine.mc_weight_ensemble(n, 64, sets[perm], u, ALL, want_x_final=True)
        assert sp.tobytes() == s[:, perm].tobytes() and xp.tobytes() == x[:, perm].tobytes()
        ss, xs = engine.mc_weight_ensemble(n, 64, sets[[2]], u, ALL, want_x_final=True)
        assert ss.tobytes() == s[:, [2]].tobytes() and xs.tobytes() == x[:, [2]].tobytes()
        s1, x1 = engine.mc_weight_ensemble(n, 40, sets, u, ALL, want_x_final=True)
        s2, x2 = engine.mc_weight_ensemble(n, 24, sets, u, ALL, r_first=40, want_x_final=True)
        assert np.concatenate([s1, s2], 2).tobytes() == s.tobytes() and np.concatenate([x1, x2], 2).tobytes() == x.tobytes()
        sel = [4, 0, 3, 0, 1]
        st, xt = engine.mc_weight_ensemble(n, 64, sets, u, ALL, trials=sel, want_x_final=True)
        assert st.tobytes() == s[sel].tobytes() and xt.tobytes() == x[sel].tobytes()
        st2, _ = engine.mc_weight_ensemble(n, 64, sets, u, ALL, trials=sel)
        assert st2.tobytes() == st.tobytes()


def test_we6_isolation(engine):
    """The kept arrays are byte-identical before and after a weight call; following replay and dispersion ensembles
    return the rows of ones before it, and a following continuation the records of one without it."""
    e = shared_ensemble()
    n = len(e["x0"])
    run(engine, e, 4, keep=2)
    tr1 = snapshot(engine, n)
    ens1, xe1 = engine.mc_replay_ensemble(n, 40, want_x_final=True)
    dis1, xd1, _ = engine.mc_dispersion_ensemble(n, 40, want_x_final=True, **ALL)
    outa, _ = engine.mc_continue(n, cont_opts(e, 7))
    run(engine, e, 4, keep=2)
    engine.mc_weight_ensemble(n, 96, four_sets(e["cfg"]), 1.0, ALL, want_x_final=True)
    tr2 = snapshot(engine, n)
    for k in ("X", "U", "X_sim", "U_sim", "B_eci", "lam", "state"):
        assert tr2[k].tobytes() == tr1[k].tobytes(), k
    ens2, xe2 = engine.mc_replay_ensemble(n, 40, want_x_final=True)
    assert ens2.tobytes() == ens1.tobytes() and xe2.tobytes() == xe1.tobytes()
    dis2, xd2, _ = engine.mc_dispersion_ensemble(n, 40, want_x_final=True, **ALL)
    assert dis2.tobytes() == dis1.tobytes() and xd2.tobytes() == xd1.tobytes()
    outb, _ = engine.mc_continue(n, cont_opts(e, 7))
    assert outb.tobytes() == outa.tobytes()


def test_errors_leave_the_outputs_untouched(engine):
    """TS_ERR_ARG (-2), every output untouched: the cases of ts_mc_dispersion_ensemble (the sigma checks with a non-null
    disp), n_sets < 1, a null sets, a negative or non-finite Qd / Qfd entry, a non-positive or non-finite Rd entry, a
    negative or non-finite u_limit."""
    import tortoisesat.jl_b200 as tb
    from tortoisesat.jl_b200 import host
    e = shared_ensemble(n=4)
    n = 4
    good = four_sets(e["cfg"])

    def call(eng, nn, n_real=2, r_first=0, trials=None, opts=True, slew=True, disp=(0.1, 0.1, 0.1, 0.1), sets=good, n_sets=None,
             u_limit=0.0):
        o = host.ReplayEnsembleOpts(n_real, r_first, QS)
        d = None if disp is None else host.DispersionOpts(*disp)
        ws = None if sets is None else host.weight_sets(sets)
        k = len(good) if n_sets is None else n_sets
        ns = nn if trials is None else len(trials)
        sl = np.full((ns, max(k, 1), max(n_real, 1)), 7.0)
        xf = np.full((ns, max(k, 1), max(n_real, 1), 8), 7.0)
        sel = None if trials is None else np.asarray(trials, dtype=np.int64)
        rc = eng.lib.ts_mc_weight_ensemble(eng.h, nn, C.byref(o) if opts else None, None if d is None else C.byref(d), k, ws, u_limit,
                                           ns, None if sel is None else sel.ctypes.data, sl.ctypes.data if slew else None, xf.ctypes.data)
        assert np.all(sl == 7.0) and np.all(xf == 7.0)
        return rc
    fresh = tb.Engine(0)
    assert call(fresh, n) == -2
    fresh.close()
    run(engine, e, 4, keep=0)
    assert call(engine, n) == -2
    run(engine, e, 4, keep=1)
    assert call(engine, n + 1) == -2
    assert call(engine, n, n_real=0) == -2
    assert call(engine, n, r_first=-1) == -2
    assert call(engine, n, n_real=2, r_first=2**30 - 1) == -2
    assert call(engine, n, trials=[0, 4]) == -2
    assert call(engine, n, trials=[-1]) == -2
    assert call(engine, n, opts=False) == -2
    assert call(engine, n, slew=False) == -2
    for k in range(4):
        for bad in (-1e-3, math.inf, math.nan, (1.0 + 1e-12) if k < 3 else math.pi * (1 + 1e-12)):
            sg = [0.1] * 4
            sg[k] = bad
            assert call(engine, n, disp=tuple(sg)) == -2, (k, bad)
    assert call(engine, n, n_sets=0) == -2
    assert call(engine, n, n_sets=-1) == -2
    assert call(engine, n, sets=None) == -2
    for col in (0, 5, 6, 11):
        for bad in (-1e-3, math.inf, math.nan):
            s = good.copy()
            s[2, col] = bad
            assert call(engine, n, sets=s) == -2, (col, bad)
    for col in (12, 14):
        for bad in (0.0, -1.0, math.inf, math.nan):
            s = good.copy()
            s[3, col] = bad
            assert call(engine, n, sets=s) == -2, (col, bad)
    for bad in (-1e-3, math.inf, math.nan):
        assert call(engine, n, u_limit=bad) == -2, bad
    # the edges that are accepted: zero Q / Qf entries, a null disp
    s = good.copy()
    s[0, 0:12] = 0.0
    sl, _ = engine.mc_weight_ensemble(n, 2, s, 1.0, None)
    assert sl.shape == (4, 4, 2) and np.all(np.isfinite(sl))


def test_multi_gpu_rows_equal_single(engine):
    """MultiEngine([0]) and, with two or more GPUs, MultiEngine([0, 1]): the rows equal the single-engine rows."""
    import torch
    from tortoisesat.jl_b200 import host
    e = shared_ensemble(n=10, seed=5)
    n = 10
    run(engine, e, 4, keep=1)
    sel = [9, 2, 5, 2, 0, 7]
    sets = four_sets(e["cfg"])
    ref = engine.mc_weight_ensemble(n, 40, sets, 1.0, ALL, trials=sel, want_x_final=True)
    cfg = e["cfg"]
    devsets = [[0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for devs in devsets:
        m = host.MultiEngine(devs)
        m.monte_carlo_run(cfg, e["kep"], e["fo"], e["x0"], e["xf"], e["Jm"], q_noise0=e["qn"], stream_id=e["sid"])
        got = m.mc_weight_ensemble(n, 40, sets, 1.0, ALL, trials=sel, want_x_final=True)
        m.close()
        for a, b in zip(got, ref):
            assert a.tobytes() == b.tobytes(), devs
    if len(devsets) == 1:
        pytest.skip("one GPU: the two-device comparison needs two")


def test_weight_ensemble_wrapper():
    """weight_ensemble on a monte_carlo() result: r_first = 1 by default, the documented shapes and per-set statistics."""
    import inspect
    from tortoisesat.jl_b200 import host
    assert inspect.signature(host.weight_ensemble).parameters["r_first"].default == 1
    o = host.default_ilqr_opts()
    o.max_outer = 5
    res = host.monte_carlo(number_sims=4, seed=3, ilqr=o)
    w = WR.run_weights(host.default_tvlqr_opts())
    sets = np.stack([w, WR.scaled(w, r=0.1), WR.scaled(w, q=10.0)])
    d = host.weight_ensemble(res, sets, n_real=24, u_limit=1.0, **ALL)
    out = res["outcomes"]
    assert d["slew_time"].shape == (4, 3, 24) and d["fails"].shape == (4, 3, 24)
    for k in ("fail_rate", "slew_mean", "slew_std"):
        assert d[k].shape == (4, 3), k
    assert d["set_fail_rate"].shape == (3,)
    s, _ = host.default_engine().mc_weight_ensemble(4, 24, sets, 1.0, ALL, r_first=1)
    assert d["slew_time"].tobytes() == s.tobytes()
    act = out["status"] != 5
    assert np.array_equal(d["fails"], d["slew_time"] == out["t_final"][:, None, None])
    assert np.allclose(d["fail_rate"][act], d["fails"][act].mean(axis=2))
    assert np.allclose(d["set_fail_rate"], d["fails"][act].mean(axis=(0, 2)))
