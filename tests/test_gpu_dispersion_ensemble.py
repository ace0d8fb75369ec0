"""GPU: dispersion ensembles of a kept Monte-Carlo run (ts_mc_dispersion_ensemble, ts_multi_mc_dispersion_ensemble;
rules DE1-DE6 of DESIGN.md section 4, K4) against the disturbance ensemble, the kept replay, the numpy restatement of
the draws, the CPU oracle's truth-model replay fed the same parameters and draws, other call shapes and later calls."""
import ctypes as C
import math
import types

import numpy as np
import pytest

import dispersion_ref as DR
import replay_ensemble_ref as RE
import slew_setup as S
from test_gpu_mc_continue import J_GEN, cont_opts, run, shared_ensemble, snapshot, sweep_ensemble

pytestmark = pytest.mark.gpu
QS = (math.pi / 180) ** 2
ALL = dict(sigma_inertia=0.2, sigma_torquer=0.1, sigma_field_scale=0.05, sigma_field_angle=math.radians(5.0))
GROUPS = {"inertia": dict(sigma_inertia=0.2), "torquer": dict(sigma_torquer=0.1), "field_scale": dict(sigma_field_scale=0.05),
          "field_angle": dict(sigma_field_angle=math.radians(5.0)), "all": ALL}
NOMINAL = np.array([1.0] * 7 + [0.0] * 3)


def sig4(sg):
    return tuple(float(sg.get(k, 0.0)) for k in ("sigma_inertia", "sigma_torquer", "sigma_field_scale", "sigma_field_angle"))


def n_sim(cfg, tf, N):
    """N_sim of the replay (tvlqr_replay_src): length(t0:dt:tf), capped at N."""
    rl = lambda a, st, b: 0 if b < a else int(math.floor((b - a) / st + 1e-9)) + 1
    ns = rl(cfg.t0, cfg.dt, tf)
    if ns > N:
        ns = rl(cfg.t0, cfg.dt, tf - cfg.dt)
    return min(ns, N)


def assert_de4(engine, n, out, n_real=40):
    """All sigmas 0: every row equals ts_mc_replay_ensemble's, bit for bit; the parameters are nominal (NaN rows for a
    NO_CUTOFF trial)."""
    s0, x0 = engine.mc_replay_ensemble(n, n_real, want_x_final=True)
    s, x, p = engine.mc_dispersion_ensemble(n, n_real, want_x_final=True, want_params=True)
    assert s.tobytes() == s0.tobytes() and x.tobytes() == x0.tobytes()
    for t in range(n):
        if out["status"][t] == 5:
            assert np.all(np.isnan(p[t]))
        else:
            assert np.all(p[t] == NOMINAL)
    g, r = engine.mc_replay_ensemble_split()
    assert g > 0 and r > 0 and engine.last_kernel_ms() > 0


@pytest.mark.parametrize("quat,J", [(0, "diag"), (1, "diag"), (0, "general")])
def test_de4_fixed_orbit(engine, quat, J):
    e = shared_ensemble(J=S.J_1U if J == "diag" else J_GEN)
    n = len(e["x0"])
    out, _ = run(engine, e, 5, keep=1, quat=quat)
    assert_de4(engine, n, out)


def test_de4_sweep(engine):
    """The sweep (ragged horizons, one NO_CUTOFF trial)."""
    e = sweep_ensemble()
    n = len(e["x0"])
    out, _ = run(engine, e, 8, keep=1)
    assert (out["status"] == 5).sum() == 1
    assert_de4(engine, n, out)


def assert_de3(engine, e, out, n):
    tr = engine.mc_trajectories(n, want=("X_sim",))
    ko = tr["knot_offs"]
    slew, xf, p = engine.mc_dispersion_ensemble(n, 3, want_x_final=True, want_params=True, **ALL)
    for t in range(n):
        if out["status"][t] == 5:
            assert np.all(np.isnan(slew[t])) and np.all(np.isnan(xf[t])) and np.all(np.isnan(p[t]))
            continue
        assert slew[t, 0] == out["slew_time"][t], t
        ns = n_sim(e["cfg"], out["t_final"][t], int(out["N"][t]))
        assert xf[t, 0].tobytes() == tr["X_sim"][ko[t] + ns - 1].tobytes(), t
        assert np.all(p[t, 0] == NOMINAL) and np.all(p[t, 1:] != NOMINAL)


def test_de3_sweep_and_after_a_continuation(engine):
    """Realisation 0 is the kept record with every sigma > 0: kept with keep_trajectories = 1, and after a continuation
    20 -> 30 against the continued records."""
    e = sweep_ensemble()
    n = len(e["x0"])
    out, _ = run(engine, e, 20, keep=1)
    assert_de3(engine, e, out, n)
    run(engine, e, 20, keep=2)
    out2, _ = engine.mc_continue(n, cont_opts(e, 30))
    assert_de3(engine, e, out2, n)


def test_oracle_for_each_group(engine):
    """(trial, r) pairs on the sweep -- the longest slew, r = 2^30 - 1 -- for each group alone and all together: params
    equal the restatement to 1e-14, and the oracle's truth-model replay fed the returned params and the restatement's
    draws matches x_final to 1e-10 with the same slew time."""
    e = sweep_ensemble()
    n = len(e["x0"])
    cfg = e["cfg"]
    out, _ = run(engine, e, 8, keep=1)
    tr = engine.mc_trajectories(n)
    ko, ro = tr["knot_offs"], tr["row_offs"]
    act = np.nonzero(out["status"] != 5)[0]
    longest = act[np.argmax(out["N"][act])]
    pairs = [(longest, 1), (act[0], 2**30 - 1), (act[1], 6)]
    seed = int(cfg.tvlqr.seed)
    o, _ = S.tvlqr_opts_pair(noise_mode=1, seed=seed, R=float(cfg.tvlqr.Rd[0]))
    moved = 0
    for name, sg in GROUPS.items():
        for t, r in pairs:
            slew, xf, p = engine.mc_dispersion_ensemble(n, 1, r_first=r, trials=[t], want_x_final=True, want_params=True, **sg)
            sid = int(e["sid"][t])
            assert np.allclose(p[0, 0], DR.dispersion_params(seed, sid, r, sig4(sg)), rtol=1e-14, atol=1e-14), (name, t, r)
            N = int(out["N"][t])
            s = types.SimpleNamespace(B=np.ascontiguousarray(tr["B_eci"][ro[t]:ro[t] + 2 * N]), index_scale=float(N),
                                      clock_rate=1.0 / (cfg.tf - cfg.t0), J=e["J"], t_final=float(out["t_final"][t]), N=N,
                                      xf=e["xf"][t])
            x0 = RE.x0_lqr(e["x0"][t], RE.initial_qnoise(seed, sid, r, QS))
            nz = RE.noise_array(seed, sid, N, r)
            a, ns, slew_a = DR.oracle_truth(s, tr["X"][ko[t]:ko[t + 1]], tr["U"][ko[t]:ko[t + 1] - 1], x0, o, p[0, 0], nz)
            assert np.max(np.abs(xf[0, 0] - a[ns - 1])) <= 1e-10, (name, t, r)
            assert slew[0, 0] == slew_a, (name, t, r, slew[0, 0], slew_a)
            s0, x00 = engine.mc_replay_ensemble(n, 1, r_first=r, trials=[t], want_x_final=True)
            moved += int(np.max(np.abs(x00[0, 0] - xf[0, 0])) > 1e-9)
    assert moved == len(GROUPS) * len(pairs)


def test_de5_call_shape(engine):
    """[0, 64) in one call equals [0, 40) + [40, 64); a permuted subset with a repeated trial equals the matching rows of
    the all-trials call."""
    e = sweep_ensemble()
    n = len(e["x0"])
    run(engine, e, 8, keep=1)
    s, x, p = engine.mc_dispersion_ensemble(n, 64, want_x_final=True, want_params=True, **ALL)
    s1, x1, p1 = engine.mc_dispersion_ensemble(n, 40, want_x_final=True, want_params=True, **ALL)
    s2, x2, p2 = engine.mc_dispersion_ensemble(n, 24, r_first=40, want_x_final=True, want_params=True, **ALL)
    assert np.concatenate([s1, s2], 1).tobytes() == s.tobytes() and np.concatenate([x1, x2], 1).tobytes() == x.tobytes()
    assert np.concatenate([p1, p2], 1).tobytes() == p.tobytes()
    sel = [4, 0, 3, 0, 1]
    sp, xp, pp = engine.mc_dispersion_ensemble(n, 64, trials=sel, want_x_final=True, want_params=True, **ALL)
    assert sp.tobytes() == s[sel].tobytes() and xp.tobytes() == x[sel].tobytes() and pp.tobytes() == p[sel].tobytes()
    sp2, _, _ = engine.mc_dispersion_ensemble(n, 64, trials=sel, **ALL)
    assert sp2.tobytes() == sp.tobytes()


def test_de6_isolation(engine):
    """The kept arrays are byte-identical before and after a dispersion call; a following ts_mc_replay_ensemble returns
    the rows of one before it, and a following continuation the records of one without it."""
    e = shared_ensemble()
    n = len(e["x0"])
    run(engine, e, 4, keep=2)
    tr1 = snapshot(engine, n)
    ens1, xe1 = engine.mc_replay_ensemble(n, 40, want_x_final=True)
    outa, _ = engine.mc_continue(n, cont_opts(e, 7))
    run(engine, e, 4, keep=2)
    engine.mc_dispersion_ensemble(n, 96, want_x_final=True, want_params=True, **ALL)
    tr2 = snapshot(engine, n)
    for k in ("X", "U", "X_sim", "U_sim", "B_eci", "lam", "state"):
        assert tr2[k].tobytes() == tr1[k].tobytes(), k
    ens2, xe2 = engine.mc_replay_ensemble(n, 40, want_x_final=True)
    assert ens2.tobytes() == ens1.tobytes() and xe2.tobytes() == xe1.tobytes()
    outb, _ = engine.mc_continue(n, cont_opts(e, 7))
    assert outb.tobytes() == outa.tobytes()


def test_errors_leave_the_outputs_untouched(engine):
    """TS_ERR_ARG (-2), every output untouched: the cases of ts_mc_replay_ensemble, a null disp, a negative, infinite or
    NaN sigma, a log-sigma above 1 and a field angle above pi."""
    import tortoisesat.jl_b200 as tb
    from tortoisesat.jl_b200 import host
    e = shared_ensemble(n=4)
    n = 4

    def call(eng, nn, n_real=2, r_first=0, trials=None, opts=True, slew=True, disp=(0.1, 0.1, 0.1, 0.1)):
        o = host.ReplayEnsembleOpts(n_real, r_first, QS)
        d = None if disp is None else host.DispersionOpts(*disp)
        ns = nn if trials is None else len(trials)
        sl = np.full((ns, max(n_real, 1)), 7.0)
        xf = np.full((ns, max(n_real, 1), 8), 7.0)
        pr = np.full((ns, max(n_real, 1), 10), 7.0)
        sel = None if trials is None else np.asarray(trials, dtype=np.int64)
        rc = eng.lib.ts_mc_dispersion_ensemble(eng.h, nn, C.byref(o) if opts else None, None if d is None else C.byref(d), ns,
                                               None if sel is None else sel.ctypes.data, sl.ctypes.data if slew else None,
                                               xf.ctypes.data, pr.ctypes.data)
        assert np.all(sl == 7.0) and np.all(xf == 7.0) and np.all(pr == 7.0)
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
    assert call(engine, n, disp=None) == -2
    for k in range(4):
        for bad in (-1e-3, math.inf, math.nan, (1.0 + 1e-12) if k < 3 else math.pi * (1 + 1e-12)):
            sg = [0.1] * 4
            sg[k] = bad
            assert call(engine, n, disp=tuple(sg)) == -2, (k, bad)
    s, _, p = engine.mc_dispersion_ensemble(n, 2, r_first=2**30 - 2, sigma_inertia=1.0, sigma_torquer=1.0, sigma_field_scale=1.0,
                                            sigma_field_angle=math.pi, want_params=True)
    assert s.shape == (4, 2) and np.all(np.isfinite(s)) and np.all(np.isfinite(p))


def test_multi_gpu_rows_equal_single(engine):
    """MultiEngine([0]) and, with two or more GPUs, MultiEngine([0, 1]): the rows equal the single-engine rows."""
    import torch
    from tortoisesat.jl_b200 import host
    e = shared_ensemble(n=10, seed=5)
    n = 10
    run(engine, e, 4, keep=1)
    sel = [9, 2, 5, 2, 0, 7]
    ref = engine.mc_dispersion_ensemble(n, 40, trials=sel, want_x_final=True, want_params=True, **ALL)
    cfg = e["cfg"]
    devsets = [[0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for devs in devsets:
        m = host.MultiEngine(devs)
        m.monte_carlo_run(cfg, e["kep"], e["fo"], e["x0"], e["xf"], e["Jm"], q_noise0=e["qn"], stream_id=e["sid"])
        got = m.mc_dispersion_ensemble(n, 40, trials=sel, want_x_final=True, want_params=True, **ALL)
        m.close()
        for a, b in zip(got, ref):
            assert a.tobytes() == b.tobytes(), devs
    if len(devsets) == 1:
        pytest.skip("one GPU: the two-device comparison needs two")


def test_dispersion_ensemble_wrapper():
    """dispersion_ensemble on a monte_carlo() result: r_first = 1 by default (the engine's rows from realisation 1), the
    documented shapes and statistics, params in DISPERSION_PARAMS order."""
    import inspect
    from tortoisesat.jl_b200 import host
    assert inspect.signature(host.dispersion_ensemble).parameters["r_first"].default == 1
    o = host.default_ilqr_opts()
    o.max_outer = 5
    res = host.monte_carlo(number_sims=4, seed=3, ilqr=o)
    d = host.dispersion_ensemble(res, n_real=24, **ALL)
    out = res["outcomes"]
    assert d["slew_time"].shape == (4, 24) and d["params"].shape == (4, 24, 10) and d["fail_rate"].shape == (4,)
    s, _, p = host.default_engine().mc_dispersion_ensemble(4, 24, r_first=1, want_params=True, **ALL)
    assert d["slew_time"].tobytes() == s.tobytes() and d["params"].tobytes() == p.tobytes()
    act = out["status"] != 5
    assert np.array_equal(d["fails"], d["slew_time"] == out["t_final"][:, None])
    assert np.allclose(d["fail_rate"][act], d["fails"][act].mean(axis=1))
    assert np.all(d["params"][act][..., :7] > 0) and np.all(d["params"][act][..., :7] != 1.0)
    assert host.DISPERSION_PARAMS[6] == "s_B"
