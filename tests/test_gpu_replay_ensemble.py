"""GPU: disturbance ensembles of a kept Monte-Carlo run (ts_mc_replay_ensemble, ts_multi_mc_replay_ensemble; rules
RE1-RE5 of DESIGN.md section 4, K4) against the kept replay, the CPU oracle fed the same draws, other call shapes and a
following continuation."""
import ctypes as C
import math
import types

import numpy as np
import pytest

import replay_ensemble_ref as RE
import slew_setup as S
from test_gpu_mc_continue import J_GEN, cont_opts, run, shared_ensemble, snapshot, sweep_ensemble

pytestmark = pytest.mark.gpu
QS = (math.pi / 180) ** 2


def n_sim(cfg, tf, N):
    """N_sim of the replay (tvlqr_replay_src): length(t0:dt:tf), capped at N."""
    rl = lambda a, st, b: 0 if b < a else int(math.floor((b - a) / st + 1e-9)) + 1
    ns = rl(cfg.t0, cfg.dt, tf)
    if ns > N:
        ns = rl(cfg.t0, cfg.dt, tf - cfg.dt)
    return min(ns, N)


def assert_re3(engine, e, out, n):
    """Realisation 0 of every trial is the kept replay: its slew_time and X_sim row N_sim - 1, bit for bit; a NO_CUTOFF
    trial has NaN rows."""
    tr = engine.mc_trajectories(n, want=("X_sim",))
    slew, xf = engine.mc_replay_ensemble(n, 3, want_x_final=True)
    ko = tr["knot_offs"]
    cfg = e["cfg"]
    for t in range(n):
        if out["status"][t] == 5:
            assert np.all(np.isnan(slew[t])) and np.all(np.isnan(xf[t]))
            continue
        assert slew[t, 0] == out["slew_time"][t], (t, slew[t, 0], out["slew_time"][t])
        ns = n_sim(cfg, out["t_final"][t], int(out["N"][t]))
        assert xf[t, 0].tobytes() == tr["X_sim"][ko[t] + ns - 1].tobytes(), t
        assert np.all(tr["X_sim"][ko[t] + ns:ko[t + 1]] == 0.0)
        assert not np.array_equal(xf[t, 1], xf[t, 2])
    assert engine.last_kernel_ms() > 0
    g, r = engine.mc_replay_ensemble_split()
    assert g > 0 and r > 0


@pytest.mark.parametrize("quat,J", [(0, "diag"), (1, "diag"), (0, "general")])
def test_re3_fixed_orbit(engine, quat, J):
    e = shared_ensemble(J=S.J_1U if J == "diag" else J_GEN)
    n = len(e["x0"])
    out, _ = run(engine, e, 5, keep=1, quat=quat)
    assert_re3(engine, e, out, n)


def test_re3_sweep_and_after_a_continuation(engine):
    """The sweep (ragged horizons, one NO_CUTOFF trial) kept with keep_trajectories = 1 and = 2, and after a continuation
    20 -> 30 against the continued records."""
    e = sweep_ensemble()
    n = len(e["x0"])
    out, _ = run(engine, e, 20, keep=1)
    assert (out["status"] == 5).sum() == 1
    assert_re3(engine, e, out, n)
    run(engine, e, 20, keep=2)
    out2, _ = engine.mc_continue(n, cont_opts(e, 30))
    assert_re3(engine, e, out2, n)


def test_oracle_for_later_realisations(engine):
    """(trial, r) pairs with r >= 1 up to 2^30 - 1 against the oracle fed the restatement's draws (explicit noise array)
    and initial state, on the fetched X, U and field table: x_final to 1e-10, the same slew time.  With q_noise_scale = 0
    a realisation starts from the unperturbed x0."""
    e = sweep_ensemble()
    n = len(e["x0"])
    cfg = e["cfg"]
    out, _ = run(engine, e, 8, keep=1)
    tr = engine.mc_trajectories(n)
    ko, ro = tr["knot_offs"], tr["row_offs"]
    act = np.nonzero(out["status"] != 5)[0]
    pairs = [(act[0], 1), (act[1], 5), (act[-1], 2**30 - 1), (act[0], 2**30 - 2)]
    o, _ = S.tvlqr_opts_pair(noise_mode=1, seed=int(cfg.tvlqr.seed), R=float(cfg.tvlqr.Rd[0]))
    for scale in (QS, 0.0):
        for t, r in pairs:
            slew, xf = engine.mc_replay_ensemble(n, 1, r_first=r, trials=[t], q_noise_scale=scale, want_x_final=True)
            N = int(out["N"][t])
            s = types.SimpleNamespace(B=np.ascontiguousarray(tr["B_eci"][ro[t]:ro[t] + 2 * N]), index_scale=float(N),
                                      clock_rate=1.0 / (cfg.tf - cfg.t0), J=e["J"], t_final=float(out["t_final"][t]), N=N,
                                      xf=e["xf"][t])
            sid = int(e["sid"][t])
            x0 = RE.x0_lqr(e["x0"][t], RE.initial_qnoise(int(cfg.tvlqr.seed), sid, r, scale))
            if scale == 0.0:
                assert np.array_equal(x0[:7], e["x0"][t, :7])
            nz = RE.noise_array(int(cfg.tvlqr.seed), sid, N, r)
            a = S.oracle_tvlqr(s, tr["X"][ko[t]:ko[t + 1]], tr["U"][ko[t]:ko[t + 1] - 1], x0, o, trial=sid, noise=nz)
            assert np.max(np.abs(xf[0, 0] - a[0][a[4] - 1])) <= 1e-10, (t, r, scale)
            assert slew[0, 0] == a[5], (t, r, scale, slew[0, 0], a[5])
            if scale == 0.0:
                break


def test_re4_call_shape(engine):
    """[0, 64) in one call equals [0, 40) + [40, 64); a permuted subset with a repeated trial equals the matching rows of
    the all-trials call; realisations r >= 1 give pairwise distinct final states."""
    e = sweep_ensemble()
    n = len(e["x0"])
    run(engine, e, 8, keep=1)
    s, x = engine.mc_replay_ensemble(n, 64, want_x_final=True)
    s1, x1 = engine.mc_replay_ensemble(n, 40, want_x_final=True)
    s2, x2 = engine.mc_replay_ensemble(n, 24, r_first=40, want_x_final=True)
    assert np.concatenate([s1, s2], 1).tobytes() == s.tobytes() and np.concatenate([x1, x2], 1).tobytes() == x.tobytes()
    sel = [4, 0, 3, 0, 1]
    sp, xp = engine.mc_replay_ensemble(n, 64, trials=sel, want_x_final=True)
    assert sp.tobytes() == s[sel].tobytes() and xp.tobytes() == x[sel].tobytes()
    sp2, _ = engine.mc_replay_ensemble(n, 64, trials=sel)
    assert sp2.tobytes() == sp.tobytes()
    for t in (0, 1, 3, 4):
        f = x[t, 1:].reshape(63, 8)
        assert len({row.tobytes() for row in f}) == 63


def test_re5_isolation(engine):
    """The kept arrays are byte-identical before and after an ensemble call, and a following continuation gives the
    records of one without the ensemble in between."""
    e = shared_ensemble()
    n = len(e["x0"])
    run(engine, e, 4, keep=2)
    tr1 = snapshot(engine, n)
    outa, _ = engine.mc_continue(n, cont_opts(e, 7))
    run(engine, e, 4, keep=2)
    engine.mc_replay_ensemble(n, 96, want_x_final=True)
    tr2 = snapshot(engine, n)
    for k in ("X", "U", "X_sim", "U_sim", "B_eci", "lam", "state"):
        assert tr2[k].tobytes() == tr1[k].tobytes(), k
    outb, _ = engine.mc_continue(n, cont_opts(e, 7))
    assert outb.tobytes() == outa.tobytes()


def test_errors_leave_the_outputs_untouched(engine):
    """TS_ERR_ARG (-2), outputs untouched: no kept run (fresh engine; last run with keep_trajectories = 0), wrong
    n_trials, n_real < 1, r_first < 0, r_first + n_real > 2^30, a trial out of range, null opts or slew_time."""
    import tortoisesat.jl_b200 as tb
    from tortoisesat.jl_b200 import host
    e = shared_ensemble(n=4)
    n = 4

    def call(eng, nn, n_real=2, r_first=0, trials=None, opts=True, slew=True):
        o = host.ReplayEnsembleOpts(n_real, r_first, QS)
        ns = nn if trials is None else len(trials)
        sl = np.full((ns, max(n_real, 1)), 7.0)
        xf = np.full((ns, max(n_real, 1), 8), 7.0)
        sel = None if trials is None else np.asarray(trials, dtype=np.int64)
        rc = eng.lib.ts_mc_replay_ensemble(eng.h, nn, C.byref(o) if opts else None, ns, None if sel is None else sel.ctypes.data,
                                           sl.ctypes.data if slew else None, xf.ctypes.data)
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
    s, _ = engine.mc_replay_ensemble(n, 2, r_first=2**30 - 2)
    assert s.shape == (4, 2) and np.all(np.isfinite(s))


def test_multi_gpu_rows_equal_single(engine):
    """MultiEngine([0]) and, with two or more GPUs, MultiEngine([0, 1]): the rows equal the single-engine rows."""
    import torch
    from tortoisesat.jl_b200 import host
    e = shared_ensemble(n=10, seed=5)
    n = 10
    run(engine, e, 4, keep=1)
    sel = [9, 2, 5, 2, 0, 7]
    ref, xref = engine.mc_replay_ensemble(n, 40, trials=sel, want_x_final=True)
    cfg = e["cfg"]
    devsets = [[0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for devs in devsets:
        m = host.MultiEngine(devs)
        m.monte_carlo_run(cfg, e["kep"], e["fo"], e["x0"], e["xf"], e["Jm"], q_noise0=e["qn"], stream_id=e["sid"])
        s, x = m.mc_replay_ensemble(n, 40, trials=sel, want_x_final=True)
        m.close()
        assert s.tobytes() == ref.tobytes() and x.tobytes() == xref.tobytes(), devs
    if len(devsets) == 1:
        pytest.skip("one GPU: the two-device comparison needs two")


def test_replay_ensemble_wrapper():
    """replay_ensemble on a monte_carlo() result: the documented shapes, fails == (slew_time == t_final), a fail_rate
    consistent with fails, and realisation 0 = the run's slew times."""
    from tortoisesat.jl_b200 import host
    o = host.default_ilqr_opts()
    o.max_outer = 5
    res = host.monte_carlo(number_sims=4, seed=3, ilqr=o)
    ens = host.replay_ensemble(res, n_real=40)
    out = res["outcomes"]
    assert ens["slew_time"].shape == (4, 40) and ens["fails"].shape == (4, 40) and ens["fail_rate"].shape == (4,)
    assert np.array_equal(ens["trials"], np.arange(4))
    act = out["status"] != 5
    assert np.array_equal(ens["slew_time"][act, 0], out["slew_time"][act])
    assert np.array_equal(ens["fails"], ens["slew_time"] == out["t_final"][:, None])
    assert np.allclose(ens["fail_rate"][act], ens["fails"][act].mean(axis=1))
    ok = ~ens["fails"][act]
    for k, t in enumerate(np.nonzero(act)[0]):
        if ok[k].any():
            assert np.isclose(ens["slew_mean"][t], ens["slew_time"][t][ok[k]].mean())
            assert np.isclose(ens["slew_std"][t], ens["slew_time"][t][ok[k]].std())
    sub = host.replay_ensemble(res, n_real=8, trials=[2, 0])
    assert sub["slew_time"].shape == (2, 8) and np.array_equal(sub["slew_time"], ens["slew_time"][[2, 0], :8])
