"""GPU: continuation of a kept Monte-Carlo run (ts_monte_carlo_run with keep_trajectories = 2, ts_mc_fetch_state,
ts_mc_continue, ts_multi_mc_continue; rules MC1-MC4 of DESIGN.md section 4, K3) against a keep_trajectories = 1 run,
the stand-alone continuation (ts_alilqr_solve_state_batch + ts_tvlqr_sim_batch), the CPU oracle's per-trial pipeline and
a direct run to the larger max_outer."""
import concurrent.futures as cf
import ctypes as C
import math

import numpy as np
import pytest

import alilqr_state as AS
import slew_setup as S
from oracle import oracle as orc
from test_gpu_mc import _perturb

pytestmark = pytest.mark.gpu
GM = S.GM
K3_FIELDS = ("status", "outer_iters", "inner_iters", "ls_rollouts", "N", "J", "c_max")
J_GEN = np.array([[2e-3, 1e-4, 0], [1e-4, 3e-3, 2e-4], [0, 2e-4, 1e-3]])


def shared_ensemble(n=6, J=S.J_1U, seed=21):
    """configs[2] in miniature: one fixed LEO orbit (N = 2044 knots), random attitudes."""
    from tortoisesat.jl_b200 import host
    rng = np.random.default_rng(seed)
    cfg = host.default_mc_config(n, shared_orbit=True, run_tvlqr=True, tf=2400.0, cutoff=30.0, alpha=0.1)
    cfg.tvlqr.noise_mode, cfg.tvlqr.seed = 2, 4242
    kep = np.array([[0, 6771.0, 96.6, 0.0, 0.0, 90.0]])
    fo = np.zeros(1, dtype=host.FIELD_OPTS_DTYPE)
    fo[0] = (GM, 58155.0, 2019.0, 6771000.0, 0, 0, 0)
    qf = np.array([math.sqrt(2) / 2, math.sqrt(2) / 2, 0, 0])
    x0 = np.zeros((n, 8))
    xf = np.tile(np.concatenate([[0, 0, 0], qf, [1.0]]), (n, 1))
    for t in range(n):
        dq = S.quat_axis_angle(rng.normal(size=3), rng.uniform(5, 40))
        q = np.zeros(4)
        orc.lib().orc_qmult(orc.P(orc.f64(qf)), orc.P(dq), orc.P(q))
        x0[t, 3:7] = q
    Jm = np.tile(np.asarray(J).reshape(-1), (n, 1))
    qn = rng.normal(size=(n, 3)) * (math.pi / 180) ** 2
    return dict(cfg=cfg, kep=kep, fo=fo, x0=x0, xf=xf, Jm=Jm, J=np.asarray(J), qn=qn, sid=np.arange(100, 100 + n).astype(np.uint32))


def sweep_ensemble():
    """Per-trial orbits (horizons of about 1100-1900 knots); trial 2 is equatorial and never reaches the cutoff within the
    scoping window (NO_CUTOFF)."""
    from tortoisesat.jl_b200 import host
    rng = np.random.default_rng(1)
    n = 5
    cfg = host.default_mc_config(n, shared_orbit=False, run_tvlqr=True, tf=600.0, cutoff=30.0, alpha=0.1)
    cfg.tvlqr.noise_mode, cfg.tvlqr.seed = 2, 9
    kep = np.zeros((n, 6))
    fo = np.zeros(n, dtype=host.FIELD_OPTS_DTYPE)
    for t in range(n):
        alt = rng.uniform(350, 800)
        inc = 0.0 if t == 2 else rng.uniform(40, 98)
        kep[t] = [0, alt + 6371.0, inc, rng.uniform(0, 360), 0, rng.uniform(0, 360)]
        fo[t] = (GM, rng.uniform(58155, 58520), 2015 + 5 * rng.random(), (alt + 6371.0) * 1000, 0, 0, 0)
    qf = np.array([math.sqrt(2) / 2, math.sqrt(2) / 2, 0, 0])
    x0 = np.zeros((n, 8))
    xf = np.tile(np.concatenate([[0, 0, 0], qf, [1.0]]), (n, 1))
    for t in range(n):
        x0[t, 3:7] = S.quat_axis_angle(rng.normal(size=3), rng.uniform(10, 60))
    Jm = np.tile(S.J_1U.reshape(-1), (n, 1))
    qn = rng.normal(size=(n, 3)) * (math.pi / 180) ** 2
    return dict(cfg=cfg, kep=kep, fo=fo, x0=x0, xf=xf, Jm=Jm, J=S.J_1U, qn=qn, sid=np.arange(n).astype(np.uint32))


def run(eng, e, max_outer, keep=2, pair=2, quat=0, equal_tols=False, run_tvlqr=1):
    cfg = e["cfg"]
    cfg.keep_trajectories, cfg.run_tvlqr = keep, run_tvlqr
    cfg.ilqr.max_outer, cfg.ilqr.k3_pair, cfg.ilqr.quat_error = max_outer, pair, quat
    if equal_tols:
        cfg.ilqr.cost_tol_intermediate = cfg.ilqr.cost_tol   # CS4
    return eng.monte_carlo_run(cfg, e["kep"], e["fo"], e["x0"], e["xf"], e["Jm"], q_noise0=e["qn"], stream_id=e["sid"])


def cont_opts(e, max_outer):
    from tortoisesat.jl_b200 import host
    o = host.IlqrOpts.from_buffer_copy(e["cfg"].ilqr)
    o.max_outer = max_outer
    return o


def snapshot(eng, n, run_tvlqr=True):
    """every kept array: trajectories, field tables, state, multipliers"""
    tr = eng.mc_trajectories(n, want=("X", "U", "X_sim", "U_sim", "B_eci") if run_tvlqr else ("X", "U", "B_eci"))
    tr["state"], tr["lam"] = eng.mc_state(n)
    return tr


def stats_tuple(st, with_flops=True):
    f = ["n_trials", "n_converged", "n_no_cutoff", "n_fail_slew", "sum_slew_time", "sum_slew_time_sq", "sum_t_final",
         "sum_inner_iters", "sum_ls_rollouts", "sum_knots"] + (["flops"] if with_flops else [])
    return tuple(getattr(st, k) for k in f) + tuple(st.n_status)


def standalone(eng, e, out, tr, opts, state=None, lam=None, X=None, U=None):
    """ts_alilqr_solve_state_batch over the run's active trials, with the run's inputs: the fetched field tables at
    row_offs (2N rows per trial), weights rebuilt by ts_slew_weights_batch (the same k_slew_prep kernel)."""
    cfg = e["cfg"]
    act = np.nonzero(out["status"] != 5)[0]
    N = out["N"][act]
    ro = tr["row_offs"]
    tf = out["t_final"][act]
    Qd, Qfd, Rd = eng.slew_weights_batch(e["x0"][act], e["xf"][act], e["Jm"][act], tf, t0=cfg.t0, dt=cfg.dt, alpha=cfg.alpha,
                                         beta=cfg.beta, eigen_axis_fix=bool(cfg.eigen_axis_fix))
    kw = {} if state is None else dict(state=state[act], lam=lam, X=X, U=U)
    return act, eng.alilqr_solve_state_batch(N, e["x0"][act], e["xf"][act], e["Jm"][act], Qd, Qfd, Rd, tr["B_eci"], ro[act], 2 * N,
                                             N.astype(float), [1.0 / (cfg.tf - cfg.t0)] * len(act), cfg.dt, opts=opts, want_K=False,
                                             **kw)


def replay_standalone(eng, e, out, tr, idx):
    """ts_tvlqr_sim_batch on the kept X, U of trials idx, with the run's stream ids and options (fused-path overrides)."""
    from tortoisesat.jl_b200 import host
    cfg = e["cfg"]
    ko, ro = tr["knot_offs"], tr["row_offs"]
    N = out["N"][idx]
    X = np.concatenate([tr["X"][ko[t]:ko[t + 1]] for t in idx])
    U = np.concatenate([tr["U"][ko[t]:ko[t + 1]] for t in idx])
    x0l = []
    for t in idx:
        x = e["x0"][t].copy()
        x[3:7] = _perturb(e["x0"][t, 3:7], e["qn"][t])
        x[7] = 0
        x0l.append(x)
    g = host.TvlqrOpts.from_buffer_copy(cfg.tvlqr)
    g.dt, g.t0, g.literal_postproc = cfg.dt, cfg.t0, 0
    return eng.tvlqr_sim_batch(N, X, U, np.stack(x0l), e["Jm"][idx], tr["B_eci"], ro[idx], 2 * N, N.astype(float),
                               [1.0 / (cfg.tf - cfg.t0)] * len(idx), out["t_final"][idx], e["xf"][idx, 3:7], opts=g,
                               stream_id=e["sid"][idx])


@pytest.mark.parametrize("quat", [0, 1])
def test_keeping_changes_nothing(engine, quat):
    """keep_trajectories = 2 gives the records, statistics (ms_* apart) and kept arrays of keep_trajectories = 1; the
    fetched state repeats each record, lam >= 0 and each trial's last lam row is 0; a NO_CUTOFF trial gets a zero state
    record with status 5."""
    for e in (shared_ensemble(), sweep_ensemble()):
        n = len(e["x0"])
        out1, st1 = run(engine, e, 5, keep=1, quat=quat)
        tr1 = engine.mc_trajectories(n)
        out2, st2 = run(engine, e, 5, keep=2, quat=quat)
        tr2 = engine.mc_trajectories(n)
        assert out1.tobytes() == out2.tobytes() and stats_tuple(st1) == stats_tuple(st2)
        for k in ("X", "U", "X_sim", "U_sim", "B_eci"):
            assert np.array_equal(tr1[k], tr2[k]), k
        state, lam = engine.mc_state(n)
        for f in ("status", "outer_iters", "inner_iters", "ls_rollouts", "J", "c_max"):
            assert np.array_equal(state[f], out2[f]), f
        nc = out2["status"] == 5
        assert np.all(state["mu"][nc] == 0) and np.all(state["lam_goal"][nc] == 0)
        ko = tr2["knot_offs"]
        assert lam.shape == (ko[-1], 6) and np.all(lam >= 0.0)
        for t in np.nonzero(~nc)[0]:
            assert np.all(lam[ko[t + 1] - 1] == 0.0)
        assert np.any(out2["status"] == 1)
    assert nc.sum() == 1 and nc[2]


@pytest.mark.parametrize("pair,quat,J", [(0, 0, "diag"), (1, 0, "diag"), (2, 1, "diag"), (2, 0, "general")])
def test_continuation_equals_standalone_bit_for_bit(engine, pair, quat, J):
    """MC4: the continued trials' X, U, state, lam and solver fields of the records equal those of
    ts_alilqr_solve_state_batch continuing from the fetched state and trajectories over the run's active trials; MC3: their
    replay equals ts_tvlqr_sim_batch on the continued X, U (N_sim and slew time exactly, X_sim / U_sim to 1e-10)."""
    e = shared_ensemble(J=S.J_1U if J == "diag" else J_GEN)
    n = len(e["x0"])
    out1, _ = run(engine, e, 4, pair=pair, quat=quat)
    tr1 = snapshot(engine, n)
    o2 = cont_opts(e, 9)
    out2, st2 = engine.mc_continue(n, o2)
    tr2 = snapshot(engine, n)
    cont = (out1["status"] == 1) & (out1["outer_iters"] < 9)
    assert cont.sum() >= 2
    assert engine.k3_last_split()[2] == cont.sum() and st2.ms_field == 0 and st2.ms_prep == 0 and st2.ms_solve > 0
    assert engine.last_kernel_ms() > 0
    act, (X, U, _, oc, offs, stc, lamc) = standalone(engine, e, out1, tr1, o2, tr1["state"], tr1["lam"], tr1["X"], tr1["U"])
    assert np.array_equal(X, tr2["X"]) and np.array_equal(U, tr2["U"]) and np.array_equal(lamc, tr2["lam"])
    assert stc.tobytes() == tr2["state"][act].tobytes()
    for f in K3_FIELDS:
        assert np.array_equal(oc[f], out2[f][act]), f
    idx = np.nonzero(cont)[0]
    assert np.all(out2["t_final"] == out1["t_final"]) and np.all(out2["outer_iters"][idx] > out1["outer_iters"][idx])
    Xs, Us, _, _, nsim, slew, soffs = replay_standalone(engine, e, out2, tr2, idx)
    ko = tr2["knot_offs"]
    for k, t in enumerate(idx):
        assert out2["slew_time"][t] == slew[k]
        assert np.all(tr2["X_sim"][ko[t] + nsim[k]:ko[t + 1]] == 0.0)
        assert np.max(np.abs(tr2["X_sim"][ko[t]:ko[t + 1]] - Xs[soffs[k]:soffs[k + 1]])) <= 1e-10
        assert np.max(np.abs(tr2["U_sim"][ko[t]:ko[t + 1]] - Us[soffs[k]:soffs[k + 1]])) <= 1e-10
    # statistics: the whole ensemble after the call; flops of this call's added work
    assert st2.n_trials == n and list(st2.n_status) == list(np.bincount(out2["status"], minlength=6)[:6])
    assert st2.sum_inner_iters == out2["inner_iters"].sum() and st2.n_converged == (out2["status"] == 0).sum()
    assert 0 < st2.flops < out2["flops"][idx].sum()


def test_continuation_matches_oracle_pipeline(engine):
    """Each continued trial through the oracle's per-trial pipeline: build_slew, the oracle's solve to M1 with its state
    exported, its continuation to M2 from that state, then the oracle replay: status and counters exact, J and c_max to
    1e-6, the same slew time."""
    e = sweep_ensemble()
    n = len(e["x0"])
    cfg = e["cfg"]
    out1, _ = run(engine, e, 3)
    out2, _ = engine.mc_continue(n, cont_opts(e, 6))
    idx = np.nonzero(out1["status"] == 1)[0]
    assert len(idx) >= 2

    def one(t):
        f = e["fo"][t]
        s = S.build_slew(e["kep"][t], e["J"], e["x0"][t, 3:7], e["xf"][t, 3:7], mjd=f["mjd"], igrf_date=f["igrf_date"],
                         field_radius_m=f["field_radius_m"], t0=cfg.t0, tf=cfg.tf, N_scope=int(cfg.N_scope), cutoff=cfg.cutoff,
                         dt=cfg.dt, alpha=cfg.alpha, beta=cfg.beta)
        o1, o2 = orc.default_ilqr_opts(), orc.default_ilqr_opts()
        o1.max_outer, o2.max_outer = 3, 6
        X, U, _, r1, st, lam = AS.oracle_state_solve([s], o1, nthreads=1)
        Xc, Uc, _, rc, _, _ = AS.oracle_state_solve([s], o2, state=st, lam=lam, X=X, U=U, nthreads=1)
        o, _ = S.tvlqr_opts_pair(noise_mode=2, seed=int(cfg.tvlqr.seed), R=float(cfg.tvlqr.Rd[0]))
        x0l = s.x0.copy()
        x0l[3:7] = _perturb(s.x0[3:7], e["qn"][t])
        x0l[7] = 0
        a = S.oracle_tvlqr(s, Xc, Uc[:s.N - 1], x0l, o, trial=int(e["sid"][t]))
        return s, r1[0], rc[0], a[5]
    AS.oracle_lib()   # built once, before the threads use it
    with cf.ThreadPoolExecutor(len(idx)) as ex:
        refs = list(ex.map(one, idx))
    for t, (s, r1, rc, slew) in zip(idx, refs):
        assert out1[t]["N"] == s.N and r1["status"] == 1
        g = out2[t]
        for f in ("status", "outer_iters", "inner_iters", "ls_rollouts"):
            assert g[f] == rc[f], (t, f, g, rc)
        assert abs(g["J"] - rc["J"]) <= 1e-6 * abs(rc["J"])
        assert abs(g["c_max"] - rc["c_max"]) <= 1e-6 * max(1.0, rc["c_max"])
        assert g["slew_time"] == slew, (t, g["slew_time"], slew)


def test_cs4_against_a_direct_run(engine):
    """With cost_tol_intermediate = cost_tol, run(M1) + continue(M2) against run(M2): status and outer count on every
    trial; inner and line-search counters on all but at most 2; where they agree, J to 1e-10 and the same slew time."""
    e = shared_ensemble(n=8, seed=4)
    n = len(e["x0"])
    run(engine, e, 4, equal_tols=True)
    oc, _ = engine.mc_continue(n, cont_opts(e, 10))
    od, _ = run(engine, e, 10, equal_tols=True)
    assert np.array_equal(oc["status"], od["status"]) and np.array_equal(oc["outer_iters"], od["outer_iters"])
    same = (oc["inner_iters"] == od["inner_iters"]) & (oc["ls_rollouts"] == od["ls_rollouts"])
    assert (~same).sum() <= 2
    assert np.all(np.abs(oc["J"][same] - od["J"][same]) <= 1e-10 * np.abs(od["J"][same]))
    assert np.array_equal(oc["slew_time"][same], od["slew_time"][same])


def test_pass_through_no_op_and_chaining(engine):
    """MC1: pass-through trials (converged, NO_CUTOFF) are byte-identical in every kept array and record; max_outer <= the
    run's continues nothing and changes nothing; two chained calls M1 -> M2 -> M3 equal the stand-alone continuation of
    the fetched intermediate state."""
    e = sweep_ensemble()
    n = len(e["x0"])
    out1, _ = run(engine, e, 3)
    tr1 = snapshot(engine, n)
    outn, stn = engine.mc_continue(n, cont_opts(e, 3))
    assert outn.tobytes() == out1.tobytes() and stn.flops == 0 and stn.ms_solve == 0
    trn = snapshot(engine, n)
    for k in ("X", "U", "X_sim", "U_sim", "B_eci", "lam", "state"):
        assert trn[k].tobytes() == tr1[k].tobytes(), k
    out2, _ = engine.mc_continue(n, cont_opts(e, 5))
    tr2 = snapshot(engine, n)
    ko = tr1["knot_offs"]
    passed = np.nonzero(out1["status"] != 1)[0]
    assert any(out1["status"][passed] == 5)
    for t in passed:
        assert out2[t].tobytes() == out1[t].tobytes() and tr2["state"][t].tobytes() == tr1["state"][t].tobytes()
        r = slice(ko[t], ko[t + 1])
        for k in ("X", "U", "X_sim", "U_sim", "lam"):
            assert tr2[k][r].tobytes() == tr1[k][r].tobytes(), (t, k)
    assert np.array_equal(tr2["B_eci"], tr1["B_eci"])
    out3, _ = engine.mc_continue(n, cont_opts(e, 8))
    tr3 = snapshot(engine, n)
    assert np.any(out3["outer_iters"] > 5)
    act, (X, U, _, oc, _, stc, lamc) = standalone(engine, e, out2, tr2, cont_opts(e, 8), tr2["state"], tr2["lam"], tr2["X"], tr2["U"])
    assert np.array_equal(X, tr3["X"]) and np.array_equal(U, tr3["U"]) and np.array_equal(lamc, tr3["lam"])
    assert stc.tobytes() == tr3["state"][act].tobytes()
    for f in K3_FIELDS:
        assert np.array_equal(oc[f], out3[f][act]), f


def test_kept_run_is_isolated_from_other_entries(engine):
    """The kept run survives every other entry: a continuation after a stand-alone state solve, a plain solve, a TVLQR
    replay, a cutoff search and a field-map evaluation is byte-identical to one made without them."""
    e = shared_ensemble()
    n = len(e["x0"])
    run(engine, e, 4)
    outa, sta = engine.mc_continue(n, cont_opts(e, 7))
    tra = snapshot(engine, n)
    out1, _ = run(engine, e, 4)
    tr1 = snapshot(engine, n)
    standalone(engine, e, out1, tr1, cont_opts(e, 7), tr1["state"], tr1["lam"], tr1["X"], tr1["U"])
    standalone(engine, e, out1, tr1, cont_opts(e, 3))
    engine.alilqr_solve_batch(**_plain_args())
    replay_standalone(engine, e, out1, tr1, np.arange(3))
    engine.condition_cutoff_batch(tr1["B_eci"], [0, 0], [100, 200], [0.48, 0.48], [30.0, 30.0])
    g = np.random.default_rng(2).normal(size=(40, 50, 3))
    engine.field_map_eval_batch(engine.field_map_prefilter(g), np.linspace(1, 40, 1000), np.linspace(1, 50, 1000))
    outb, stb = engine.mc_continue(n, cont_opts(e, 7))
    trb = snapshot(engine, n)
    assert outb.tobytes() == outa.tobytes() and stats_tuple(stb) == stats_tuple(sta)
    for k in ("X", "U", "X_sim", "U_sim", "B_eci", "lam", "state"):
        assert trb[k].tobytes() == tra[k].tobytes(), k


def _plain_args():
    s = [S.build_slew([0, 6578, 96, 0, 0, 90], S.J_1P, S.quat_axis_angle([1, 0, 1], a), np.array([1.0, 0, 0, 0]), t_final=20.0)
         for a in (2.0, 4.0)]
    p = AS.pack(s)
    return dict(N_i=p["N_i"], x0=p["x0"], xf=p["xf"], Jmat=p["J"], Qd=p["Qd"], Qfd=p["Qfd"], Rd=p["Rd"], B_eci=p["B_eci"],
                B_offs=p["B_offs"], B_rows=p["B_rows"], index_scale=p["index_scale"], clock_rate=p["clock_rate"], dt=p["dt"])


def test_errors_leave_out_and_stats_untouched(engine):
    """TS_ERR_ARG (-2), out and stats untouched: a fresh engine, after a keep_trajectories = 1 run, after a keep = 2 run
    followed by a keep = 0 run, and with a wrong n_trials."""
    import tortoisesat.jl_b200 as tb
    from tortoisesat.jl_b200 import host
    e = shared_ensemble(n=4)
    n = 4
    o = cont_opts(e, 8)

    def call(eng, nn):
        out = np.frombuffer(np.full(nn * host.OUTCOME_DTYPE.itemsize, 0x5A, dtype=np.uint8).tobytes(), dtype=host.OUTCOME_DTYPE).copy()
        before = out.tobytes()
        st = host.McStats()
        st.n_trials, st.flops = 77, 1.5
        rc = eng.lib.ts_mc_continue(eng.h, nn, C.byref(o), out.ctypes.data, C.byref(st))
        assert out.tobytes() == before and st.n_trials == 77 and st.flops == 1.5
        return rc
    fresh = tb.Engine(0)
    assert call(fresh, n) == -2
    fresh.close()
    run(engine, e, 4, keep=1)
    assert call(engine, n) == -2
    run(engine, e, 4, keep=2)
    run(engine, e, 4, keep=0)
    assert call(engine, n) == -2
    run(engine, e, 4, keep=2)
    assert call(engine, n + 1) == -2
    out, _ = engine.mc_continue(n, o)
    assert out["status"].size == n


def test_kept_run_without_active_trials(engine):
    """A keep = 2 run in which no trial reaches the solver, after one in which some did: nothing of the first run leaks
    through.  The fetched states are zero records with status 5, a continuation returns the run's records and does no
    work, the ensemble gives NaN rows, and the trajectory layout (hence mc_trajectories and mc_state) refuses the run."""
    import tortoisesat.jl_b200 as tb
    from tortoisesat.jl_b200 import host
    e = shared_ensemble()
    n = len(e["x0"])
    out1, _ = run(engine, e, 4)
    assert np.all(out1["status"] != 5)
    e["cfg"].cutoff = 1.0   # a condition number is >= 1: no orbit reaches this cutoff
    out2, _ = run(engine, e, 4)
    ref = np.zeros(n, dtype=host.OUTCOME_DTYPE)
    ref["status"] = 5
    assert out2.tobytes() == ref.tobytes()
    state = np.frombuffer(np.full(n * host.AL_STATE_DTYPE.itemsize, 0x5A, dtype=np.uint8).tobytes(), dtype=host.AL_STATE_DTYPE).copy()
    assert engine.lib.ts_mc_fetch_state(engine.h, state.ctypes.data, None) == 0
    ref_state = np.zeros(n, dtype=host.AL_STATE_DTYPE)
    ref_state["status"] = 5
    assert state.tobytes() == ref_state.tobytes()
    oc, st = engine.mc_continue(n, cont_opts(e, 9))
    assert oc.tobytes() == out2.tobytes() and st.ms_solve == 0 and st.ms_tvlqr == 0 and st.flops == 0
    slew, xfin = engine.mc_replay_ensemble(n, 3, want_x_final=True)
    assert slew.shape == (n, 3) and np.all(np.isnan(slew)) and np.all(np.isnan(xfin))
    with pytest.raises(tb.TortoiseError):
        engine.mc_trajectories(n)
    with pytest.raises(tb.TortoiseError):
        engine.mc_state(n)


def test_no_replay(engine):
    """A kept run with run_tvlqr = 0 continues, with slew_time 0; fetching X_sim still fails."""
    import tortoisesat.jl_b200 as tb
    e = shared_ensemble(n=4)
    n = 4
    out1, _ = run(engine, e, 4, run_tvlqr=0)
    out2, st2 = engine.mc_continue(n, cont_opts(e, 8))
    assert np.any(out2["outer_iters"] > out1["outer_iters"]) and np.all(out2["slew_time"] == 0) and st2.ms_tvlqr == 0
    with pytest.raises(tb.TortoiseError):
        engine.mc_trajectories(n)
    engine.mc_trajectories(n, want=("X", "U"))


def test_multi_gpu_continuation_matches_single(engine):
    """MultiEngine([0]) and over min(device_count, 2) devices: run with keep = 2, then continue; the records equal the
    single-engine continuation field for field."""
    import torch
    from tortoisesat.jl_b200 import host
    e = shared_ensemble(n=10, seed=5)
    n = 10
    run(engine, e, 4)
    ref, st_ref = engine.mc_continue(n, cont_opts(e, 8))
    cfg = e["cfg"]
    for devs in ([0], list(range(min(torch.cuda.device_count(), 2)))):
        m = host.MultiEngine(devs)
        m.monte_carlo_run(cfg, e["kep"], e["fo"], e["x0"], e["xf"], e["Jm"], q_noise0=e["qn"], stream_id=e["sid"])
        out, st = m.mc_continue(n, cont_opts(e, 8))
        m.close()
        for f in out.dtype.names:
            assert np.array_equal(out[f], ref[f]), (devs, f)
        assert st.n_trials == n and list(st.n_status) == list(st_ref.n_status)
        assert st.sum_inner_iters == st_ref.sum_inner_iters and st.ms_field == 0


def test_continue_monte_carlo_wrapper():
    """continue_monte_carlo on a monte_carlo(..., resumable=True) result updates outcomes, fails and the trajectory lists
    of the continued trials, and returns their indices."""
    from tortoisesat.jl_b200 import host
    o = host.default_ilqr_opts()
    o.max_outer = 3
    res = host.monte_carlo(number_sims=4, seed=3, trajectories=True, resumable=True, ilqr=o)
    prev = res["outcomes"].copy()
    states = [s.copy() for s in res["states"]]
    idx = host.continue_monte_carlo(res, max_outer=6)
    assert np.array_equal(idx, np.nonzero(prev["status"] == 1)[0]) and idx.size >= 1
    out = res["outcomes"]
    assert np.all(out["outer_iters"][idx] > 3)
    assert np.array_equal(res["fails"], (out["slew_time"] == out["t_final"]).astype(float))
    assert np.array_equal(res["slew_time"], out["slew_time"])
    tr = host.default_engine().mc_trajectories(4)
    ko = tr["knot_offs"]
    for t in range(4):
        assert np.array_equal(res["states"][t], tr["X"][ko[t]:ko[t + 1]].T)
        assert np.array_equal(res["sim_states"][t], tr["X_sim"][ko[t]:ko[t + 1]].T)
        if t not in idx:
            assert np.array_equal(res["states"][t], states[t])
