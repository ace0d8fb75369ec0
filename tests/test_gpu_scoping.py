"""The Monte-Carlo scoping cutoff (k2c_cutoff_scan over the sample ranges [0, 4096) and [4096, 2 N_scope), the running
gramian carried between chunks and between the ranges) and the long-horizon trials it produces, against a
high-precision reference of the gramian's condition number and the CPU oracle.

The fused call (ts_monte_carlo_run) sets every trial's horizon from the first scoping sample whose gramian condition
number is below the cutoff; the first range covers most orbits, the second one runs only for the orbits without a hit
in the first.  The tests place hits on chunk and range edges, mix IGRF degrees and a never-hitting orbit in one call,
and replay the benchmark sweep's longest slews (10^4 - 2.4*10^4 knots)."""
import concurrent.futures as cf
import functools
import math

import numpy as np
import pytest

import bench as B
import slew_setup as S
from oracle import oracle as orc

T0, TF = 0.0, 2400.0
SPLIT = 4096          # end of the first scoping range (tortoise_b200.cu, stage 1)
TIE = 1e-9            # a cond() this close to the cutoff may round either way in the kernel's pairwise prefix sums
NO_CUTOFF = 5
SWEEP_N = 8192        # bench.py's sweep shard; its trials are independent, so any subset is a valid run


# ------------------------------------------------------------------ reference
def cond_curve(kep, fo, N_scope, t0=T0, tf=TF):
    """cond() of the running magnetic gramian at every scoping sample: the oracle's field table, terms hat(b)hat(b)' =
    |b|^2 I - b b' (the first without dt, quirk Q9), prefix sums in long double, |eigenvalue| ratio from eigvalsh.
    Returns (cond, field table, dt)."""
    Bt, _, _, rc = orc.magnetic_simulation(kep, S.GM, fo[1], fo[2], fo[3], t0, tf, N_scope)
    assert rc == 0
    dt = (tf - t0) / N_scope
    h = np.einsum("ij,ij->i", Bt, Bt)[:, None, None] * np.eye(3) - Bt[:, :, None] * Bt[:, None, :]
    h = h.astype(np.longdouble)
    h[1:] *= np.longdouble(dt)
    ev = np.abs(np.linalg.eigvalsh(np.cumsum(h, axis=0).astype(np.float64)))
    with np.errstate(divide="ignore", invalid="ignore"):
        c = ev.max(axis=1) / ev.min(axis=1)
    c[np.isnan(c)] = np.inf
    return c, Bt, dt


def first_below(c, cutoff):
    """First 1-based sample with c < cutoff, 0 if there is none."""
    i = np.flatnonzero(c < cutoff)
    return int(i[0]) + 1 if len(i) else 0


def reference_cutoff(kep, fo, N_scope, cutoff):
    """(index, accepted indices, tie) of the cutoff search.  A cond() within TIE of the cutoff before or at the first
    hit is a tie: the kernel may return the index of either neighbour.  Without a tie the index must also be the
    oracle's condition_based_time of the oracle's gramian."""
    c, Bt, dt = cond_curve(kep, fo, N_scope)
    idx = first_below(c, cutoff)
    lo, hi = first_below(c, cutoff * (1 + TIE)), first_below(c, cutoff * (1 - TIE))
    tie = lo != hi
    if not tie:
        assert orc.condition_based_time(orc.magnetic_gramian(Bt, dt), cutoff) == idx
    return idx, {lo, hi}, tie


@functools.lru_cache(maxsize=None)
def sweep():
    return B.make_trials("mc_sweep", SWEEP_N, 0)


@functools.lru_cache(maxsize=None)
def long_selection():
    """Every sweep trial with inclination < 15 deg (the ones whose cutoff can lie beyond the first range) plus 128
    others, with their reference cutoffs at the benchmark's cutoff and N_scope 5000."""
    tr = sweep()
    inc = tr["kep"][:, 2]
    low = np.flatnonzero(inc < 15.0)
    rest = np.flatnonzero(inc >= 15.0)
    sel = np.sort(np.concatenate([low, np.random.default_rng(11).choice(rest, 128, replace=False)]))

    def one(t):
        return reference_cutoff(tr["kep"][t], tr["fo"][t], 5000, tr["cutoff"])
    with cf.ThreadPoolExecutor(orc.lib().orc_max_threads()) as ex:      # the oracle calls release the GIL (ctypes)
        refs = list(ex.map(one, sel))
    return sel, refs


# ------------------------------------------------------------------ CPU
def test_sweep_composition_and_reference_agree_with_oracle():
    """The benchmark sweep reaches the second scoping range (so the GPU tests below cover it), and the long-double
    reference agrees with the oracle's condition_based_time on every non-tie orbit (checked inside reference_cutoff)."""
    tr = sweep()
    sel, refs = long_selection()
    low = tr["kep"][sel, 2] < 15.0
    idx = np.array([r[0] for r in refs])
    assert np.all(idx[low] > 0)
    assert np.sum(idx[low] > SPLIT) >= 20
    assert sum(r[2] for r in refs) == 0


# ------------------------------------------------------------------ GPU helpers
def _fo_array(fos):
    from tortoisesat.jl_b200 import host
    fo = np.zeros(len(fos), dtype=host.FIELD_OPTS_DTYPE)
    for i, f in enumerate(fos):
        fo[i] = tuple(f)
    return fo


def _horizon_only_config(n, shared, N_scope, cutoff):
    """The fused call with a one-iteration solve and no replay: what it computes here is the horizon."""
    from tortoisesat.jl_b200 import host
    cfg = host.default_mc_config(n, shared_orbit=shared, run_tvlqr=False, t0=T0, tf=TF, N_scope=N_scope, cutoff=cutoff, dt=0.2,
                                 alpha=0.1, beta=1e3)
    cfg.ilqr.max_outer, cfg.ilqr.max_inner = 1, 2
    return cfg


def _check_horizon(g, accepted, N_scope, dt=0.2):
    """t_final is idx*(tf-t0)/N_scope (the host's expression, compared exactly), N = floor((t_final-t0)/dt); no hit or
    fewer than 2 knots: NO_CUTOFF with N = 0."""
    if g["status"] == NO_CUTOFF and g["N"] == 0:
        idx = 0
        assert g["t_final"] == 0.0
    else:
        idx = int(round(g["t_final"] * N_scope / (TF - T0)))
        assert g["t_final"] == idx * (TF - T0) / N_scope
        assert g["N"] == int(math.floor((g["t_final"] - T0) / dt)) and g["N"] >= 2
    assert idx in accepted, (idx, accepted)
    if idx == 0:
        assert g["status"] == NO_CUTOFF and g["N"] == 0
    return idx


# ------------------------------------------------------------------ targeted boundaries
# (N_scope, 0-based target sample, sweep trial whose cond() curve has a strict new running minimum there).  Chunk edges
# 127 / 128, the range edge 4095 / 4096 / 4097, the second range's first chunk edge 4223 / 4224, the last live row
# 2 N_scope - 2; N_scope 1000: one range; 2048: the second range is empty; 2049: the second range is two rows.
TARGETS = [(5000, 127, 715), (5000, 128, 715), (5000, 4095, 564), (5000, 4096, 564), (5000, 4097, 564), (5000, 4223, 564),
           (5000, 4224, 564), (5000, 9998, 1542), (1000, 127, 94), (1000, 128, 94), (1000, 1998, 1542), (2048, 127, 1121),
           (2048, 4094, 1542), (2049, 4095, 1542), (2049, 4096, 1542)]


@pytest.mark.gpu
@pytest.mark.parametrize("N_scope,target,trial", TARGETS)
def test_cutoff_on_chunk_and_range_edges(engine, N_scope, target, trial):
    """One orbit, a cutoff between cond[target] and the running minimum before it (geometric mean): the first hit is
    exactly sample target (1-based index target + 1)."""
    tr = sweep()
    kep, fo = tr["kep"][trial], tr["fo"][trial]
    c, _, _ = cond_curve(kep, fo, N_scope)
    assert target <= 2 * N_scope - 2                           # the last live row; row 2 N_scope - 1 is zero
    prev = np.min(c[:target])
    assert c[target] < prev / (1 + 1e-6)                       # a strict new running minimum, far from a tie
    cutoff = math.sqrt(c[target] * prev)
    idx, accepted, tie = reference_cutoff(kep, fo, N_scope, cutoff)
    assert idx == target + 1 and not tie
    cfg = _horizon_only_config(1, True, N_scope, cutoff)
    out, st = engine.monte_carlo_run(cfg, kep[None], _fo_array([fo]), tr["x0"][trial][None], tr["xf"][trial][None],
                                     tr["Jm"][trial][None])
    assert _check_horizon(out[0], accepted, N_scope) == target + 1
    assert out[0]["status"] != NO_CUTOFF and st.n_no_cutoff == 0


@pytest.mark.gpu
def test_cutoff_mixed_orbits_and_degrees(engine):
    """One call, one orbit per trial (shared_orbit = 0): hits in the first range (a degree-13 and a degree-10 orbit, the
    latter skipped by both k2b_field_rows instantiations in the second range), hits in the second range (degree 13 and
    a pre-1995 degree-10 date), and an orbit that never reaches the cutoff."""
    tr = sweep()
    cutoff, N_scope = 70.0, 5000
    # (sweep trial, IGRF date override or None, expected range: 1, 2 or 0 = never)
    plan = [(30, None, 1), (1542, 1990.0, 1), (564, None, 2), (429, 1990.0, 2), (6472, 1990.0, 2), (2389, None, 0)]
    kep = np.stack([tr["kep"][t] for t, _, _ in plan])
    fos = []
    for t, date, _ in plan:
        f = list(tr["fo"][t])
        if date is not None:
            f[2] = date
        fos.append(f)
    assert {13 if f[2] >= 1995 else 10 for f in fos} == {10, 13}
    refs = [reference_cutoff(kep[k], fos[k], N_scope, cutoff) for k in range(len(plan))]
    for (t, date, rng_), (idx, _, tie) in zip(plan, refs):
        assert not tie
        assert {0: idx == 0, 1: 0 < idx <= SPLIT, 2: idx > SPLIT}[rng_], (t, date, idx)
    n = len(plan)
    cfg = _horizon_only_config(n, False, N_scope, cutoff)
    sel = [t for t, _, _ in plan]
    out, st = engine.monte_carlo_run(cfg, kep, _fo_array(fos), tr["x0"][sel], tr["xf"][sel], tr["Jm"][sel])
    for k in range(n):
        assert _check_horizon(out[k], refs[k][1], N_scope) == refs[k][0], (plan[k], out[k])
    assert st.n_no_cutoff == 1


# ------------------------------------------------------------------ the benchmark's long trials
LONG_MAX_OUTER, LONG_MAX_INNER = 2, 5       # a truncated solve: ~3.5 s of oracle time per 2.4*10^4-knot slew


def _truncated(opts):
    opts.max_outer, opts.max_inner = LONG_MAX_OUTER, LONG_MAX_INNER
    return opts


@pytest.fixture(scope="module")
def long_run(engine):
    """The selected sweep trials in one fused call with the benchmark's configuration, no replay, a truncated solve and
    the trajectories kept."""
    from tortoisesat.jl_b200 import host
    tr = sweep()
    sel, refs = long_selection()
    n = len(sel)
    sub = dict(tr)
    for k in ("kep", "x0", "xf", "Jm", "qn"):
        sub[k] = tr[k][sel]
    sub["fo"] = [tr["fo"][t] for t in sel]
    cfg = B.mc_config(host, sub, n)
    cfg.run_tvlqr, cfg.keep_trajectories = 0, 1
    _truncated(cfg.ilqr)
    out, st = engine.monte_carlo_run(cfg, sub["kep"], _fo_array(sub["fo"]), sub["x0"], sub["xf"], sub["Jm"], q_noise0=sub["qn"])
    trj = engine.mc_trajectories(n, want=("B_eci",))
    second = [k for k in range(n) if refs[k][0] > SPLIT]
    return dict(sub=sub, sel=sel, refs=refs, out=out, trj=trj, second=second, cfg=cfg)


def _row_limit(N, dt=0.2):
    """Rows of a fine table the fused path fills: floor(x8max*N + 1) + 4, at most 2N - 1 (tortoise_b200.cu, stage 2)."""
    x8max = (N + 1) * dt / (TF - T0)
    return min(int(math.floor(x8max * N + 1.0)) + 4, 2 * N - 1)


@pytest.mark.gpu
def test_long_trials_horizons(long_run):
    """Every selected trial's horizon equals the reference's; at least 20 of them hit in the second range."""
    out, refs = long_run["out"], long_run["refs"]
    for k in range(len(refs)):
        assert _check_horizon(out[k], refs[k][1], 5000) == refs[k][0], (long_run["sel"][k], out[k], refs[k])
    assert len(long_run["second"]) >= 20
    assert max(out[k]["N"] for k in long_run["second"]) > 20000


@pytest.mark.gpu
def test_long_trials_fine_tables(long_run):
    """Second-range trials: rows [0, lim) of the kept fine field table are the oracle's magnetic_simulation over
    [t0, t_final] with N knots (1e-10 relative), the rows from lim on are zero."""
    sub, out, trj = long_run["sub"], long_run["out"], long_run["trj"]
    ro = trj["row_offs"]
    for k in long_run["second"]:
        g = out[k]
        N = int(g["N"])
        f = sub["fo"][k]
        Bo, _, _, rc = orc.magnetic_simulation(sub["kep"][k], S.GM, f[1], f[2], f[3], T0, float(g["t_final"]), N)
        assert rc == 0 and ro[k + 1] - ro[k] == 2 * N
        Bg = trj["B_eci"][ro[k]:ro[k + 1]]
        lim = _row_limit(N)
        assert np.max(np.abs(Bg[:lim] - Bo[:lim])) <= 1e-10 * np.max(np.abs(Bo[:lim])), k
        assert np.all(Bg[lim:] == 0.0) and np.all(np.any(Bg[:lim] != 0.0, axis=1)), k


@pytest.mark.gpu
def test_long_trials_solve_matches_oracle(long_run):
    """Second-range trials (10^4 - 2.4*10^4 knots): the fused truncated AL-iLQR solve against the oracle's with the same
    options: same status and outer count, J and c_max to 1e-6, inner and line-search counters identical on all but at
    most one trial."""
    sub, out = long_run["sub"], long_run["out"]
    cfg = long_run["cfg"]
    oo = _truncated(orc.default_ilqr_opts())

    def one(k):
        f = sub["fo"][k]
        s = S.build_slew(sub["kep"][k], S.J_1U, sub["x0"][k, 3:7], sub["xf"][k, 3:7], mjd=f[1], igrf_date=f[2], field_radius_m=f[3],
                         t0=T0, tf=TF, dt=cfg.dt, alpha=cfg.alpha, beta=cfg.beta, t_final=float(out[k]["t_final"]))
        return S.oracle_solve([s], oo, want_K=False)[3][0], s.N
    with cf.ThreadPoolExecutor(orc.lib().orc_max_threads()) as ex:
        refs = list(ex.map(one, long_run["second"]))
    n_diff = 0
    for k, (r, N) in zip(long_run["second"], refs):
        g = out[k]
        assert g["N"] == N
        assert (g["status"], g["outer_iters"]) == (r["status"], r["outer_iters"]), (k, g, r)
        assert abs(g["J"] - r["J"]) <= 1e-6 * abs(r["J"]), (k, g, r)
        assert abs(g["c_max"] - r["c_max"]) <= 1e-6 * max(1.0, r["c_max"]), (k, g, r)
        n_diff += (g["inner_iters"], g["ls_rollouts"]) != (r["inner_iters"], r["ls_rollouts"])
    assert n_diff <= 1


@pytest.mark.gpu
def test_long_trials_never_read_past_row_limit(engine, long_run):
    """The solver and the TVLQR replay never read a fine-table row at or after the first all-zero tail row: with those
    rows set to NaN, the stand-alone solve of the longest second-range slews (kept tables, weights from
    slew_weights_batch) and their replay with device noise give the same bits as on the kept tables."""
    from tortoisesat.jl_b200 import host
    sub, out, trj = long_run["sub"], long_run["out"], long_run["trj"]
    ks = sorted(long_run["second"], key=lambda k: -out[k]["N"])[:4]
    ro = trj["row_offs"]
    N_i = np.array([out[k]["N"] for k in ks], dtype=np.int64)
    tfin = np.array([out[k]["t_final"] for k in ks])
    x0, xf, Jm = sub["x0"][ks], sub["xf"][ks], sub["Jm"][ks]
    tables = [trj["B_eci"][ro[k]:ro[k + 1]] for k in ks]
    rows = np.array([len(b) for b in tables], dtype=np.int64)
    B_offs = np.concatenate([[0], np.cumsum(rows)[:-1]]).astype(np.int64)
    Qd, Qfd, Rd = engine.slew_weights_batch(x0, xf, Jm, tfin, t0=T0, dt=0.2, alpha=0.1, beta=1e3)
    isc, cr = N_i.astype(np.float64), np.full(len(ks), 1.0 / (TF - T0))
    _, g = S.tvlqr_opts_pair(noise_mode=2, seed=int(B.SEED), R=0.5e3)
    x0l = x0.copy()
    x0l[:, 7] = 0.0

    def run(Ball):
        X, U, _, res, _ = engine.alilqr_solve_batch(N_i, x0, xf, Jm, Qd, Qfd, Rd, Ball, B_offs, rows, isc, cr, 0.2,
                                                    opts=_truncated(host.default_ilqr_opts()), want_K=False)
        Xs, Us, _, _, nsim, slew, _ = engine.tvlqr_sim_batch(N_i, X, U, x0l, Jm, Ball, B_offs, rows, isc, cr, tfin,
                                                             xf[:, 3:7], opts=g, stream_id=np.arange(len(ks)))
        return res, X, U, Xs, Us, nsim, slew

    kept = np.concatenate(tables)
    poisoned = []
    for b in tables:
        nz = np.flatnonzero(np.any(b != 0.0, axis=1))
        first_zero_tail = int(nz[-1]) + 1
        assert first_zero_tail == _row_limit(len(b) // 2)
        p = b.copy()
        p[first_zero_tail:] = np.nan
        poisoned.append(p)
    a, b = run(kept), run(np.concatenate(poisoned))
    assert a[0].tobytes() == b[0].tobytes()
    for x, y in zip(a[1:], b[1:]):
        assert np.array_equal(x, y, equal_nan=False)
    assert np.all(np.isfinite(a[1])) and np.all(a[5] > 1)
