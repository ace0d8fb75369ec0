"""Weight-sweep ensembles of a kept Monte-Carlo run (ts_mc_weight_ensemble) on bench.py's ensembles -> one JSON line.

  1. the fixed-orbit ensemble (bench.make_trials("mc_fixed_orbit", 4096, 0)), kept with keep_trajectories = 1: 16
     tracking weightings (R in {75, 750, 7.5e3, 7.5e4} x Q scale in {0.1, 1, 10, 100} of the run's Q = 10 I, Qf = 100 Q)
     at realisations 1 .. 64, every truth-model group on (sigma_inertia 0.1, sigma_torquer 0.05, sigma_field_scale 0.05,
     sigma_field_angle 3 deg), with u_limit 0 and 1 (the planner's u_max): device ms of the gains (K4a + every set's
     Riccati sweep) and of the replay (K4w), replays/s, and the share of the FP64 peak measured by ts_fp64_peak_probe on
     tools/flopcount.cpp's dispersed replay-step count (part (d); the clamp adds compares, not FLOPs).  Alternated in the
     same process with ts_mc_dispersion_ensemble at the run's weighting over the same number of replays (n_real = 64 x 16).
  2. the sweep (("mc_sweep", 8192, 0)): 4 weightings x 32 realisations, the ragged case.
  3. from the timed calls, and from the same calls without truth-model errors: the fail rate and the mean slew time of
     the non-failing draws per weighting, with and without the limit (paired draws, WE2).
The run's own weighting (default_mc_config's, as bench.mc_config: Q = 10 I, Qf = 100 Q, R = 0.5e3 I, not on the grid)
is a row of the table of its own: its unlimited rows are checked against ts_mc_dispersion_ensemble's and, without
truth-model errors, against ts_mc_replay_ensemble's (WE3).
The card name and power limit are read in the same call.
Usage: python tools/weight_ensemble_bench.py [--out FILE] [--fixed N] [--sweep N] [--n-real R] [--reps K]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

import tortoisesat.jl_b200 as tb  # noqa: E402
from dispersion_bench import ALL, flops_per_step, kept_run  # noqa: E402
from tortoisesat.jl_b200 import host  # noqa: E402
from replay_ensemble_bench import card  # noqa: E402

R_GRID = (75.0, 750.0, 7.5e3, 7.5e4)
Q_GRID = (0.1, 1.0, 10.0, 100.0)


def weighting(q_scale, r):
    """Qd 6 | Qfd 6 | Rd 3 of Q = 10 q_scale I, Qf = 100 Q, R = r I."""
    q = 10.0 * q_scale
    return [q] * 6 + [100.0 * q] * 6 + [r] * 3


def stats(slew, act, tf):
    """Per set: fail rate and mean / std of the non-failing slew times over the active trials' rows."""
    rows = []
    for w in range(slew.shape[1]):
        s = slew[act, w]
        fails = s == tf
        ok = ~fails
        rows.append(dict(fail_rate=float(fails.mean()), slew_mean_ok=float(s[ok].mean()) if ok.any() else None,
                         slew_std_ok=float(s[ok].std()) if ok.any() else None))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--fixed", type=int, default=4096)
    ap.add_argument("--sweep", type=int, default=8192)
    ap.add_argument("--n-real", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    eng = tb.Engine(0)
    peak = eng.fp64_peak_tflops()
    fl_d, _ = flops_per_step()
    res = dict(card=card(), fp64_peak_tflops_probe=peak)
    labels = [dict(q_scale=q, R=r) for r in R_GRID for q in Q_GRID]
    sets = np.array([weighting(l["q_scale"], l["R"]) for l in labels])
    n_sets, R = len(labels), a.n_real
    # 1. fixed orbit: K4w (u_limit 0 and 1) against K4d over the same number of replays, alternated
    out, act, steps = kept_run(eng, "mc_fixed_orbit", a.fixed)
    eng.mc_weight_ensemble(a.fixed, 32, sets[:2], 0.0, ALL, r_first=1)   # warm-up of the kernels
    eng.mc_weight_ensemble(a.fixed, 32, sets[:2], 1.0, ALL, r_first=1)
    eng.mc_dispersion_ensemble(a.fixed, 32, r_first=1, **ALL)
    timing = {"u_limit=0": [], "u_limit=1": [], "dispersion": []}
    slews = {}
    for _ in range(a.reps):
        for u in (0.0, 1.0):
            slews[u], _ = eng.mc_weight_ensemble(a.fixed, R, sets, u, ALL, r_first=1)
            timing["u_limit=%g" % u].append(eng.mc_replay_ensemble_split())
        eng.mc_dispersion_ensemble(a.fixed, R * n_sets, r_first=1, **ALL)
        timing["dispersion"].append(eng.mc_replay_ensemble_split())
    replays = int(act.size) * R * n_sets

    def summary(ts):
        best = min(r for _, r in ts)
        return dict(gains_ms=[g for g, _ in ts], replay_ms=[r for _, r in ts], replays_per_s=replays / (best / 1e3),
                    flops_per_replay_step=fl_d, fp64_share_of_peak=fl_d * steps * R * n_sets / (best / 1e3) / (peak * 1e12))
    fx = {k: summary(v) for k, v in timing.items()}
    res["fixed_orbit"] = dict(n_trials=a.fixed, active=int(act.size), n_sets=n_sets, n_real=R, realisations=[1, R],
                              replay_steps_per_realisation=steps, sigmas=ALL, weight_ensemble_u0=fx["u_limit=0"],
                              weight_ensemble_u1=fx["u_limit=1"], dispersion_same_replays=dict(fx["dispersion"], n_real=R * n_sets),
                              replay_time_ratio_u0=min(fx["u_limit=0"]["replay_ms"]) / min(fx["dispersion"]["replay_ms"]),
                              replay_time_ratio_u1=min(fx["u_limit=1"]["replay_ms"]) / min(fx["dispersion"]["replay_ms"]))
    # 3. the per-set table: every group on (the timed calls) and disturbances only, with and without the limit
    tf = out["t_final"][act][:, None]
    quiet = {u: eng.mc_weight_ensemble(a.fixed, R, sets, u, None, r_first=1)[0] for u in (0.0, 1.0)}
    tv = host.default_mc_config(1).tvlqr
    run_w = np.array([list(tv.Qd) + list(tv.Qfd) + list(tv.Rd)])
    own = {(d, u): eng.mc_weight_ensemble(a.fixed, R, run_w, u, ALL if d == "all" else None, r_first=1)[0]
           for d in ("all", "none") for u in (0.0, 1.0)}
    ref_d, _, _ = eng.mc_dispersion_ensemble(a.fixed, R, r_first=1, **ALL)
    ref_e, _ = eng.mc_replay_ensemble(a.fixed, R, r_first=1)
    row = dict(q_scale="run", R=float(tv.Rd[0]), weights=[float(v) for v in run_w[0]],
               equals_dispersion_ensemble=bool(own[("all", 0.0)][:, 0].tobytes() == ref_d.tobytes()),
               equals_replay_ensemble=bool(own[("none", 0.0)][:, 0].tobytes() == ref_e.tobytes()))
    for d in ("all", "none"):
        for u in (0.0, 1.0):
            row["%s_u%d" % (d, u)] = stats(own[(d, u)], act, tf)[0]
    table = [row]
    for w, l in enumerate(labels):
        row = dict(l)
        for key, sl in (("all_u0", slews[0.0]), ("all_u1", slews[1.0]), ("none_u0", quiet[0.0]), ("none_u1", quiet[1.0])):
            row[key] = stats(sl[:, w:w + 1], act, tf)[0]
        table.append(row)
    res["fail_table"] = dict(workload="mc_fixed_orbit", n_trials=a.fixed, active=int(act.size), realisations=[1, R], sigmas=ALL,
                             rows=table)
    # 2. the sweep: 4 weightings (R in R_GRID at the run's Q) x 32 realisations
    if a.sweep:
        sw = np.array([weighting(1.0, r) for r in R_GRID])
        out, act, steps = kept_run(eng, "mc_sweep", a.sweep)
        eng.mc_weight_ensemble(a.sweep, 32, sw, 1.0, ALL, r_first=1)
        ts = []
        for _ in range(2):
            eng.mc_weight_ensemble(a.sweep, 32, sw, 1.0, ALL, r_first=1)
            ts.append(eng.mc_replay_ensemble_split())
        best = min(r for _, r in ts)
        res["sweep"] = dict(n_trials=a.sweep, active=int(act.size), n_sets=4, R=list(R_GRID), n_real=32, u_limit=1.0, sigmas=ALL,
                            replay_steps_per_realisation=steps, gains_ms=[g for g, _ in ts], replay_ms=[r for _, r in ts],
                            replays_per_s=int(act.size) * 4 * 32 / (best / 1e3),
                            fp64_share_of_peak=fl_d * steps * 4 * 32 / (best / 1e3) / (peak * 1e12))
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
