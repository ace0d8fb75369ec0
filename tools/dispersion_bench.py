"""Dispersion ensembles of a kept Monte-Carlo run (ts_mc_dispersion_ensemble) on bench.py's ensembles -> one JSON line.

  1. the fixed-orbit ensemble (bench.make_trials("mc_fixed_orbit", 4096, 0)), kept with keep_trajectories = 1, at
     n_real = 256: device ms of the replay (K4d, every dispersion group on) against ts_mc_replay_ensemble (K4e) at the
     same shape, alternated in one process; replays/s, FLOPs per dispersed replay-step (profiles/flop_counts_r2.json,
     tools/flopcount.cpp part (d)) and the share of the FP64 peak measured by ts_fp64_peak_probe;
  2. the sweep (("mc_sweep", 8192, 0)) at n_real = 32;
  3. on the fixed-orbit run, realisations 1 .. n_table: the fail rate and the mean slew time of the non-failing draws,
     one dispersion group at a time and all together, next to the undispersed ensemble (paired draws, DE2).
Each table row also checks DE4 once: sigmas 0 give ts_mc_replay_ensemble's rows bit for bit.  The card name and power
limit are read in the same call.
Usage: python tools/dispersion_bench.py [--out FILE] [--fixed N] [--sweep N] [--n-real R] [--n-table R]"""
import argparse
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

import bench as B  # noqa: E402
import tortoisesat.jl_b200 as tb  # noqa: E402
from tortoisesat.jl_b200 import host  # noqa: E402
from replay_ensemble_bench import card, n_sim  # noqa: E402

DEG = math.pi / 180
ALL = dict(sigma_inertia=0.1, sigma_torquer=0.05, sigma_field_scale=0.05, sigma_field_angle=3 * DEG)
TABLE = [("none", {})] + [("sigma_inertia=%g" % v, dict(sigma_inertia=v)) for v in (0.05, 0.1, 0.2)] + \
        [("sigma_torquer=%g" % v, dict(sigma_torquer=v)) for v in (0.05, 0.1)] + \
        [("sigma_field_angle=%gdeg" % v, dict(sigma_field_angle=v * DEG)) for v in (1, 3, 5)] + \
        [("sigma_field_scale=0.05", dict(sigma_field_scale=0.05)), ("all: inertia 0.1, torquer 0.05, scale 0.05, angle 3deg", ALL)]


def flops_per_step():
    d = json.load(open(os.path.join(ROOT, "profiles", "flop_counts_r2.json")))
    return d["dispersion_replay_step"], d["ensemble_replay_step"]


def kept_run(eng, name, n):
    tr = B.make_trials(name, n, 0)
    cfg = B.mc_config(host, tr, n)
    cfg.keep_trajectories = 1
    out, st = eng.monte_carlo_run(cfg, tr["kep"], B.field_opts_array(tr), tr["x0"], tr["xf"], tr["Jm"], q_noise0=tr["qn"],
                                  stream_id=np.arange(n).astype(np.uint32))
    act = np.nonzero(out["status"] != 5)[0]
    steps = sum(n_sim(cfg, out["t_final"][t], int(out["N"][t])) - 1 for t in act)
    return out, act, int(steps)


def rates(eng, n, R, act, steps, peak, fl, dispersed, reps):
    ms = []
    for _ in range(reps):
        if dispersed:
            eng.mc_dispersion_ensemble(n, R, r_first=1, **ALL)
        else:
            eng.mc_replay_ensemble(n, R, r_first=1)
        ms.append(eng.mc_replay_ensemble_split()[1])
    best = min(ms)
    return dict(replay_ms=ms, gains_ms=eng.mc_replay_ensemble_split()[0], replays_per_s=act.size * R / (best / 1e3),
                flops_per_replay_step=fl, fp64_share_of_peak=fl * steps * R / (best / 1e3) / (peak * 1e12))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--fixed", type=int, default=4096)
    ap.add_argument("--sweep", type=int, default=8192)
    ap.add_argument("--n-real", type=int, default=256)
    ap.add_argument("--n-table", type=int, default=64)
    a = ap.parse_args()
    eng = tb.Engine(0)
    peak = eng.fp64_peak_tflops()
    fl_d, fl_e = flops_per_step()
    res = dict(card=card(), fp64_peak_tflops_probe=peak)
    # 1. fixed orbit: K4d against K4e at the same shape, alternated
    out, act, steps = kept_run(eng, "mc_fixed_orbit", a.fixed)
    eng.mc_replay_ensemble(a.fixed, 32, r_first=1)                  # warm-up of both kernels
    eng.mc_dispersion_ensemble(a.fixed, 32, r_first=1, **ALL)
    disp, ens = [], []
    for _ in range(3):
        ens.append(rates(eng, a.fixed, a.n_real, act, steps, peak, fl_e, False, 1))
        disp.append(rates(eng, a.fixed, a.n_real, act, steps, peak, fl_d, True, 1))
    best = lambda rows: min(rows, key=lambda r: r["replay_ms"][0])
    bd, be = best(disp), best(ens)
    res["fixed_orbit"] = dict(n_trials=a.fixed, active=int(act.size), n_real=a.n_real, replay_steps_per_realisation=steps,
                              sigmas=ALL, dispersion=dict(bd, replay_ms=[r["replay_ms"][0] for r in disp]),
                              replay_ensemble=dict(be, replay_ms=[r["replay_ms"][0] for r in ens]),
                              replay_time_ratio=bd["replay_ms"][0] / be["replay_ms"][0])
    # 3. the fail-rate / slew-time table on the same kept run (paired draws: realisations 1 .. n_table of every trial)
    tf = out["t_final"][act][:, None]
    base, _ = eng.mc_replay_ensemble(a.fixed, a.n_table, r_first=1)
    table = []
    for name, sg in TABLE:
        slew, _, prm = eng.mc_dispersion_ensemble(a.fixed, a.n_table, r_first=1, want_params=True, **sg)
        s = slew[act]
        fails = s == tf
        ok = ~fails
        row = dict(case=name, sigmas=sg, fail_rate=float(fails.mean()),
                   slew_mean_ok=float(s[ok].mean()) if ok.any() else None, slew_std_ok=float(s[ok].std()) if ok.any() else None,
                   param_std=[float(v) for v in np.nanstd(prm[act].reshape(-1, 10), axis=0)])
        if not sg:
            row["equals_replay_ensemble"] = bool(slew.tobytes() == base.tobytes())   # DE4
        table.append(row)
    res["fail_table"] = dict(workload="mc_fixed_orbit", n_trials=a.fixed, active=int(act.size), realisations=[1, a.n_table], rows=table)
    # 2. the sweep
    if a.sweep:
        out, act, steps = kept_run(eng, "mc_sweep", a.sweep)
        eng.mc_dispersion_ensemble(a.sweep, 32, r_first=1, **ALL)
        res["sweep"] = dict(n_trials=a.sweep, active=int(act.size), n_real=32, replay_steps_per_realisation=steps, sigmas=ALL,
                            dispersion=rates(eng, a.sweep, 32, act, steps, peak, fl_d, True, 2))
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
