"""Continuation of a kept Monte-Carlo run (ts_mc_continue) on bench.py's ensembles -> one JSON line.

For the fixed-orbit ensemble (bench.make_trials("mc_fixed_orbit", 4096, 0)) and the sweep (("mc_sweep", 8192, 0)):
  1. cost of keeping: ms_solve of a max_outer = 20 run with keep_trajectories 0 and 2, alternated, two each, and whether
     the outcome records are byte-identical;
  2. the continuation of the last kept run to max_outer = 30: ms_solve, ms_tvlqr, trials continued, trials that
     converge, status histogram;
  3. a direct run to max_outer = 30: ms_solve, ms_tvlqr, histogram, the continue / direct time ratio, and the continued
     trials whose status or outer count differ (CS4: the default tolerance pairs differ, so outer iteration 20 ran with
     the final tolerances in the kept run and with the intermediate ones in the direct run).
One warm-up run precedes the timed ones.  Usage: python tools/mc_continue_bench.py [--out FILE] [--fixed N] [--sweep N]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import bench as B  # noqa: E402
import tortoisesat.jl_b200 as tb  # noqa: E402
from tortoisesat.jl_b200 import host  # noqa: E402

STATUS = ["converged", "max_outer", "cost_blowup", "reg_max", "nan", "no_cutoff"]


def hist(out):
    h = np.bincount(out["status"], minlength=6)[:6]
    return {STATUS[k]: int(h[k]) for k in range(6)}


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as ex:  # pragma: no cover
        return "unknown (%s)" % ex


def ensemble(eng, workload, n):
    tr = B.make_trials(workload, n, 0)
    cfg = B.mc_config(host, tr, n)
    fo = B.field_opts_array(tr)
    sid = np.arange(n).astype(np.uint32)

    def run(keep, max_outer):
        cfg.keep_trajectories = keep
        cfg.ilqr.max_outer = max_outer
        return eng.monte_carlo_run(cfg, tr["kep"], fo, tr["x0"], tr["xf"], tr["Jm"], q_noise0=tr["qn"], stream_id=sid)

    run(0, 20)   # warm-up: module load, scratch allocation
    keep = {0: [], 2: []}
    recs = {}
    for k in (0, 2, 0, 2):
        out, st20 = run(k, 20)
        keep[k].append(st20.ms_solve)
        recs.setdefault(k, out)
        assert out.tobytes() == recs[k].tobytes()
    out20 = recs[2]
    o30 = host.IlqrOpts.from_buffer_copy(cfg.ilqr)
    o30.max_outer = 30
    cont = out20["status"] == 1
    outc, stc = eng.mc_continue(n, o30)
    split = eng.k3_last_split()
    outd, std = run(0, 30)
    return {
        "workload": B.workload_name(workload, n), "trials": n,
        "keep_cost": {"ms_solve_keep0": keep[0], "ms_solve_keep2": keep[2],
                      "records_identical": recs[0].tobytes() == recs[2].tobytes(),
                      "ratio_keep2_over_keep0": float(np.mean(keep[2]) / np.mean(keep[0]))},
        "run20": {"status": hist(out20), "ms_field": st20.ms_field, "ms_prep": st20.ms_prep, "ms_tvlqr": st20.ms_tvlqr},
        "continue20to30": {"ms_solve": stc.ms_solve, "ms_tvlqr": stc.ms_tvlqr, "continued": int(cont.sum()),
                           "converged_of_continued": int((outc["status"][cont] == 0).sum()), "status": hist(outc),
                           "k3_split_ms": [split[0], split[1]], "parked": split[2]},
        "direct30": {"ms_solve": std.ms_solve, "ms_tvlqr": std.ms_tvlqr, "ms_field": std.ms_field, "ms_prep": std.ms_prep,
                     "status": hist(outd)},
        "continue_over_direct_time": (stc.ms_solve + stc.ms_tvlqr) / (std.ms_field + std.ms_prep + std.ms_solve + std.ms_tvlqr),
        "continue_over_direct_solve": stc.ms_solve / std.ms_solve,
        "cs4_differences_on_continued": {
            "status": int((outc["status"][cont] != outd["status"][cont]).sum()),
            "outer_iters": int((outc["outer_iters"][cont] != outd["outer_iters"][cont]).sum())},
        "passed_through_identical": outc[~cont].tobytes() == out20[~cont].tobytes(),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fixed", type=int, default=4096)
    ap.add_argument("--sweep", type=int, default=8192)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    eng = tb.Engine(0)
    sm, name = eng.device_info()
    line = {"tool": "mc_continue_bench", "device": name, "power_limit": power_limit(),
            "mc_fixed_orbit": ensemble(eng, "mc_fixed_orbit", a.fixed), "mc_sweep": ensemble(eng, "mc_sweep", a.sweep)}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(s + "\n")
    eng.close()


if __name__ == "__main__":
    main()
