"""Disturbance ensembles of a kept Monte-Carlo run (ts_mc_replay_ensemble) on bench.py's ensembles -> one JSON line.

  1. the fixed-orbit ensemble (bench.make_trials("mc_fixed_orbit", 4096, 0)), kept with keep_trajectories = 1, at
     n_real = 32 and 256: device ms of the gains (K4a + K4b) and of the ensemble replay (K4e), replays/s, replay-steps/s,
     FLOPs per replay-step (profiles/flop_counts_r2.json, tools/flopcount.cpp) and the achieved share of the FP64 peak
     measured by ts_fp64_peak_probe, the histogram of the per-trial fail rates;
  2. against it, alternated in the same process, the loop a user has without the entry: n_real calls of
     ts_tvlqr_sim_batch (seed + r) on device-resident copies of the kept trajectories, summed ts_last_kernel_ms;
  3. the sweep (("mc_sweep", 8192, 0)) at n_real = 32.
The card name and power limit are read in the same call.
Usage: python tools/replay_ensemble_bench.py [--out FILE] [--fixed N] [--sweep N] [--loop-real R]"""
import argparse
import ctypes as C
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


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as ex:  # pragma: no cover
        return "unknown (%s)" % ex


def n_sim(cfg, tf, N):
    rl = lambda a, st, b: 0 if b < a else int(np.floor((b - a) / st + 1e-9)) + 1
    ns = rl(cfg.t0, cfg.dt, tf)
    if ns > N:
        ns = rl(cfg.t0, cfg.dt, tf - cfg.dt)
    return min(ns, N)


def qmult(a, b):
    s1, v1, s2, v2 = a[0], a[1:], b[0], b[1:]
    return np.concatenate([[s1 * s2 - v1 @ v2], s1 * v2 + s2 * v1 + np.cross(v1, v2)])


def flops_per_step():
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "flop_counts_r2.json")))
        return d.get("ensemble_replay_step")
    except Exception:
        return None


def fail_hist(slew, tf):
    fails = slew == tf[:, None]
    rate = fails.mean(axis=1)
    h, _ = np.histogram(rate, bins=[0, 1e-12, 0.05, 0.25, 0.5, 0.75, 1 - 1e-12, 1.0 + 1e-12])
    return dict(zip(["0", "(0,0.05)", "[0.05,0.25)", "[0.25,0.5)", "[0.5,0.75)", "[0.75,1)", "1"], [int(v) for v in h])), \
        float(fails.mean())


def workload(eng, name, n, reals, loop_real, peak, fl):
    import torch
    tr = B.make_trials(name, n, 0)
    cfg = B.mc_config(host, tr, n)
    fo = B.field_opts_array(tr)
    sid = np.arange(n).astype(np.uint32)
    cfg.keep_trajectories = 1
    out, st = eng.monte_carlo_run(cfg, tr["kep"], fo, tr["x0"], tr["xf"], tr["Jm"], q_noise0=tr["qn"], stream_id=sid)
    act = np.nonzero(out["status"] != 5)[0]
    steps = sum(n_sim(cfg, out["t_final"][t], int(out["N"][t])) - 1 for t in act)
    res = dict(workload=name, n_trials=n, active=int(act.size), ms_tvlqr_run=st.ms_tvlqr, ms_solve_run=st.ms_solve,
               replay_steps_per_realisation=int(steps))
    eng.mc_replay_ensemble(n, 32)   # warm-up
    # the loop of ts_tvlqr_sim_batch calls on device-resident kept trajectories
    loop = None
    if loop_real:
        k = eng.mc_trajectories(n, want=("X", "U", "B_eci"))
        ko, ro = k["knot_offs"], k["row_offs"]
        dX = torch.from_numpy(k["X"]).cuda()
        dU = torch.from_numpy(k["U"]).cuda()
        dB = torch.from_numpy(k["B_eci"]).cuda()
        N = out["N"][act].astype(np.int64)
        offs = np.ascontiguousarray(ko[act], dtype=np.int64)
        x0l = np.zeros((act.size, 8))
        for a, t in enumerate(act):
            qn = tr["qn"][t]
            th = np.linalg.norm(qn)
            x0l[a, :3] = tr["x0"][t, :3]
            x0l[a, 3:7] = qmult(tr["x0"][t, 3:7], np.concatenate([[np.cos(th / 2)], qn / th * np.sin(th / 2)]))
        arrs = dict(N=N, offs=offs, x0l=x0l, J=np.ascontiguousarray(tr["Jm"][act]), Bo=np.ascontiguousarray(ro[act], dtype=np.int64),
                    Br=2 * N, isc=N.astype(float), cr=np.full(act.size, 1.0 / (cfg.tf - cfg.t0)), tf=np.ascontiguousarray(out["t_final"][act]),
                    qf=np.ascontiguousarray(tr["xf"][act, 3:7]), sid=np.ascontiguousarray(sid[act]))
        l_nsim, l_slew = np.zeros(act.size, dtype=np.int64), np.zeros(act.size)   # the loop's outputs (discarded)
        g = host.TvlqrOpts.from_buffer_copy(cfg.tvlqr)
        g.dt, g.t0, g.literal_postproc, g.noise_mode = cfg.dt, cfg.t0, 0, 2
        p = lambda a: a.ctypes.data
        torch.cuda.synchronize()

        def loop_ms(R):
            ms = 0.0
            for r in range(R):
                g.seed = int(cfg.tvlqr.seed) + r
                rc = eng.lib.ts_tvlqr_sim_batch(eng.h, act.size, p(arrs["N"]), p(arrs["offs"]), dX.data_ptr(), dU.data_ptr(), p(arrs["x0l"]),
                                                p(arrs["J"]), dB.data_ptr(), p(arrs["Bo"]), p(arrs["Br"]), p(arrs["isc"]), p(arrs["cr"]),
                                                p(arrs["tf"]), p(arrs["qf"]), p(arrs["sid"]), C.byref(g), None, None, None, None, None,
                                                p(l_nsim), p(l_slew), 1)
                assert rc == 0, eng.lib.ts_last_error(eng.h)
                ms += eng.last_kernel_ms()
            return ms
        loop_ms(2)   # warm-up
        loop = []
    rows = []
    for R in reals:
        rec = dict(n_real=R, gains_ms=[], replay_ms=[], total_ms=[])
        for rep in range(2):
            slew, _ = eng.mc_replay_ensemble(n, R)
            gms, rms = eng.mc_replay_ensemble_split()
            rec["gains_ms"].append(gms)
            rec["replay_ms"].append(rms)
            rec["total_ms"].append(eng.last_kernel_ms())
            if loop is not None and R == loop_real:
                loop.append(loop_ms(R))
        rms = min(rec["replay_ms"])
        rec["replays_per_s"] = act.size * R / (rms / 1e3)
        rec["replay_steps_per_s"] = steps * R / (rms / 1e3)
        if fl:
            rec["flops_per_replay_step"] = fl
            rec["fp64_share_of_peak"] = fl * steps * R / (rms / 1e3) / (peak * 1e12)
        rec["fail_rate_hist"], rec["mean_fail_rate"] = fail_hist(slew[act], out["t_final"][act])
        rec["realisation0_equals_run"] = bool(np.array_equal(slew[act, 0], out["slew_time"][act]))
        rows.append(rec)
    res["ensemble"] = rows
    if loop is not None:
        ens = [r for r in rows if r["n_real"] == loop_real][0]
        res["sim_batch_loop"] = dict(n_real=loop_real, total_ms=loop, ensemble_total_ms=ens["total_ms"],
                                     speedup=min(loop) / min(ens["total_ms"]))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--fixed", type=int, default=4096)
    ap.add_argument("--sweep", type=int, default=8192)
    ap.add_argument("--loop-real", type=int, default=256)
    a = ap.parse_args()
    eng = tb.Engine(0)
    peak = eng.fp64_peak_tflops()
    fl = flops_per_step()
    res = dict(card=card(), fp64_peak_tflops_probe=peak)
    res["fixed_orbit"] = workload(eng, "mc_fixed_orbit", a.fixed, (32, 256), a.loop_real, peak, fl)
    if a.sweep:
        res["sweep"] = workload(eng, "mc_sweep", a.sweep, (32,), 0, peak, fl)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
