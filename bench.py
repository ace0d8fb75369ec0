#!/usr/bin/env python3
"""bench.py -- MC slew trials/sec (AL-iLQR + rollout) on N B200s, one process per GPU.

A "step" is one pass of the hot path (ts_monte_carlo_run: scoping field -> gramian cutoff -> fine field table ->
eigen-axis/Bryson weights -> AL-iLQR -> TVLQR replay -> slew-time rule, then the NCCL gather of outcome records +
statistics) over one ensemble of synthetic trials.

Workloads (config.workload):
  mc_fixed_orbit  BASELINE configs[2]: 4,096 slews per GPU, random initial attitudes (uniform on S^3), fixed LEO orbit
                  of src/monte_carlo.jl:122-127 (RAAN 0, anomaly 90), 1U inertia, tf 2400 s, cutoff 30, alpha 0.1.  [default]
  mc_sweep        BASELINE configs[3]: 8,192 slews per GPU (65,536 on 8) with per-trial inclination / altitude / RAAN /
                  anomaly / MJD / IGRF date (magnetic-diversity sweep, heatmap.jl:114-123), cutoff 100.
  tvlqr16k        BASELINE configs[4]: K4 alone -- closed-loop TVLQR tracking (attitude_controller.jl:1-48 with
                  simulator.jl / gain_simulator.jl) of 2,048 optimised sweep slews per GPU (16,384 on 8), Philox draws.
  igrf            BASELINE configs[1]: 10^8 random LEO points through K1 (evals/s).
The default line also carries `sweep`, `tvlqr16k` and `igrf12` blocks (one timed pass each) unless --no-extras.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--trials T] [--dump-outputs DIR]
For N > 1 launch under torchrun (one rank per GPU).  Rank 0 prints ONE JSON line.
--impl reference: the reference algorithm on the host cores (the C++ oracle; Julia is not in the image), rank 0 only.
--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step returned as DIR/<name>.npy (float64), so
  that two builds can be compared output by output on identical seeded inputs.  row.npy holds the row of the full output
  each dumped row comes from; outputs over 64 MB in all are a fixed seeded sample of rows.
    mc_fixed_orbit, mc_sweep  one file per outcome-record field (status ... flops) of the gathered outcomes, and
                              stats.npy (the reduced statistics vector, fields in parallel.STAT_FIELDS order)
    tvlqr16k                  n_sim.npy, slew_time.npy per slew
    igrf                      B_north.npy, B_east.npy, B_down.npy (nT) per point of rank 0
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)

GM = 3.986004418E14 * (1 / 1000) ** 3
J_1U = np.diag([0.00125] * 3)
QF = np.array([math.sqrt(2) / 2, math.sqrt(2) / 2, 0.0, 0.0])   # monte_carlo.jl:114
SEED = 0x5EED
FIELD_OPTS_DTYPE = np.dtype([("GM", "<f8"), ("mjd", "<f8"), ("igrf_date", "<f8"), ("field_radius_m", "<f8"), ("t0", "<f8"),
                             ("tf", "<f8"), ("N", "<i8")])
# Algorithmic FLOP per unit (DESIGN.md section 4).  Three models, all reported: (1) COUNTED kernel math -- the 7-state
# JVP-linearisation + dense Riccati + rollout arithmetic the kernels execute, counted with an instrumented scalar
# (tools/flopcount.cpp -> profiles/flop_counts_r2.json): the roofline numerator; (2) the same count on the oracle = the
# literal reference algorithm (8-state, 11-seed forward-mode duals); (3) SURVEY 8d's round-1 ESTIMATE (6100 / 500).
FL_ITER, FL_ROLL, FL_TVLQR, FL_IGRF = 6100.0, 500.0, 7700.0, 2243.0
FL_MODELS = {"survey_estimate": (6100.0, 500.0)}
try:
    _fc = json.load(open(os.path.join(ROOT, "profiles", "flop_counts_r2.json")))
    # the benchmark ensembles use the 1U inertia (diagonal): K3 runs its diagonal-inertia instantiations
    FL_ITER, FL_ROLL = float(_fc["per_knot_iteration_diag"]), float(_fc["per_rollout_knot_diag"])
    FL_TVLQR = float(_fc.get("tvlqr_per_knot", FL_TVLQR))
    FL_MODELS["reference_algorithm_counted"] = (float(_fc["oracle_per_knot_iteration"]), float(_fc["oracle_per_rollout_knot"]))
    FL_MODELS["general_inertia_kernels_counted"] = (float(_fc["per_knot_iteration"]), float(_fc["per_rollout_knot"]))
    FL_MODELS["first_round2_count"] = (float(_fc["first_round2_count"]["per_knot_iteration"]), float(_fc["first_round2_count"]["per_rollout_knot"]))
    FLOP_SOURCE = "counted kernel math (diagonal-inertia instantiation), %.0f FLOP per knot-iteration (JVP linearisation %d + cost gradients " \
                  "%d + Riccati step %d + gradient measure %d) + %.0f per line-search rollout knot: tools/flopcount.cpp -> " \
                  "profiles/flop_counts_r2.json" % (FL_ITER, _fc["linearise_diag"], _fc["cost_gradients"], _fc["riccati"],
                                                   _fc["gradient_measure"], FL_ROLL)
except Exception:
    FLOP_SOURCE = "SURVEY 8d estimate: 6100 per knot-iteration (rk3 Jacobian 2600 + Riccati step 3500) + 500 per rollout knot"
# HBM traffic of K3 per knot-iteration: ncu dram__bytes_read+write of THIS configuration (N = 2044, 4096 trials)
K3_TRAFFIC = {"bytes_per_knot_iter": 1650.0, "source": "profiles/k3_traffic_r3.csv"}
try:
    K3_TRAFFIC = json.load(open(os.path.join(ROOT, "profiles", "k3_traffic_r3.json")))
except Exception:
    pass
STATUS = ["converged", "max_outer", "cost_blowup", "reg_max", "nan", "no_cutoff"]
DUMP_BYTES = 60 << 20                # --dump-outputs: array data of all files; with the .npy headers < 64 MB


def dump_rows(n, row_bytes, budget=DUMP_BYTES):
    """Rows of an n-row output that --dump-outputs writes: all of them, or a fixed seeded sample within `budget` bytes."""
    cap = budget // row_bytes
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(SEED).choice(n, size=cap, replace=False, shuffle=False))


def write_dump(directory, arrays):
    """directory/<name>.npy in float64 for every array."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    assert sum(v.nbytes for v in arrays.values()) <= DUMP_BYTES
    os.makedirs(directory, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), v)


# --------------------------------------------------------------------------- synthetic ensembles
def make_trials(workload, n, rank, seed=SEED):
    """Synthetic inputs of one rank's shard; reproducible from (seed, rank)."""
    rng = np.random.default_rng([seed, rank])
    q0 = rng.normal(size=(n, 4))
    q0 /= np.linalg.norm(q0, axis=1, keepdims=True)               # uniform on S^3
    x0 = np.concatenate([np.zeros((n, 3)), q0, np.zeros((n, 1))], axis=1)
    xf = np.tile(np.concatenate([[0, 0, 0], QF, [1.0]]), (n, 1))
    Jm = np.tile(J_1U.reshape(-1), (n, 1))
    qn = rng.normal(size=(n, 3)) * (math.pi / 180) ** 2           # TortoiseSat.jl:231
    if workload == "mc_fixed_orbit":
        kep = np.array([[0.0, 400.0 + 6371.0, 96.6, 0.0, 0.0, 90.0]])
        fo = [(GM, 58155.0, 2019.0, (400.0 + 6371.0) * 1000.0, 0.0, 0.0, 0)]
        shared, cutoff = True, 30.0
    else:                                                           # mc_sweep (SURVEY 8d config 4)
        alt = rng.uniform(350, 800, size=n)
        kep = np.stack([np.zeros(n), alt + 6371.0, rng.uniform(0, 98, size=n), rng.uniform(0, 360, size=n), np.zeros(n),
                        rng.uniform(0, 360, size=n)], axis=1)
        fo = [(GM, rng.uniform(58155, 58520), 2015 + 5 * rng.random(), (a + 6371.0) * 1000.0, 0.0, 0.0, 0) for a in alt]
        shared, cutoff = False, 100.0
    return dict(kep=kep, fo=fo, x0=x0, xf=xf, Jm=Jm, qn=qn, shared=shared, cutoff=cutoff)


def field_opts_array(tr):
    fo = np.zeros(len(tr["fo"]), dtype=FIELD_OPTS_DTYPE)
    for i, f in enumerate(tr["fo"]):
        fo[i] = f
    return fo


def mc_config(host, tr, n):
    """Constants of src/monte_carlo.jl: tf 2400, N 5000, dt 0.2, alpha 0.1, beta 1e3, TVLQR Q 10 / Qf 1000 / R 0.5e3 (:216-227)."""
    cfg = host.default_mc_config(n, shared_orbit=tr["shared"], run_tvlqr=True, tf=2400.0, N_scope=5000, cutoff=tr["cutoff"], dt=0.2,
                                 alpha=0.1, beta=1e3)
    cfg.tvlqr.noise_mode = 2
    cfg.tvlqr.seed = SEED
    return cfg


def workload_name(workload, n, points=0):
    if workload == "igrf":
        return "igrf (BASELINE configs[1]): %d random LEO points per GPU, date 2019.0" % points
    if workload == "tvlqr16k":
        return "tvlqr16k (BASELINE configs[4]): closed-loop TVLQR tracking of %d optimised sweep slews per GPU, Philox disturbance draws " \
               "in every rk4 stage, Q 10 / Qf 1000 / R 0.5e3, dt 0.2" % n
    return "%s (BASELINE configs[%d]): %d slews per GPU, 1U inertia, tf 2400 s, cutoff %g, alpha 0.1, goal_mask 0x7F, " \
           "AL-iLQR 20x50, TVLQR replay with Philox noise" % (workload, 2 if workload == "mc_fixed_orbit" else 3, n,
                                                              30.0 if workload == "mc_fixed_orbit" else 100.0)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.gpu, self.rows, self.p = gpu, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.p:
            self.p.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# --------------------------------------------------------------------------- CPU baseline (oracle): reference arm + cpu_baseline
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_mc_sample(workload, n_ensemble, idx, nthreads):
    """The reference algorithm (CPU oracle: C++ restatement, Julia is not available) on the trials `idx` of the workload's
    ensemble: whole per-trial pipeline inside one OpenMP region, schedule(dynamic,1).  Touches only oracle/.
    Returns (wall seconds, per-trial CPU seconds, outcomes)."""
    from oracle import oracle as orc
    tr = make_trials(workload, n_ensemble, 0)
    idx = np.asarray(idx)
    cfg = orc.mc_config(len(idx), shared_orbit=tr["shared"], run_tvlqr=True, tf=2400.0, N_scope=5000, cutoff=tr["cutoff"], dt=0.2,
                        alpha=0.1, beta=1e3, noise_mode=2, seed=SEED, R_lqr=0.5e3)
    fo = field_opts_array(tr)
    kep = tr["kep"] if tr["shared"] else tr["kep"][idx]
    fo = fo if tr["shared"] else fo[idx]
    t0 = time.perf_counter()
    out, secs = orc.mc_run(cfg, kep, fo, tr["x0"][idx], tr["xf"][idx], tr["Jm"][idx], q_noise0=tr["qn"][idx],
                           stream_id=idx.astype(np.uint32), nthreads=nthreads)
    return time.perf_counter() - t0, secs, out


def cpu_igrf_sample(n, nthreads):
    from oracle import oracle as orc
    rng = np.random.default_rng(SEED)
    lat = np.arcsin(2 * rng.random(n) - 1)
    lon = math.pi * (2 * rng.random(n) - 1)
    r = 6371200.0 + 300000.0 + 900000.0 * rng.random(n)
    t0 = time.time()
    orc.igrf12_batch(2019.0, r, lat, lon, nthreads=nthreads)
    dt = time.time() - t0
    return n / dt, dt


def reference_arm(a, cores, metric, unit):
    """--impl reference: honours --steps / --warmup; every step is a bounded, strided sample of the ensemble sized so that
    the whole run stays within a few minutes (the line reports the step counts really run).  value = cores x trials / (sum of per-trial CPU seconds): the throughput of
    the host with every core kept busy (a small sample's wall clock would be its slowest trial)."""
    from oracle import oracle as orc
    orc.build()
    steps, warm = max(1, a.steps), max(0, a.warmup)
    if a.workload == "igrf":
        n = 2_000_000
        vals, walls = [], []
        for i in range(warm + steps):
            v, dt = cpu_igrf_sample(n, cores)
            if i >= warm:
                vals.append(v)
                walls.append(dt)
        v = float(np.mean(vals))
        sample = "%d of the 1e8 points per step, oracle igrf12 (C++ restatement of src/igrf.jl), %d OpenMP threads" % (n, cores)
        ms = 1e3 * float(np.mean(walls))
        extra = {}
    else:
        wl = a.workload if a.workload in ("mc_fixed_orbit", "mc_sweep") else "mc_fixed_orbit"
        n_ens = a.trials or (4096 if wl == "mc_fixed_orbit" else 8192)
        # A trial costs 1..50 CPU-seconds (mean ~9) and cannot be truncated, so the number of steps that fit a few minutes is
        # bounded: steps are run until `budget` seconds of wall clock are used (at least one), and the counts REALLY run are
        # what the line reports.
        budget = 200.0
        n_s = 2 * cores
        stride = max(1, n_ens // n_s)
        warm = min(warm, 1)
        walls, secs_all, n_done, t_begin, steps_run = [], [], 0, time.perf_counter(), 0
        for i in range(warm + steps):
            if i > warm and time.perf_counter() - t_begin > budget:
                break
            idx = (i + stride * np.arange(n_s)) % n_ens
            wall, secs, out = cpu_mc_sample(wl, n_ens, idx, cores)
            if i >= warm:
                walls.append(wall)
                secs_all.append(secs)
                n_done += n_s
                steps_run += 1
        steps = steps_run
        secs_all = np.concatenate(secs_all)
        v = cores * n_done / float(secs_all.sum())
        ms = 1e3 * float(np.mean(walls))
        sample = "%d trials per step taken by stride %d across the %d-trial ensemble (a different offset every step), whole pipeline " \
                 "(field, cutoff, AL-iLQR, TVLQR replay) in one OpenMP region with schedule(dynamic,1) on %d threads; value = cores x " \
                 "trials / sum of per-trial CPU seconds; C++ restatement of the reference algorithm (Julia unavailable)" % (
                     n_s, stride, n_ens, cores)
        extra = {"value_wall": n_done / float(np.sum(walls)), "cpu_seconds_per_trial_mean": float(secs_all.mean()),
                 "cpu_seconds_per_trial_max": float(secs_all.max()), "trials_timed": int(n_done)}
        a.trials = n_ens
    line = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": a.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(a.workload, a.trials, a.points), "trials_per_gpu": a.trials},
            "cpu_baseline": dict({"value": v, "unit": unit, "cores": cores, "kind": "port", "sample": sample}, **extra),
            "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="mc_fixed_orbit", choices=["mc_fixed_orbit", "mc_sweep", "tvlqr16k", "igrf"])
    ap.add_argument("--trials", type=int, default=0, help="trials per GPU (weak scaling); default 4096 / 8192 (sweep) / 2048 (tvlqr16k)")
    ap.add_argument("--points", type=int, default=100_000_000, help="igrf workload: points per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="default line without the sweep / tvlqr16k / igrf12 blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = host_cores()
    metric = "igrf12_evals_per_sec" if a.workload == "igrf" else ("tvlqr_slews_per_sec" if a.workload == "tvlqr16k" else "mc_slew_trials_per_sec")
    unit = "evals/s" if a.workload == "igrf" else ("slews/s" if a.workload == "tvlqr16k" else "trials/s")

    if a.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(a, cores, metric, unit)

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    import torch.distributed as dist
    import tortoisesat.jl_b200 as tb
    from tortoisesat.jl_b200 import host, parallel
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints a "NCCL version ..." banner on STDOUT when the first communicator is created; keep stdout
        # clean for the single JSON line by pointing fd 1 at stderr while the communicator comes up
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    eng = tb.Engine(local_rank)
    peak_fp64 = eng.fp64_peak_tflops()
    peak_src = "measured live: register-resident DFMA micro-benchmark (ts_fp64_peak_probe; MEASURED_PEAKS.json has no FP64 row; " \
               "nominal 148 SM x 64 DFMA/clk x 2 x 1.965 GHz = 37.2)"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        eng.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor(np.atleast_1d(np.asarray(x, dtype=np.float64)), dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.cpu().numpy() if t.numel() > 1 else float(t.item())

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"

    # ---- K1 throughput (BASELINE's second metric): device-resident inputs after their own warm-up, and host-buffer e2e
    def igrf_block(n, reps, with_e2e=True, dump=None):
        g = torch.Generator(device=dev).manual_seed(SEED + rank)
        u = torch.rand(3, n, generator=g, device=dev, dtype=torch.float64)
        lat = torch.asin(2 * u[0] - 1)
        lon = math.pi * (2 * u[1] - 1)
        r = 6371200.0 + 300000.0 + 900000.0 * u[2]
        del u
        o = [torch.empty(n, device=dev, dtype=torch.float64) for _ in range(3)]
        ms = []
        for i in range(3 + reps):
            eng.igrf12_batch(2019.0, r, lat, lon, out=o)
            if i >= 3:
                ms.append(eng.last_kernel_ms())
        if dump and rank == 0:
            eng.synchronize()
            rows = dump_rows(n, 4 * 8)
            sel = torch.from_numpy(rows).to(dev)
            write_dump(dump, dict(row=rows, **{k: b[sel].cpu().numpy() for k, b in zip(("B_north", "B_east", "B_down"), o)}))
        kms = max_over_ranks(float(np.mean(ms)))
        blk = {"evals_per_s": world * n / (kms * 1e-3), "points_per_gpu": n, "ms": kms,
               "roofline": {"bound": "fp64", "achieved": FL_IGRF * n / (kms * 1e-3) / 1e12, "peak": peak_fp64, "unit": "TFLOP/s",
                            "frac": FL_IGRF * n / (kms * 1e-3) / 1e12 / peak_fp64, "hbm_gbs_algorithmic": 48.0 * n / (kms * 1e-3) / 1e9}}
        if with_e2e:
            n_e = min(n, 20_000_000)
            pin = [torch.empty(n_e, dtype=torch.float64).pin_memory() for _ in range(6)]
            for dst, src in zip(pin[:3], (r, lat, lon)):
                dst.copy_(src[:n_e])
            hin = [x.numpy() for x in pin[:3]]
            hout = [x.numpy() for x in pin[3:]]
            for _ in range(2):
                eng.igrf12_batch(2019.0, hin[0], hin[1], hin[2], out=hout)
            barrier()
            t0 = time.perf_counter()
            for _ in range(3):
                eng.igrf12_batch(2019.0, hin[0], hin[1], hin[2], out=hout)
            barrier()
            e2e_s = max_over_ranks(time.perf_counter() - t0) / 3
            blk["e2e"] = {"value": world * n_e / e2e_s, "unit": "evals/s", "h2d_bytes_per_step": 24 * n_e, "d2h_bytes_per_step": 24 * n_e,
                          "note": "%d points per call through ts_igrf12_batch with pinned HOST buffers (H2D + kernel + D2H inside the "
                                  "call, chunked double-buffered pipeline): PCIe-bound" % n_e}
        del r, lat, lon, o
        return blk

    if a.workload == "igrf":
        n = a.points
        clk = ClockSampler(local_rank)
        clk.start()
        l0 = eng.launch_count()
        blk = igrf_block(n, a.steps, dump=a.dump_outputs)
        launches = eng.launch_count() - l0
        clocks = clk.stop()
        line = {"metric": metric, "value": blk["evals_per_s"], "unit": unit, "n_gpus": world, "steps": a.steps, "warmup": 3,
                "ms_per_step": blk["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": {"workload": workload_name("igrf", 0, n), "l2": "inputs+outputs 4.8 GB per GPU > L2"},
                "roofline": dict(blk["roofline"], traffic=None, peak_source=peak_src, hbm_peak_gbs=hbm_peak), "e2e": blk["e2e"],
                "gpu_launches": launches, "clocks": clocks}
        if rank == 0 and not a.no_cpu_baseline:
            from oracle import oracle as orc
            orc.build()
            v, dt = cpu_igrf_sample(4_000_000, cores)
            line["cpu_baseline"] = {"value": v, "unit": unit, "cores": cores, "kind": "port",
                                    "sample": "4e6 of the points, oracle igrf12 (C++ restatement of src/igrf.jl), OpenMP"}
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- Monte-Carlo workloads ------------------------------------------------------------------------------------
    def mc_pass(workload, n, steps, warmup, keep=False, dump=None):
        """`warmup` untimed + `steps` timed passes of ts_monte_carlo_run over this rank's shard; returns a result dict."""
        tr = make_trials(workload, n, rank)
        cfg = mc_config(host, tr, n)
        cfg.keep_trajectories = 1 if keep else 0
        fo = field_opts_array(tr)
        sid = (np.arange(n) + rank * n).astype(np.uint32)

        def step():
            t0 = time.perf_counter()
            out, st = eng.monte_carlo_run(cfg, tr["kep"], fo, tr["x0"], tr["xf"], tr["Jm"], q_noise0=tr["qn"], stream_id=sid)
            t_call = time.perf_counter() - t0
            allout = parallel.gather_outcomes(out, device=dev)          # NCCL all-gather of 64-byte records
            vec = parallel.reduce_stats(parallel.stats_vector(st), device=dev)
            return out, st, allout, vec, t_call

        for _ in range(warmup):
            step()
        barrier()
        l0 = eng.launch_count()
        t0 = time.perf_counter()
        acc = {k: [] for k in ("dev_ms", "call_s", "field", "prep", "solve", "tvlqr", "flops", "p_ms", "s_ms", "parked", "ki", "kr")}
        last = None
        for _ in range(steps):
            out, st, allout, vec, t_call = step()
            acc["dev_ms"].append(st.ms_field + st.ms_prep + st.ms_solve + st.ms_tvlqr)
            acc["call_s"].append(t_call)
            for k in ("field", "prep", "solve", "tvlqr"):
                acc[k].append(getattr(st, "ms_" + k))
            kn = (out["N"] - 1).astype(np.float64)
            acc["flops"].append(float(np.sum(kn * (out["inner_iters"] * FL_ITER + out["ls_rollouts"] * FL_ROLL))))
            acc["ki"].append(float(np.sum(kn * out["inner_iters"])))
            acc["kr"].append(float(np.sum(kn * out["ls_rollouts"])))
            sp = eng.k3_last_split()
            acc["p_ms"].append(sp[0])
            acc["s_ms"].append(sp[1])
            acc["parked"].append(sp[2])
            last = (out, st, allout, vec)
        barrier()
        wall = max_over_ranks(time.perf_counter() - t0)
        launches = eng.launch_count() - l0
        out, st, allout, vec = last
        if dump and rank == 0:
            fields = host.OUTCOME_DTYPE.names
            rows = dump_rows(len(allout), 8 * (1 + len(fields)), DUMP_BYTES - vec.nbytes)
            write_dump(dump, dict(row=rows, stats=vec, **{f: allout[f][rows] for f in fields}))
        dev_s = max_over_ranks(float(np.mean(acc["dev_ms"])) * 1e-3)      # device time of the kernels (CUDA events), max over ranks
        solve_s = float(np.mean(acc["solve"])) * 1e-3
        act = allout["status"] != 5
        it = allout["inner_iters"][act].astype(np.float64)
        hist = np.bincount(allout["status"], minlength=6)[:6]
        knot_iters = float(np.sum((out["N"] - 1).astype(np.float64) * out["inner_iters"]))
        ach = float(np.mean(acc["flops"])) / solve_s / 1e12
        total = world * n
        res = dict(
            tr=tr, cfg=cfg, fo=fo, sid=sid, out=out, value=total / dev_s, e2e=total / (wall / steps), wall_step_s=wall / steps, launches=launches,
            stage_ms={k: float(np.mean(acc[k])) for k in ("field", "prep", "solve", "tvlqr")},
            k3_split={"persistent_ms": float(np.mean(acc["p_ms"])), "straggler_ms": float(np.mean(acc["s_ms"])),
                      "handed_over": float(np.mean(acc["parked"]))},
            results={"status": {STATUS[k]: int(hist[k]) for k in range(6)}, "trials": int(total),
                     "knots_mean": float(allout["N"][act].mean()) if act.any() else 0.0, "knots_max": int(allout["N"].max()),
                     "inner_iters_mean": float(it.mean()) if it.size else 0.0,
                     "inner_iters_quantiles_50_75_90_95_99_100": np.percentile(it, [50, 75, 90, 95, 99, 100]).tolist() if it.size else [],
                     "outer_iters_quantiles_50_90_100": np.percentile(allout["outer_iters"][act], [50, 90, 100]).tolist() if act.any() else [],
                     "ls_rollouts_mean": float(allout["ls_rollouts"][act].mean()) if act.any() else 0.0,
                     "slew_fail": int(vec[3]), "mean_slew_time_s": float(vec[4] / max(1.0, vec[0] - vec[2]))},
            roofline={"bound": "fp64", "kernel": "K3 AL-iLQR solve: k3_alilqr_diag_kernel (4 trials per warp) + k3_wide_diag_kernel (one warp per straggler): the diagonal-inertia instantiations of k3_alilqr_kernel / k3_wide_kernel",
                      "achieved": ach, "peak": peak_fp64, "unit": "TFLOP/s", "frac": ach / peak_fp64,
                      "traffic": K3_TRAFFIC["bytes_per_knot_iter"] * knot_iters, "traffic_source": "%s: %.0f B per knot-iteration (ncu "
                      "dram__bytes_read+write of this configuration) x this run's knot-iterations" % (K3_TRAFFIC["source"], K3_TRAFFIC["bytes_per_knot_iter"]),
                      "hbm_gbs_from_traffic": K3_TRAFFIC["bytes_per_knot_iter"] * knot_iters / solve_s / 1e9, "hbm_peak_gbs": hbm_peak,
                      "hbm_peak_source": hbm_src, "peak_source": peak_src, "flop_model": FLOP_SOURCE,
                      "frac_other_flop_models": {k: (float(np.mean(acc["ki"])) * v[0] + float(np.mean(acc["kr"])) * v[1]) / solve_s / 1e12 / peak_fp64
                                                 for k, v in FL_MODELS.items()},
                      "kernel_share_of_step": solve_s / float(np.mean(acc["dev_ms"]) * 1e-3)})
        res["h2d"] = int(n * (8 + 8 + 9 + 3) * 8 + n * 4 + len(fo) * (6 * 8 + 56))
        res["d2h"] = int(n * 64 + 8 * len(fo))
        return res

    def tvlqr_block(n_tv, reps, dump=None):
        """K4 alone on the first n_tv optimised slews of the run whose trajectories are resident (keep_trajectories)."""
        tj = eng.mc_trajectories(last_sweep["n"], want=("X", "U", "B_eci"))
        ko, ro = tj["knot_offs"], tj["row_offs"]
        out, tr = last_sweep["out"], last_sweep["tr"]
        ok = np.nonzero(out["status"] != 5)[0][:n_tv]
        n_ok = len(ok)
        N_i = out["N"][ok].astype(np.int64)
        offs = np.concatenate([[0], np.cumsum(N_i)])
        X = np.concatenate([tj["X"][ko[t]:ko[t + 1]] for t in ok])
        U = np.concatenate([tj["U"][ko[t]:ko[t + 1]] for t in ok])
        rows = 2 * N_i
        B = np.concatenate([tj["B_eci"][ro[t]:ro[t] + 2 * out["N"][t]] for t in ok])
        B_offs = np.concatenate([[0], np.cumsum(rows)])[:-1]
        x0l = tr["x0"][ok].copy()
        x0l[:, 7] = 0.0
        opts = host.default_tvlqr_opts()
        opts.noise_mode, opts.seed = 2, SEED
        for i in range(3):
            opts.Rd[i] = 0.5e3
        args = (N_i, X, U, x0l, tr["Jm"][ok], B, B_offs, rows, N_i.astype(np.float64), np.full(n_ok, 1.0 / 2400.0), out["t_final"][ok],
                tr["xf"][ok, 3:7])
        kms, walls = [], []
        for i in range(1 + reps):
            t0 = time.perf_counter()
            r = eng.tvlqr_sim_batch(*args, opts=opts, stream_id=(ok + rank * last_sweep["n"]).astype(np.uint32), want_traj=False)
            if i >= 1:
                walls.append(time.perf_counter() - t0)
                kms.append(eng.last_kernel_ms())
        if dump and rank == 0:
            rows = dump_rows(n_ok, 3 * 8)
            write_dump(dump, dict(row=rows, n_sim=r[4][rows], slew_time=r[5][rows]))
        k_s = max_over_ranks(float(np.mean(kms)) * 1e-3)
        w_s = max_over_ranks(float(np.mean(walls)))
        knots = float(np.sum(N_i - 1))
        fails = int(np.sum(r[5] == out["t_final"][ok]))
        return {"workload": workload_name("tvlqr16k", n_ok), "slews_per_s": world * n_ok / k_s, "ms": k_s * 1e3, "slews_per_gpu": int(n_ok),
                "knots_mean": float(N_i.mean()), "slew_fail": int(sum_over_ranks(fails)),
                "roofline": {"bound": "fp64", "kernel": "K4 replay: k4a_linearise (thread per knot) + k4b_riccati + k4n_records + k4c_replay (thread per slew)", "achieved": FL_TVLQR * knots / k_s / 1e12, "peak": peak_fp64,
                             "unit": "TFLOP/s", "frac": FL_TVLQR * knots / k_s / 1e12 / peak_fp64,
                             "flop_model": "%.0f FLOP per knot (rk4 Jacobian with the dt^2 quirk, G(q) projection, 6x6 Riccati, 4 noisy dynamics calls)" % FL_TVLQR,
                             "hbm_gbs_algorithmic": (11 + 9 + 18 * 2) * 8 * knots / k_s / 1e9},
                "e2e": {"value": world * n_ok / w_s, "unit": "slews/s", "h2d_bytes_per_step": int((X.size + U.size + B.size) * 8),
                        "d2h_bytes_per_step": int(n_ok * 16), "note": "ts_tvlqr_sim_batch with HOST trajectories (X, U, field tables uploaded inside the call)"}}

    last_sweep = {}
    clk = ClockSampler(local_rank)
    clk.start()
    if a.workload == "tvlqr16k":
        n_sw = 2 * (a.trials or 2048)
        sw = mc_pass("mc_sweep", n_sw, 1, 0, keep=True)
        last_sweep.update(n=n_sw, out=sw["out"], tr=sw["tr"])
        blk = tvlqr_block(a.trials or 2048, a.steps, dump=a.dump_outputs)
        clocks = clk.stop()
        line = {"metric": metric, "value": blk["slews_per_s"], "unit": unit, "n_gpus": world, "steps": a.steps, "warmup": 1,
                "ms_per_step": blk["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": blk["workload"], "trials_per_gpu": blk["slews_per_gpu"]}, "roofline": blk["roofline"], "e2e": blk["e2e"],
                "gpu_launches": a.steps, "clocks": clocks}
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return 0

    n = a.trials or (4096 if a.workload == "mc_fixed_orbit" else 8192)
    main_r = mc_pass(a.workload, n, a.steps, a.warmup, dump=a.dump_outputs)
    clocks = clk.stop()
    line = {"metric": metric, "value": main_r["value"], "unit": unit, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": main_r["wall_step_s"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_name(a.workload, n), "trials_per_gpu": n},
            "results": dict(main_r["results"], l2="per-GPU K3 working set (arena + parked state + regions) >> L2 (126 MB): no flush needed"),
            "roofline": main_r["roofline"],
            "e2e": {"value": main_r["e2e"], "unit": unit, "h2d_bytes_per_step": main_r["h2d"], "d2h_bytes_per_step": main_r["d2h"],
                    "note": "ts_monte_carlo_run with HOST per-trial inputs + outcome D2H + NCCL gather; trajectories stay in HBM"},
            "stage_ms": main_r["stage_ms"], "k3_split": main_r["k3_split"], "gpu_launches": main_r["launches"], "clocks": clocks,
            "fp64_peak_probe": {"tflops": peak_fp64, "sm_mhz": clocks.get("sm_mhz")}}

    if not a.no_extras:
        # second end-to-end figure: the same step with the trajectories the reference script keeps (states, control_inputs,
        # sim_states, sim_control_inputs: monte_carlo.jl:52-66) brought back to the host
        try:
            tr, cfg, fo, sid = main_r["tr"], main_r["cfg"], main_r["fo"], main_r["sid"]
            cfg.keep_trajectories = 1
            barrier()
            t0 = time.perf_counter()
            out, st = eng.monte_carlo_run(cfg, tr["kep"], fo, tr["x0"], tr["xf"], tr["Jm"], q_noise0=tr["qn"], stream_id=sid)
            tj = eng.mc_trajectories(n, want=("X", "U", "X_sim", "U_sim"))
            barrier()
            w = max_over_ranks(time.perf_counter() - t0)
            line["e2e_with_trajectories"] = {"value": world * n / w, "unit": unit, "h2d_bytes_per_step": main_r["h2d"],
                                             "d2h_bytes_per_step": int(main_r["d2h"] + sum(tj[k].nbytes for k in ("X", "U", "X_sim", "U_sim"))),
                                             "note": "one step + ts_mc_fetch_trajectories (X, U, X_sim, U_sim to pageable host arrays)"}
            cfg.keep_trajectories = 0
            del tj
        except Exception as ex:  # pragma: no cover
            line["e2e_with_trajectories"] = {"error": str(ex)}
        # BASELINE configs[3]: one timed pass of the magnetic-diversity sweep (8192 slews per GPU: 65,536 on 8 GPUs)
        if a.workload == "mc_fixed_orbit":
            try:
                n_sw = 8192 if n >= 4096 else 2 * n
                sw = mc_pass("mc_sweep", n_sw, 1, 0, keep=True)
                last_sweep.update(n=n_sw, out=sw["out"], tr=sw["tr"])
                line["sweep"] = {"workload": workload_name("mc_sweep", n_sw), "trials_per_s": sw["value"], "e2e_trials_per_s": sw["e2e"],
                                 "converged_per_s": sw["value"] * sw["results"]["status"]["converged"] / max(1, sw["results"]["trials"]),
                                 "results": sw["results"], "stage_ms": sw["stage_ms"], "k3_split": sw["k3_split"],
                                 "roofline_frac": sw["roofline"]["frac"], "steps": 1, "warmup": 0}
                # BASELINE configs[4]: K4 alone on 2,048 of those optimised slews per GPU (16,384 on 8 GPUs)
                line["tvlqr16k"] = tvlqr_block(2048 if n >= 4096 else n // 2, 3)
            except Exception as ex:  # pragma: no cover
                line.setdefault("sweep", {"error": str(ex)})
        # SURVEY 8(f2): the quaternion-aware solver variant the reference's Monte-Carlo script requests (monte_carlo.jl:158,192),
        # one pass over the same ensemble (the QUAT instantiations of both K3 kernels)
        if a.workload == "mc_fixed_orbit":
            try:
                tr, cfg, fo, sid = main_r["tr"], main_r["cfg"], main_r["fo"], main_r["sid"]
                cfg.ilqr.quat_error = 1
                barrier()
                out, st = eng.monte_carlo_run(cfg, tr["kep"], fo, tr["x0"], tr["xf"], tr["Jm"], q_noise0=tr["qn"], stream_id=sid)
                cfg.ilqr.quat_error = 0
                dev_s = max_over_ranks((st.ms_field + st.ms_prep + st.ms_solve + st.ms_tvlqr) * 1e-3)
                hist = np.bincount(out["status"], minlength=6)[:6]
                act = out["status"] != 5
                line["quaternion_variant"] = {"workload": workload_name(a.workload, n) + " with ts_ilqr_opts.quat_error = 1",
                                              "trials_per_s": world * n / dev_s, "ms_solve": st.ms_solve, "steps": 1, "warmup": 0,
                                              "status_rank0": {STATUS[k]: int(hist[k]) for k in range(6)},
                                              "inner_iters_mean_rank0": float(out["inner_iters"][act].mean()),
                                              "slew_fail_rank0": int(st.n_fail_slew)}
            except Exception as ex:  # pragma: no cover
                line["quaternion_variant"] = {"error": str(ex)}
        try:
            line["igrf12"] = igrf_block(100_000_000 if n >= 1024 else 1_000_000, 3)
        except Exception as ex:  # pragma: no cover
            line["igrf12"] = {"error": str(ex)}
    if rank == 0 and not a.no_cpu_baseline:
        from oracle import oracle as orc
        orc.build()
        ns = max(cores, 1) * 2
        stride = max(1, n // ns)
        wall, secs, _ = cpu_mc_sample(a.workload, n, (stride * np.arange(ns)) % n, cores)
        line["cpu_baseline"] = {"value": cores * ns / float(secs.sum()), "unit": unit, "cores": cores, "kind": "port", "value_wall": ns / wall,
                                "sample": "%d trials taken by stride %d across this rank's ensemble, whole pipeline in one OpenMP region "
                                          "(schedule(dynamic,1), %d threads), %.1f s wall; value = cores x trials / sum of per-trial CPU "
                                          "seconds; C++ restatement of the reference algorithm (Julia unavailable)" % (ns, stride, cores, wall)}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
