"""K8 measurement: prefilter time of the igrf_data map (n = 1000) and evaluation rate of ts_field_map_eval_batch at
10^8 seeded device-resident points, next to K1 (igrf12) on the same points.  Prints one JSON line (with the device
name and power limit) and, with --out FILE, writes it there too.

Traffic model (algorithmic, per point): 16 taps x 24 B of coefficients + 16 B of indices in + 24 B out.  The
coefficients of a 1000^2 map (24 MB; 32 MB in the kernel's padded copy, whose taps are 32 B each) stay in the 126 MB
L2, so only the 40 B of indices and outputs have to come from or go to DRAM; the taps are served by L2."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBS = 7.7            # B200 data sheet, one GPU
TAP_B, IN_B, OUT_B = 16 * 24, 16, 24
TAP_B_PADDED = 16 * 32             # what the kernel reads: one 256-bit load per tap


def gpu_power_limit(dev):
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        p, c = [v.strip() for v in r.stdout.strip().split(",")]
        return float(p), float(c)
    except Exception:
        return None, None


def timed(fn, eng, reps, warmup):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(reps):
        fn()
        ms.append(eng.last_kernel_ms())
    return statistics.median(ms), min(ms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=100_000_000)
    ap.add_argument("--n", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=0x5EED)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import tortoisesat.jl_b200 as tb
    if not torch.cuda.is_available():
        sys.exit("field_map_bench: no CUDA device (this measures the GPU; there is nothing to fall back to)")
    eng = tb.Engine(0)
    n, N = a.n, a.points
    grid = torch.from_numpy(tb.host.igrf_data(400, 2019, n=n).grid).cuda()
    coefs = torch.empty((n + 2, n + 2, 3), dtype=torch.float64, device="cuda")
    pre_med, pre_min = timed(lambda: eng.field_map_prefilter(grid, out=coefs), eng, a.reps, a.warmup)

    g = torch.Generator(device="cuda").manual_seed(a.seed)
    x0 = 1.0 + (n - 1) * torch.rand(N, generator=g, device="cuda", dtype=torch.float64)
    x1 = 1.0 + (n - 1) * torch.rand(N, generator=g, device="cuda", dtype=torch.float64)
    out = torch.empty((N, 3), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ev_med, ev_min = timed(lambda: eng.field_map_eval_batch(coefs, x0, x1, out=out), eng, a.reps, a.warmup)
    del out

    # K1 at the same points: the map's node i / j sits at lat -pi/2 + (i-1) pi/(n-1), long -pi + (j-1) 2pi/(n-1)
    lat = -math.pi / 2 + (x0 - 1.0) * (math.pi / (n - 1))
    lon = -math.pi + (x1 - 1.0) * (2 * math.pi / (n - 1))
    del x0, x1
    r = torch.full((N,), (400 + 6378) * 1000.0, dtype=torch.float64, device="cuda")
    o = [torch.empty(N, dtype=torch.float64, device="cuda") for _ in range(3)]
    torch.cuda.synchronize()
    k1_med, k1_min = timed(lambda: eng.igrf12_batch(2019.0, r, lat, lon, out=o), eng, a.reps, a.warmup)

    name = torch.cuda.get_device_name(0)
    plim, clk = gpu_power_limit(0)
    t = ev_med * 1e-3
    dram = N * (IN_B + OUT_B) / t
    row = {
        "what": "K8 field-map interpolant (igrf_data 1000x1000 map, cubic B-spline)",
        "device": name, "power_limit_W": plim, "max_sm_clock_MHz": clk,
        "library": os.path.basename(tb.lib_path()),
        "n": n, "points": N, "reps": a.reps, "seed": a.seed,
        "prefilter_ms_median": round(pre_med, 4), "prefilter_ms_min": round(pre_min, 4),
        "eval_ms_median": round(ev_med, 3), "eval_ms_min": round(ev_min, 3),
        "eval_per_s": N / t,
        "k1_igrf12_ms_median": round(k1_med, 3), "k1_igrf12_per_s": N / (k1_med * 1e-3),
        "eval_speedup_vs_k1": k1_med / ev_med,
        "bytes_per_point_algorithmic": TAP_B + IN_B + OUT_B,
        "achieved_B_per_s_algorithmic": N * (TAP_B + IN_B + OUT_B) / t,
        "achieved_B_per_s_dram_part": dram,
        "dram_part_share_of_7p7TBs": dram / (HBM_TBS * 1e12),
        "tap_B_per_s_from_L2": N * TAP_B / t,
        "padded_tap_B_per_s_from_L2": N * TAP_B_PADDED / t,
    }
    row["bound"] = ("DRAM (indices + outputs)" if row["dram_part_share_of_7p7TBs"] >= 0.5 else
                    "L2 / load path (tap gathers): the DRAM part is under half of HBM bandwidth")
    line = json.dumps(row)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
