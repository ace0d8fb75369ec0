"""Continuation of max-outer trials (ts_alilqr_solve_state_batch) on bench.py's fixed-orbit ensemble -> one JSON line.

The solver inputs of bench.make_trials("mc_fixed_orbit", 4096, 0) are built through the stand-alone K2 entries
(scoping table, gramian cutoff, fine table) and ts_slew_weights_batch, as ts_monte_carlo_run builds them.  Then:
  0. how many outcome records differ from ts_monte_carlo_run (run_tvlqr = 0) on the same ensemble (expected 0);
  1. solve with max_outer = 20, exporting the state;
  2. continue the trials that ended at TS_ST_MAX_OUTER to max_outer = 30;
  3. solve directly with max_outer = 30.
For each step: K3 device time (ts_last_kernel_ms), the status histogram, the trials converged.  The default tolerance
pairs differ (cost_tol_intermediate 1e-3 vs cost_tol 1e-4), so outer iteration 20 runs with the final tolerances in
step 1 and with the intermediate ones in step 3 (CS4): the line also counts the continued trials whose status differs
from the direct solve.  Usage: python tools/continue_bench.py [--trials 4096] [--out FILE]"""
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
FIELDS = ("status", "outer_iters", "inner_iters", "ls_rollouts", "N", "J", "c_max")


def hist(out):
    h = np.bincount(out["status"], minlength=6)[:6]
    return {STATUS[k]: int(h[k]) for k in range(6)}


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as ex:  # pragma: no cover
        return "unknown (%s)" % ex


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trials", type=int, default=4096)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    n = a.trials
    eng = tb.Engine(0)
    tr = B.make_trials("mc_fixed_orbit", 4096, 0)
    for k in ("x0", "xf", "Jm", "qn"):
        tr[k] = tr[k][:n]
    cfg = B.mc_config(host, tr, n)
    cfg.run_tvlqr = 0
    f = tr["fo"][0]
    # K2: the scoping table over [t0, tf] with N_scope knots, its gramian cutoff, then the fine table over [t0, t_final]
    t0, tf, Ns, dt = float(cfg.t0), float(cfg.tf), int(cfg.N_scope), float(cfg.dt)
    fo = np.zeros(1, dtype=host.FIELD_OPTS_DTYPE)
    fo[0] = (f[0], f[1], f[2], f[3], t0, tf, Ns)
    Bs, offs_s = eng.magnetic_simulation_batch(tr["kep"], fo)
    idx = eng.condition_cutoff_batch(Bs, offs_s[:-1], [offs_s[1]], [(tf - t0) / Ns], [tr["cutoff"]])
    t_final = int(idx[0]) * (tf - t0) / Ns
    N = int(np.floor((t_final - t0) / dt))
    fo[0] = (f[0], f[1], f[2], f[3], t0, t_final, N)
    Bt, _ = eng.magnetic_simulation_batch(tr["kep"], fo)
    Qd, Qfd, Rd = eng.slew_weights_batch(tr["x0"], tr["xf"], tr["Jm"], [t_final] * n, t0=t0, dt=dt, alpha=float(cfg.alpha),
                                         beta=float(cfg.beta))
    args = dict(N_i=[N] * n, x0=tr["x0"], xf=tr["xf"], Jmat=tr["Jm"], Qd=Qd, Qfd=Qfd, Rd=Rd, B_eci=Bt, B_offs=[0] * n,
                B_rows=[Bt.shape[0]] * n, index_scale=[float(N)] * n, clock_rate=[1.0 / (tf - t0)] * n, dt=dt, want_K=False)
    fo_mc = np.zeros(1, dtype=host.FIELD_OPTS_DTYPE)
    fo_mc[0] = f
    mc, _ = eng.monte_carlo_run(cfg, tr["kep"], fo_mc, tr["x0"], tr["xf"], tr["Jm"], q_noise0=tr["qn"])
    o20 = host.default_ilqr_opts()
    o30 = host.default_ilqr_opts()
    o30.max_outer = 30
    eng.alilqr_solve_state_batch(**args, opts=o20)   # warm-up (module load, scratch allocation)
    X, U, _, out20, offs, st20, lam20 = eng.alilqr_solve_state_batch(**args, opts=o20)
    ms20 = eng.last_kernel_ms()
    n_mismatch = int(sum(any(out20[t][k] != mc[t][k] for k in FIELDS) for t in range(n)))
    cont_mask = out20["status"] == 1
    _, _, _, outc, _, stc, _ = eng.alilqr_solve_state_batch(**args, opts=o30, state=st20, lam=lam20, X=X, U=U)
    msc = eng.last_kernel_ms()
    split_c = eng.k3_last_split()
    _, _, _, out30, _, _, _ = eng.alilqr_solve_state_batch(**args, opts=o30)
    ms30 = eng.last_kernel_ms()
    sm, name = eng.device_info()
    line = {
        "tool": "continue_bench", "device": name, "power_limit": power_limit(), "workload": "mc_fixed_orbit rank 0",
        "trials": n, "N": N, "t_final": t_final,
        "mismatch_vs_monte_carlo_run": n_mismatch,
        "solve20": {"k3_ms": ms20, "status": hist(out20), "converged": int((out20["status"] == 0).sum())},
        "continue20to30": {"k3_ms": msc, "continued": int(cont_mask.sum()), "status_of_continued": hist(outc[cont_mask]),
                           "converged_of_continued": int((outc["status"][cont_mask] == 0).sum()), "status_all": hist(outc),
                           "k3_split_ms": [split_c[0], split_c[1]], "parked": split_c[2]},
        "solve30": {"k3_ms": ms30, "status": hist(out30), "converged": int((out30["status"] == 0).sum())},
        "continue_vs_solve30": {
            "status_differs_on_continued": int((outc["status"][cont_mask] != out30["status"][cont_mask]).sum()),
            "outer_differs_on_continued": int((outc["outer_iters"][cont_mask] != out30["outer_iters"][cont_mask]).sum()),
            "passed_through_identical": bool(all(outc[t][k] == out20[t][k] for t in np.nonzero(~cont_mask)[0] for k in FIELDS)),
            "note": "CS4: default tolerance pairs differ, so outer iteration 20 used the final tolerances in solve20"},
        "time_fraction_continue_over_solve30": msc / ms30 if ms30 > 0 else None,
    }
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(s + "\n")
    eng.close()


if __name__ == "__main__":
    main()
