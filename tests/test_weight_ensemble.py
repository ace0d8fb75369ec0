"""CPU: the weight-sweep ensemble's replay (rules WE2-WE4 of DESIGN.md section 4, K4) -- the host build of the kernel
source with the torquer-limit switch against the oracle's limited truth-model replay under the same weighting, draws
and parameters; with the switch off and the run's weighting, against the dispersion ensemble's host replay bit for bit;
the layout of ts_tvlqr_weights across C, ctypes and Julia; and the SASS of the K4w kernels."""
import ctypes as C
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import dispersion_ref as DR
import replay_ensemble_ref as RE
import slew_setup as S
import weight_ref as WR
from test_dispersion_ensemble import GROUPS, _product_opts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QS = (np.pi / 180) ** 2
SEED, STREAM = 2026, 5


@pytest.fixture(scope="module")
def solved():
    s = S.build_slew([0, 6578, 96, 0, 0, 90], S.J_1P, S.quat_axis_angle([1, 0, 1], 5.0), np.array([1.0, 0, 0, 0]), t_final=60.0)
    Xs, Us, Ks, out = S.oracle_solve([s])
    return s, Xs[0], Us[0]


def _sets(g):
    w = WR.run_weights(g)
    return {"run": w, "R/100": WR.scaled(w, r=0.01), "Qx10": WR.scaled(w, q=10.0), "Qf=Q": WR.scaled(w, qf_equals_q=True)}


@pytest.mark.parametrize("u_limit", [0.0, 1.0, 0.05])
def test_host_weighted_replay_matches_the_oracle(solved, u_limit):
    """Each weighting, every truth-model group on, r = 1 and 2^30 - 1: the host replay of the kernel source equals the
    oracle's limited truth-model replay to 1e-10 with the same slew time.  The weightings move the final state, and the
    limit binds (a limited replay differs from the unlimited one) in at least one case."""
    s, X, U = solved
    o = S.oracle_tvlqr_opts(noise_mode=1, seed=SEED)
    g = _product_opts(SEED)
    bound = 0
    for name, w in _sets(g).items():
        for r in (1, 2**30 - 1):
            prm = DR.host_params(SEED, STREAM, r, GROUPS["all"])
            x0 = RE.x0_lqr(s.x0, RE.initial_qnoise(SEED, STREAM, r, QS))
            nz = RE.noise_array(SEED, STREAM, s.N, r)
            a, ns_a, slew_a = WR.oracle_truth_weighted(s, X, U, x0, o, prm, nz, w, u_limit)
            h, ns, slew, xl = WR.host_weight_real(s, X, U, x0, g, STREAM, r, prm, w, u_limit)
            assert ns == ns_a
            assert np.max(np.abs(h - a)) < 1e-10, (name, r, u_limit, np.max(np.abs(h - a)))
            assert slew == slew_a, (name, r, u_limit, slew, slew_a)
            assert np.array_equal(xl, h[ns - 1])
            if u_limit > 0:
                _, _, _, xf = WR.host_weight_real(s, X, U, x0, g, STREAM, r, prm, w, 0.0)
                bound += int(np.max(np.abs(xf - xl)) > 1e-12)
            if name != "run":
                _, _, _, xr = WR.host_weight_real(s, X, U, x0, g, STREAM, r, prm, WR.run_weights(g), u_limit)
                assert np.max(np.abs(xr - xl)) > 1e-12, (name, r)
    if u_limit > 0:
        assert bound >= 1


def test_unlimited_run_weighting_is_the_dispersion_replay(solved):
    """Switch off and the run's weighting: the host replay equals hsd_tvlqr_disp_real (the dispersion ensemble's) bit
    for bit, with every group on and with nominal parameters (WE3)."""
    s, X, U = solved
    g = _product_opts(SEED)
    w = WR.run_weights(g)
    for r in (0, 1, 7, 2**30 - 1):
        x0 = RE.x0_lqr(s.x0, RE.initial_qnoise(SEED, STREAM, r, QS)) if r else s.x0 * np.array([1] * 7 + [0])
        for sg in (GROUPS["all"], (0, 0, 0, 0)):
            prm = DR.host_params(SEED, STREAM, r, sg)
            h, ns, slew, xl = WR.host_weight_real(s, X, U, x0, g, STREAM, r, prm, w, 0.0)
            d, nd, sd, xd = DR.host_disp_real(s, X, U, x0, g, STREAM, r, prm)
            assert ns == nd and h.tobytes() == d.tobytes() and xl.tobytes() == xd.tobytes() and slew == sd


def test_weights_struct_layout():
    """sizeof and offsets of ts_tvlqr_weights are the same in C (the header, compiled), ctypes and the Julia mirror:
    fifteen doubles, 120 bytes, no padding; the (n_sets, 15) array form maps onto it in order."""
    from tortoisesat.jl_b200 import host
    names = ("Qd", "Qfd", "Rd")
    hdr = os.path.join(ROOT, "include")
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"tortoise_b200.h\"\nint main(void){printf(\"%zu" + " %zu" * 3 + "\", " \
          "sizeof(ts_tvlqr_weights), " + ", ".join("offsetof(ts_tvlqr_weights, %s)" % n for n in names) + ");return 0;}\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "layout.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "layout")
        subprocess.run(["/usr/bin/gcc", "-I", hdr, "-o", exe, c], check=True, capture_output=True)
        got = tuple(int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split())
    assert got == (C.sizeof(host.TvlqrWeights),) + tuple(getattr(host.TvlqrWeights, n).offset for n in names) == (120, 0, 48, 96)
    jl = open(os.path.join(ROOT, "julia", "TortoiseB200.jl")).read()
    m = re.search(r"struct TvlqrWeights\s*#[^\n]*\n(.*?)\nend", jl, re.S)
    assert re.findall(r"(\w+)::NTuple\{(\d+), Float64\}", m.group(1)) == [("Qd", "6"), ("Qfd", "6"), ("Rd", "3")]
    a = np.arange(30, dtype=np.float64).reshape(2, 15)
    ws = host.weight_sets(a)
    assert len(ws) == 2 and list(ws[1].Qd) == list(a[1, :6]) and list(ws[1].Qfd) == list(a[1, 6:12]) and list(ws[1].Rd) == list(a[1, 12:])
    assert host.weight_sets(ws) is ws and list(host.weight_sets([ws[1]])[0].Rd) == list(a[1, 12:])
    with pytest.raises(ValueError):
        host.weight_sets(np.zeros((2, 14)))


def test_k4w_loops_have_no_local_memory_traffic():
    """Static check of the shipped library (cuobjdump, no GPU): in both instantiations of the weight-sweep replay kernel
    and in the per-set Riccati kernel, every loop with 200 or more FP64 instructions (the step loop, the stage-record
    loop, the Riccati step) contains no LDL / STL."""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import __graft_entry__ as gr
    gr.build()
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sass_hot_loops as shl
    sass = subprocess.run([exe, "-sass", shl.LIB], capture_output=True, text=True, check=True).stdout
    fns = {n: ins for n, ins in shl.functions(sass).items() if "k4w_weight_replay_kernel" in n or "k4w_riccati_sets_kernel" in n}
    assert len(fns) == 3
    for name, ins in fns.items():
        hot = 0
        for a, t in ins:
            if shl.opcode(t) != "BRA":
                continue
            m = re.search(r"0x([0-9a-f]+)", t)
            if not m or int(m.group(1), 16) > a:
                continue
            ops = [shl.opcode(x) for b, x in ins if int(m.group(1), 16) <= b <= a]
            if sum(ops.count(o) for o in ("DFMA", "DMUL", "DADD")) >= 200:
                hot += 1
                assert ops.count("LDL") == 0 and ops.count("STL") == 0, (name, hex(a))
        assert hot >= (1 if "riccati" in name else 2), name
