"""CPU: the disturbance ensemble's draws and replay (rules RE2 of DESIGN.md section 4, K4) -- the numpy restatement of its
counter layout against the Random123 known answers and the K4 source compiled for the host, one realisation's host
replay against the oracle fed the same draws, the layout of ts_replay_ensemble_opts across C, ctypes and Julia, and the
SASS of the ensemble kernel K4e."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import replay_ensemble_ref as RE
import slew_setup as S
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REALS = (0, 1, 7, 2**30 - 1)
KEYS = [(0, 0, 0, 0), (4242, 100, 2043, 3), (2**63 + 5, 4095, 17, 1), (12345678901234, 7, 99, 2)]


def test_philox_restatement_known_answers():
    kats = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
            ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
            ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, exp in kats:
        got = RE.philox4x32_10(*ctr, *key)
        assert tuple(int(v) for v in got) == exp


def test_stage_draws_match_the_kernel_source():
    """tvlqr_noise with realisation r, host-compiled, equals the restatement for r in {0, 1, 7, 2^30 - 1}; at r = 0 it is
    the single replay's stream (hs_tvlqr_noise)."""
    L = RE.hostsim_ensemble()
    hs = S.hostsim()
    a, b = np.zeros(9), np.zeros(9)
    for seed, tr, st, sg in KEYS:
        for r in REALS:
            L.hse_tvlqr_noise(seed, tr, st, sg, r, orc.P(a))
            ref = RE.tvlqr_noise(seed, tr, st, sg, r)
            assert np.allclose(a, ref, rtol=1e-14, atol=0), (seed, tr, st, sg, r)
        L.hse_tvlqr_noise(seed, tr, st, sg, 0, orc.P(a))
        hs.hs_tvlqr_noise(seed, tr, st, sg, orc.P(b))
        assert a.tobytes() == b.tobytes()
    # realisations are distinct streams
    L.hse_tvlqr_noise(9, 3, 5, 1, 1, orc.P(a))
    L.hse_tvlqr_noise(9, 3, 5, 1, 2, orc.P(b))
    assert not np.any(a == b)


def test_initial_draw_matches_the_kernel_source():
    L = RE.hostsim_ensemble()
    q = np.zeros(3)
    scale = (np.pi / 180) ** 2
    for seed, tr, _, _ in KEYS:
        for r in REALS[1:]:
            L.hse_initial_qnoise(seed, tr, r, scale, orc.P(q))
            assert np.allclose(q, RE.initial_qnoise(seed, tr, r, scale), rtol=1e-14, atol=0)
    # x0_lqr: the rotation of ts_monte_carlo_run; a zero row leaves x0's attitude, and the clock is 0
    x0 = np.array([1e-3, -2e-3, 5e-4, 0.5, 0.5, 0.5, 0.5, 3.0])
    xl = np.zeros(8)
    L.hse_x0_lqr(orc.P(x0), orc.P(q), orc.P(xl))
    assert np.allclose(xl, RE.x0_lqr(x0, q), rtol=0, atol=1e-15) and xl[7] == 0
    L.hse_x0_lqr(orc.P(x0), orc.P(np.zeros(3)), orc.P(xl))
    assert np.array_equal(xl[:7], x0[:7]) and xl[7] == 0


@pytest.fixture(scope="module")
def solved():
    s = S.build_slew([0, 6578, 96, 0, 0, 90], S.J_1P, S.quat_axis_angle([1, 0, 1], 5.0), np.array([1.0, 0, 0, 0]), t_final=60.0)
    Xs, Us, Ks, out = S.oracle_solve([s])
    return s, Xs[0], Us[0]


@pytest.mark.parametrize("r", [1, 7, 2**30 - 1])
def test_host_replay_of_a_realisation_matches_the_oracle(solved, r):
    """One realisation replayed by the host build of the K4 source (draws inline, TvlqrIn::real = r) against the oracle
    fed the same draws as an explicit noise array (mode 1) from the restatement: states to 1e-10, the same slew time."""
    s, X, U = solved
    seed, stream = 2026, 5
    o, g = S.tvlqr_opts_pair(noise_mode=1, seed=seed)
    g.noise_mode = 2
    qn = RE.initial_qnoise(seed, stream, r, (np.pi / 180) ** 2)
    x0 = RE.x0_lqr(s.x0, qn)
    nz = RE.noise_array(seed, stream, s.N, r)
    a = S.oracle_tvlqr(s, X, U, x0, o, trial=stream, noise=nz)
    L = RE.hostsim_ensemble()
    N = s.N
    Xs, K, xl, slew = np.zeros((N, 8)), np.zeros((N, 18)), np.zeros(8), np.zeros(1)
    Up = np.zeros((N, 3))
    Up[:N - 1] = U
    B = np.ascontiguousarray(s.B)
    ns = L.hse_tvlqr_real(N, orc.P(orc.f64(X)), orc.P(Up), orc.P(orc.f64(x0)), orc.P(orc.f64(s.J.reshape(-1))), orc.P(B), B.shape[0],
                          s.index_scale, s.clock_rate, s.t_final, orc.P(orc.f64(s.xf[3:7])), stream, r, C.addressof(g), orc.P(Xs),
                          orc.P(K), orc.P(xl), orc.P(slew))
    assert ns == a[4]
    assert np.max(np.abs(Xs[:ns] - a[0])) < 1e-10
    assert np.array_equal(xl, Xs[ns - 1])
    assert slew[0] == a[5]


def test_opts_struct_layout():
    """sizeof(ts_replay_ensemble_opts) is the same in C (the header, compiled), ctypes and the Julia mirror."""
    from tortoisesat.jl_b200 import host
    hdr = os.path.join(ROOT, "include")
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"tortoise_b200.h\"\nint main(void){printf(\"%zu %zu %zu\", " \
          "sizeof(ts_replay_ensemble_opts), offsetof(ts_replay_ensemble_opts, r_first), offsetof(ts_replay_ensemble_opts, q_noise_scale));return 0;}\n"
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "layout.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "layout")
        subprocess.run(["/usr/bin/gcc", "-I", hdr, "-o", exe, c], check=True, capture_output=True)
        size, o1, o2 = (int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split())
    assert (size, o1, o2) == (C.sizeof(host.ReplayEnsembleOpts), host.ReplayEnsembleOpts.r_first.offset,
                              host.ReplayEnsembleOpts.q_noise_scale.offset) == (24, 8, 16)
    jl = open(os.path.join(ROOT, "julia", "TortoiseB200.jl")).read()
    m = re.search(r"struct ReplayEnsembleOpts\s*#[^\n]*\n(.*?)\nend", jl, re.S)
    fields = re.findall(r"(\w+)::(\w+)", m.group(1))
    assert fields == [("n_real", "Int64"), ("r_first", "Int64"), ("q_noise_scale", "Float64")]
    assert [f for f, _ in host.ReplayEnsembleOpts._fields_] == [f for f, _ in fields]


def test_k4e_step_loop_has_no_local_memory_traffic():
    """Static check of the shipped library (cuobjdump, no GPU): the ensemble kernel's step loop and its stage-record loop
    -- every loop of the kernel with 200 or more FP64 instructions -- contain no LDL / STL."""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import __graft_entry__ as gr
    gr.build()
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sass_hot_loops as shl
    sass = subprocess.run([exe, "-sass", shl.LIB], capture_output=True, text=True, check=True).stdout
    fns = {n: ins for n, ins in shl.functions(sass).items() if "k4e_ensemble_replay_kernel" in n}
    assert len(fns) == 1
    ins = next(iter(fns.values()))
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
            assert ops.count("LDL") == 0 and ops.count("STL") == 0, hex(a)
    assert hot >= 2
