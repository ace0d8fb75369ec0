"""CPU: the dispersion ensemble's truth-model draws and replay (rules DE2-DE4 of DESIGN.md section 4, K4) -- the numpy
restatement of the draws against the K4 source compiled for the host, one dispersed realisation's host replay against
the oracle's truth-model replay fed the same parameters and stage draws, the null dispersion against the disturbance
ensemble's host replay, the layout of ts_dispersion_opts across C, ctypes and Julia, and the SASS of the kernel K4d."""
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
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REALS = (0, 1, 7, 2**30 - 1)
KEYS = [(0, 0), (4242, 100), (2**63 + 5, 4095), (12345678901234, 7)]
SIGMAS = [(0.1, 0.05, 0.05, np.radians(3.0)), (1.0, 1.0, 1.0, np.pi), (0.2, 0.0, 0.0, 0.0), (0.0, 0.0, 0.0, np.radians(5.0))]
GROUPS = {"inertia": (0.2, 0, 0, 0), "torquer": (0, 0.1, 0, 0), "field_scale": (0, 0, 0.05, 0), "field_angle": (0, 0, 0, np.radians(5.0)),
          "all": (0.2, 0.1, 0.05, np.radians(5.0))}
NOMINAL = np.array([1.0] * 7 + [0.0] * 3)


def test_draws_match_the_kernel_source():
    """dispersion_params, host-compiled, equals the restatement to 1e-14 for the keys and realisations of the disturbance
    ensemble's tests (r up to 2^30 - 1)."""
    for seed, stream in KEYS:
        for r in REALS:
            for sg in SIGMAS:
                got = DR.host_params(seed, stream, r, sg)
                ref = DR.dispersion_params(seed, stream, r, sg)
                assert np.allclose(got, ref, rtol=1e-14, atol=1e-14), (seed, stream, r, sg, got, ref)


def test_nominal_realisation_and_groups():
    """r = 0 and every group with sigma 0 are exactly nominal; changing one sigma leaves the other groups' parameters
    unchanged bit for bit (fixed normals per group); realisations r >= 1 are distinct draws."""
    groups = [slice(0, 3), slice(3, 6), slice(6, 7), slice(7, 10)]
    for seed, stream in KEYS:
        assert np.array_equal(DR.host_params(seed, stream, 0, SIGMAS[1]), NOMINAL)
        for r in REALS[1:]:
            assert np.array_equal(DR.host_params(seed, stream, r, (0, 0, 0, 0)), NOMINAL)
            base = DR.host_params(seed, stream, r, (0.1, 0.05, 0.05, 0.05))
            for gi, gs in enumerate(groups):
                sg = [0.1, 0.05, 0.05, 0.05]
                sg[gi] = 0.0
                p0 = DR.host_params(seed, stream, r, sg)
                assert np.array_equal(p0[gs], NOMINAL[gs])
                sg[gi] = 0.3
                p1 = DR.host_params(seed, stream, r, sg)
                assert not np.array_equal(p1[gs], base[gs])
                for gj, gt in enumerate(groups):
                    if gj != gi:
                        assert p0[gt].tobytes() == base[gt].tobytes() and p1[gt].tobytes() == base[gt].tobytes(), (gi, gj)
    assert not np.array_equal(DR.host_params(9, 3, 1, SIGMAS[0]), DR.host_params(9, 3, 2, SIGMAS[0]))


@pytest.fixture(scope="module")
def solved():
    s = S.build_slew([0, 6578, 96, 0, 0, 90], S.J_1P, S.quat_axis_angle([1, 0, 1], 5.0), np.array([1.0, 0, 0, 0]), t_final=60.0)
    Xs, Us, Ks, out = S.oracle_solve([s])
    return s, Xs[0], Us[0]


def _product_opts(seed):
    from tortoisesat.jl_b200 import host
    g = host.TvlqrOpts()
    g.dt, g.t0, g.dt_squared, g.noise_mode, g.seed = 0.2, 0.0, 1, 2, seed
    for i in range(6):
        g.Qd[i], g.Qfd[i] = 10.0, 1000.0
    for i in range(3):
        g.Rd[i] = 7.5e3
    g.w_limit, g.ang_limit, g.literal_postproc = 0.05, 0.08727, 0
    return g


@pytest.mark.parametrize("group", list(GROUPS))
def test_host_dispersed_replay_matches_the_oracle(solved, group):
    """One dispersed realisation replayed by the host build of the kernel source against the oracle's truth-model
    replay fed the same parameters and the restatement's stage draws: states to 1e-10, the same slew time; the
    dispersion moves the final state away from the undispersed realisation's."""
    s, X, U = solved
    seed, stream = 2026, 5
    o = S.oracle_tvlqr_opts(noise_mode=1, seed=seed)
    g = _product_opts(seed)
    for r in (1, 2**30 - 1):
        prm = DR.host_params(seed, stream, r, GROUPS[group])
        x0 = RE.x0_lqr(s.x0, RE.initial_qnoise(seed, stream, r, (np.pi / 180) ** 2))
        nz = RE.noise_array(seed, stream, s.N, r)
        a, ns_a, slew_a = DR.oracle_truth(s, X, U, x0, o, prm, nz)
        h, ns, slew, xl = DR.host_disp_real(s, X, U, x0, g, stream, r, prm)
        assert ns == ns_a
        assert np.max(np.abs(h - a)) < 1e-10, (group, r, np.max(np.abs(h - a)))
        assert slew == slew_a, (group, r, slew, slew_a)
        assert np.array_equal(xl, h[ns - 1])
        h0, _, _, xl0 = DR.host_disp_real(s, X, U, x0, g, stream, r, NOMINAL)
        assert np.max(np.abs(xl - xl0)) > 1e-9, group


def test_null_dispersion_is_the_disturbance_ensemble(solved):
    """With nominal parameters the host dispersed replay is bit-identical to the disturbance ensemble's (hse_tvlqr_real),
    and the oracle's truth-model replay to the oracle's replay."""
    s, X, U = solved
    seed, stream = 2026, 5
    g = _product_opts(seed)
    o = S.oracle_tvlqr_opts(noise_mode=1, seed=seed)
    L = RE.hostsim_ensemble()
    N = s.N
    Up = np.zeros((N, 3))
    Up[:N - 1] = U
    B = np.ascontiguousarray(s.B)
    for r in (0, 1, 7):
        x0 = RE.x0_lqr(s.x0, RE.initial_qnoise(seed, stream, r, (np.pi / 180) ** 2)) if r else s.x0 * np.array([1] * 7 + [0])
        h, ns, slew, xl = DR.host_disp_real(s, X, U, x0, g, stream, r, NOMINAL)
        Xs, K, xe, se = np.zeros((N, 8)), np.zeros((N, 18)), np.zeros(8), np.zeros(1)
        ne = L.hse_tvlqr_real(N, orc.P(orc.f64(X)), orc.P(Up), orc.P(orc.f64(x0)), orc.P(orc.f64(s.J.reshape(-1))), orc.P(B), B.shape[0],
                              s.index_scale, s.clock_rate, s.t_final, orc.P(orc.f64(s.xf[3:7])), stream, r, C.addressof(g), orc.P(Xs),
                              orc.P(K), orc.P(xe), orc.P(se))
        assert ne == ns and h.tobytes() == Xs[:ns].tobytes() and xl.tobytes() == xe.tobytes() and slew == se[0]
        nz = RE.noise_array(seed, stream, N, r)
        a, ns_a, slew_a = DR.oracle_truth(s, X, U, x0, o, NOMINAL, nz)
        b = S.oracle_tvlqr(s, X, U, x0, o, trial=stream, noise=nz)
        assert ns_a == b[4] and a.tobytes() == b[0].tobytes() and slew_a == b[5]


def test_opts_struct_layout():
    """sizeof and offsets of ts_dispersion_opts are the same in C (the header, compiled), ctypes and the Julia mirror:
    four doubles, 32 bytes, no padding."""
    from tortoisesat.jl_b200 import host
    names = ("sigma_inertia", "sigma_torquer", "sigma_field_scale", "sigma_field_angle")
    hdr = os.path.join(ROOT, "include")
    src = "#include <stdio.h>\n#include <stddef.h>\n#include \"tortoise_b200.h\"\nint main(void){printf(\"%zu" + " %zu" * 4 + "\", " \
          "sizeof(ts_dispersion_opts), " + ", ".join("offsetof(ts_dispersion_opts, %s)" % n for n in names) + ");return 0;}\n"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "layout.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "layout")
        subprocess.run(["/usr/bin/gcc", "-I", hdr, "-o", exe, c], check=True, capture_output=True)
        got = tuple(int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split())
    assert got == (C.sizeof(host.DispersionOpts),) + tuple(getattr(host.DispersionOpts, n).offset for n in names) == (32, 0, 8, 16, 24)
    jl = open(os.path.join(ROOT, "julia", "TortoiseB200.jl")).read()
    m = re.search(r"struct DispersionOpts\s*#[^\n]*\n(.*?)\nend", jl, re.S)
    fields = re.findall(r"(\w+)::(\w+)", m.group(1))
    assert fields == [(n, "Float64") for n in names]
    assert [f for f, _ in host.DispersionOpts._fields_] == list(names)


def test_k4d_loops_have_no_local_memory_traffic():
    """Static check of the shipped library (cuobjdump, no GPU): the dispersion kernel's step loop and its stage-record
    loop -- every loop of the kernel with 200 or more FP64 instructions -- contain no LDL / STL."""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    import __graft_entry__ as gr
    gr.build()
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import sass_hot_loops as shl
    sass = subprocess.run([exe, "-sass", shl.LIB], capture_output=True, text=True, check=True).stdout
    fns = {n: ins for n, ins in shl.functions(sass).items() if "k4d_dispersion_replay_kernel" in n}
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
