"""CPU: continuation of the AL-iLQR solve from an exported state (rules CS1-CS4, DESIGN.md section 4, K3).

The oracle with the state in and out (tests/alilqr_state_ref) must give, bit for bit, "solve to M1, continue to M2" ==
"solve to M2" whenever the tolerance pairs agree (CS4); the kernel source's export / import pair does the same under the
lane emulator, across team widths (export from an 8-lane team, import into a whole warp)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import alilqr_state as AS
import slew_setup as S
from oracle import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("status", "outer_iters", "inner_iters", "ls_rollouts", "N", "J", "c_max")


def slews():
    """the slews of test_hostsim: under the default goal mask two converge after 10-11 outer iterations and two use all
    20; under the literal goal mask (0xFF) all four blow up at outer iteration 10"""
    mk = lambda angle, tfin: S.build_slew([0, 6578, 96, 0, 0, 90], S.J_1P, S.quat_axis_angle([1, 0, 1], angle), np.array([1.0, 0, 0, 0]),
                                          t_final=tfin)
    return [mk(5.0, 60.0), mk(20.0, 30.0), mk(8.0, 40.0), mk(2.0, 20.0)]


_SLEWS = None


def get_slews():
    global _SLEWS
    if _SLEWS is None:
        _SLEWS = slews()
    return _SLEWS


def opts_for(variant, max_outer, mask=0x7F):
    o = orc.default_ilqr_opts()
    o.max_outer = max_outer
    o.goal_mask = mask
    o.cost_tol_intermediate = o.cost_tol   # CS4: equal tolerance pairs
    if variant != "default":
        setattr(o, variant, 1)
    if variant == "a4_no_intermediate":
        o.cost_tol_intermediate = 1e-3     # equal schedules through A4, with the default (different) pairs
    return o


def assert_same(a, b):
    Xa, Ua, Ka, oa, sa, la = a
    Xb, Ub, Kb, ob, sb, lb = b
    assert np.array_equal(Xa, Xb) and np.array_equal(Ua, Ub) and np.array_equal(Ka, Kb)
    for f in FIELDS:
        assert np.array_equal(oa[f], ob[f]), f
    assert sa.tobytes() == sb.tobytes()
    assert np.array_equal(la, lb)


@pytest.mark.parametrize("variant", ["default", "a6_penalty_conditional", "a7_carry_cost", "a5_dual_active_only", "quat_error",
                                     "a4_no_intermediate"])
def test_fresh_solve_with_state_out_is_the_oracle(variant):
    """Without a state in, the restatement with the state in and out computes what the oracle's alilqr_solve computes,
    bit for bit, under every option the continuation tests use."""
    o = orc.default_ilqr_opts()
    if variant != "default":
        setattr(o, variant, 1)
    o.max_outer = 12
    sl = get_slews() if variant != "quat_error" else get_slews()[:2]
    Xs, Us, Ks, out = S.oracle_solve(sl, o, nthreads=4)
    X, U, K, oc, st, lam = AS.oracle_state_solve(sl, o)
    offs = AS.pack(sl)["offs"]
    for t in range(len(sl)):
        assert np.array_equal(X[offs[t]:offs[t + 1]], Xs[t]) and np.array_equal(U[offs[t]:offs[t + 1] - 1], Us[t])
        assert np.array_equal(K[offs[t]:offs[t + 1] - 1], Ks[t])
        for f in FIELDS:
            assert oc[t][f] == out[t][f], f
        assert st[t]["J"] == oc[t]["J"] and st[t]["c_max"] == oc[t]["c_max"] and st[t]["outer_iters"] == oc[t]["outer_iters"]
        assert np.all(lam[offs[t + 1] - 1] == 0.0) and np.all(lam >= 0.0)
    assert 1 in oc["status"]


@pytest.mark.parametrize("variant", ["default", "a6_penalty_conditional", "a7_carry_cost", "a5_dual_active_only", "quat_error",
                                     "a4_no_intermediate"])
def test_oracle_continuation_equals_direct_solve(variant):
    """CS1-CS4: solve to M1, continue to M2 == solve to M2, bit for bit (X, U, K, every outcome field, state, lam), on a
    batch where one slew converges before M1, one runs out of outer iterations, one blows up and one converges fast."""
    sl = get_slews() if variant != "quat_error" else get_slews()[:2]
    for M1, M2 in ((7, 12), (12, 20)):
        first = AS.oracle_state_solve(sl, opts_for(variant, M1))
        assert 1 in first[3]["status"]
        cont = AS.oracle_state_solve(sl, opts_for(variant, M2), state=first[4], lam=first[5], X=first[0], U=first[1], K=first[2])
        direct = AS.oracle_state_solve(sl, opts_for(variant, M2))
        assert_same(cont, direct)
    assert direct[3]["outer_iters"][1] == 20   # the slew that runs all 20 outer iterations
    assert 0 in first[3]["status"]               # and one that converged before M1 and passed through


def test_oracle_pass_through():
    """CS2: continuing to max_outer = M1 changes nothing, and converged / blown-up trials pass through in any case."""
    sl = get_slews()
    o = opts_for("default", 12)
    first = AS.oracle_state_solve(sl, o)
    K0 = np.random.default_rng(1).normal(size=first[2].shape)
    same = AS.oracle_state_solve(sl, o, state=first[4], lam=first[5], X=first[0], U=first[1], K=K0)
    assert np.array_equal(same[0], first[0]) and np.array_equal(same[1], first[1]) and np.array_equal(same[2], K0)
    for f in FIELDS:
        assert np.array_equal(same[3][f], first[3][f]), f
    assert same[4].tobytes() == first[4].tobytes() and np.array_equal(same[5], first[5])
    more = AS.oracle_state_solve(sl, opts_for("default", 16), state=first[4], lam=first[5], X=first[0], U=first[1], K=K0)
    offs = AS.pack(sl)["offs"]
    for t in range(len(sl)):
        if first[3]["status"][t] != 1:
            r = slice(offs[t], offs[t + 1])
            assert np.array_equal(more[0][r], first[0][r]) and np.array_equal(more[2][r], K0[r])
            assert more[4][t].tobytes() == first[4][t].tobytes()
        else:
            assert more[3]["outer_iters"][t] > 12
    # blown-up trials (literal goal mask): nothing continues
    blown = AS.oracle_state_solve(sl, opts_for("default", 12, 0xFF))
    assert list(blown[3]["status"]) == [2] * len(sl)
    again = AS.oracle_state_solve(sl, opts_for("default", 20, 0xFF), state=blown[4], lam=blown[5], X=blown[0], U=blown[1], K=K0)
    assert np.array_equal(again[0], blown[0]) and np.array_equal(again[2], K0) and again[4].tobytes() == blown[4].tobytes()


@pytest.mark.parametrize("variant", ["default", "a7_carry_cost", "quat_error"])
def test_lane_emulator_continuation_across_widths(variant):
    """The kernel source's export (8-lane team) and import (whole-warp team): continuation == direct solve, bit for bit,
    and the same iteration path as the oracle's continuation."""
    s = get_slews()[1]
    M1, M2 = 4, 9
    X1, U1, K1, o1, s1, l1 = AS.hostsim_state_solve(s, opts_for(variant, M1), width=8)
    assert o1["status"] == 1 and s1["outer_iters"] == M1
    cont = AS.hostsim_state_solve(s, opts_for(variant, M2), width=32, state=s1, lam=l1, X=X1, U=U1)
    direct = AS.hostsim_state_solve(s, opts_for(variant, M2), width=8)
    assert np.array_equal(cont[0], direct[0]) and np.array_equal(cont[1], direct[1]) and np.array_equal(cont[2], direct[2])
    for f in FIELDS:
        assert cont[3][f] == direct[3][f], f
    assert cont[4].tobytes() == direct[4].tobytes() and np.array_equal(cont[5], direct[5])
    ref = AS.oracle_state_solve([s], opts_for(variant, M2))
    for f in ("status", "outer_iters", "inner_iters", "ls_rollouts"):
        assert cont[3][f] == ref[3][0][f], f
    assert cont[4]["mu"] == ref[4][0]["mu"]
    assert np.max(np.abs(cont[5] - ref[5])) <= 1e-8 * max(1.0, np.max(np.abs(ref[5])))
    # exported from the first call: the oracle's state after M1 outer iterations
    ref1 = AS.oracle_state_solve([s], opts_for(variant, M1))
    assert s1["mu"] == ref1[4][0]["mu"] and s1["outer_iters"] == ref1[4][0]["outer_iters"]
    assert np.allclose(s1["lam_goal"], ref1[4][0]["lam_goal"], rtol=1e-8, atol=1e-12)


def test_al_state_layout_and_export(tmp_path):
    """sizeof(ts_al_state) is 104 in gcc, in the ctypes / numpy mirrors and in the parsed Julia struct; the library
    exports the new entry."""
    from tortoisesat.jl_b200 import host
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "tortoise_b200.h"\nint main(void){printf("%zu\\n", sizeof(ts_al_state));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    assert int(subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout) == 104
    assert ctypes.sizeof(host.AlState) == 104 and host.AL_STATE_DTYPE.itemsize == 104 and AS.AL_STATE_DTYPE == host.AL_STATE_DTYPE
    jl = open(os.path.join(ROOT, "julia", "TortoiseB200.jl")).read()
    body = re.search(r"^struct AlState\b.*?\n(.*?)^end", jl, re.S | re.M).group(1)
    size = {"Float64": 8, "Int32": 4, "NTuple{8,Float64}": 64}
    assert sum(size[t] for t in re.findall(r"::\s*([A-Za-z0-9_{},]+)", re.sub(r"#.*", "", body))) == 104
    import __graft_entry__ as g
    g.build()
    import tortoisesat.jl_b200 as tb
    lib = ctypes.CDLL(tb.lib_path())
    assert hasattr(lib, "ts_alilqr_solve_state_batch")
    assert lib.ts_version() >= 102
