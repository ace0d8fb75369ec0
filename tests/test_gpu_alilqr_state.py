"""GPU: ts_alilqr_solve_state_batch -- the exported solver state and continuation from it (CS1-CS4, DESIGN.md
section 4, K3) against the direct solve and the CPU oracle's continuation (tests/alilqr_state_ref)."""
import ctypes as C

import numpy as np
import pytest

import alilqr_state as AS
import slew_setup as S
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
FIELDS = ("status", "outer_iters", "inner_iters", "ls_rollouts", "N", "J", "c_max")


@pytest.fixture(scope="module")
def slews():
    """a ragged batch (N = 100 ... 300): under the default goal mask two slews converge after 10-11 outer iterations,
    two use all 20"""
    mk = lambda angle, tfin: S.build_slew([0, 6578, 96, 0, 0, 90], S.J_1P, S.quat_axis_angle([1, 0, 1], angle), np.array([1.0, 0, 0, 0]),
                                          t_final=tfin)
    return [mk(5.0, 60.0), mk(20.0, 30.0), mk(8.0, 40.0), mk(2.0, 20.0)]


def gpu_opts(max_outer, pair=2, quat=0, suspend=150, equal_tols=True):
    import tortoisesat.jl_b200 as tb
    o = tb.host.default_ilqr_opts()
    o.max_outer, o.k3_pair, o.quat_error, o.k3_suspend_after = max_outer, pair, quat, suspend
    if equal_tols:
        o.cost_tol_intermediate = o.cost_tol   # CS4
    return o


def oracle_opts(max_outer, quat=0):
    o = orc.default_ilqr_opts()
    o.max_outer, o.quat_error = max_outer, quat
    o.cost_tol_intermediate = o.cost_tol
    return o


def args_of(sl):
    p = AS.pack(sl)
    return dict(N_i=p["N_i"], x0=p["x0"], xf=p["xf"], Jmat=p["J"], Qd=p["Qd"], Qfd=p["Qfd"], Rd=p["Rd"], B_eci=p["B_eci"],
                B_offs=p["B_offs"], B_rows=p["B_rows"], index_scale=p["index_scale"], clock_rate=p["clock_rate"], dt=p["dt"])


def raw_call(engine, p, opts, X, U, K, out, dev, state_in=None, lam_in=None, state_out=None, lam_out=None):
    """ts_alilqr_solve_state_batch on host numpy arrays (dev = 0) or torch CUDA tensors (dev = 1) for X, U, K, lam."""
    from tortoisesat.jl_b200.host import _ptr
    P = lambda a: None if a is None else _ptr(a)
    return engine.lib.ts_alilqr_solve_state_batch(
        engine.h, len(p["N_i"]), P(p["N_i"]), P(p["offs"]), P(p["x0"]), P(p["xf"]), P(p["J"]), P(p["Qd"]), P(p["Qfd"]), P(p["Rd"]),
        P(p["B_eci"]) if not dev else _ptr(p["B_dev"]), P(p["B_offs"]), P(p["B_rows"]), P(p["index_scale"]), P(p["clock_rate"]),
        p["dt"], None, C.byref(opts), P(X), P(U), P(K), out.ctypes.data, dev, None if state_in is None else state_in.ctypes.data,
        P(lam_in), None if state_out is None else state_out.ctypes.data, P(lam_out))


@pytest.mark.parametrize("pair,suspend,quat", [(0, 150, 0), (1, 150, 0), (2, 0, 0), (2, 150, 1)])
def test_null_state_is_the_plain_solve(engine, slews, pair, suspend, quat):
    """state_in = NULL: bit-identical to ts_alilqr_solve_batch (hand-over on and off, with K, quat_error = 1), and the
    exported state repeats the outcome record."""
    a = args_of(slews)
    o = gpu_opts(6, pair, quat, suspend, equal_tols=False)
    X0, U0, K0, out0, offs = engine.alilqr_solve_batch(**a, opts=o)
    X1, U1, K1, out1, offs1, st, lam = engine.alilqr_solve_state_batch(**a, opts=o)
    assert np.array_equal(X0, X1) and np.array_equal(U0, U1) and np.array_equal(K0, K1) and out0.tobytes() == out1.tobytes()
    for f in ("J", "c_max", "status", "outer_iters", "inner_iters", "ls_rollouts"):
        assert np.array_equal(st[f], out1[f]), f
    assert np.all(lam[offs[1:] - 1] == 0.0) and np.all(lam >= 0.0)


def test_exported_state_matches_oracle(engine, slews):
    """CS1: status, counters and mu exactly as the oracle's export; multipliers to 1e-8 relative."""
    a = args_of(slews)
    for M1 in (7, 12):
        X, U, K, out, offs, st, lam = engine.alilqr_solve_state_batch(**a, opts=gpu_opts(M1))
        ref = AS.oracle_state_solve(slews, oracle_opts(M1))
        for f in ("status", "outer_iters", "inner_iters", "ls_rollouts"):
            assert np.array_equal(st[f], ref[4][f]), f
        assert np.array_equal(st["mu"], ref[4]["mu"])
        assert np.max(np.abs(st["lam_goal"] - ref[4]["lam_goal"])) <= 1e-8 * max(1.0, np.max(np.abs(ref[4]["lam_goal"])))
        assert np.max(np.abs(lam - ref[5])) <= 1e-8 * max(1.0, np.max(np.abs(ref[5])))
        assert np.max(np.abs(st["J"] - ref[4]["J"]) / np.abs(ref[4]["J"])) <= 1e-6


def check_continuation(engine, sl, M1, M2, pair=2, quat=0, generic=0):
    """Solve to M1 (exporting), continue to M2, and check the continued trials against the oracle's continuation and the
    direct GPU solve to M2; returns the statuses after M1 and after the continuation."""
    a = args_of(sl)
    o1, o2 = gpu_opts(M1, pair, quat), gpu_opts(M2, pair, quat)
    o1.k3_generic_inertia = o2.k3_generic_inertia = generic
    X, U, K, out, offs, st, lam = engine.alilqr_solve_state_batch(**a, opts=o1)
    Xc, Uc, Kc, oc, _, stc, lamc = engine.alilqr_solve_state_batch(**a, opts=o2, state=st, lam=lam, X=X, U=U)
    cont = out["status"] == 1
    split = engine.k3_last_split()
    assert split[0] < 0.05 and split[2] == int(cont.sum())   # no persistent launch; every continuing trial handed over
    Xd, Ud, Kd, od, _, std, lamd = engine.alilqr_solve_state_batch(**a, opts=o2)
    rX, rU, rK, ro, rs, rl = AS.oracle_state_solve(sl, oracle_opts(M2, quat), state=st, lam=lam, X=X, U=U)
    # against the oracle's continuation from the same exported state: the same iteration path on every trial
    for f in ("status", "outer_iters", "inner_iters", "ls_rollouts"):
        assert np.array_equal(oc[f], ro[f]), f
    assert np.array_equal(stc["mu"], rs["mu"])
    assert np.all(np.abs(oc["J"] - ro["J"]) <= 1e-6 * np.abs(ro["J"]))
    assert np.max(np.abs(stc["lam_goal"] - rs["lam_goal"])) <= 1e-8 * max(1.0, np.max(np.abs(rs["lam_goal"])))
    assert np.max(np.abs(lamc - rl)) <= 1e-8 * max(1.0, np.max(np.abs(rl)))
    assert np.max(np.abs(Xc - rX)) < 1e-6 and np.max(np.abs(Uc - rU)) < 1e-6
    # against the direct GPU solve to M2 (CS4: equal tolerance pairs): status and outer everywhere; counters on all but
    # at most 2 trials (the one-warp kernel is a separate compilation: last-bit differences can move a line search);
    # where the paths agree, J to 1e-10 and the trajectories and multipliers closely
    assert np.array_equal(oc["status"], od["status"]) and np.array_equal(oc["outer_iters"], od["outer_iters"])
    same = (oc["inner_iters"] == od["inner_iters"]) & (oc["ls_rollouts"] == od["ls_rollouts"])
    assert (~same).sum() <= 2
    assert np.all(np.abs(oc["J"][same] - od["J"][same]) <= 1e-10 * np.abs(od["J"][same]))
    for t in np.nonzero(same)[0]:
        r = slice(offs[t], offs[t + 1])
        assert np.max(np.abs(Xc[r] - Xd[r])) < 1e-8 and np.max(np.abs(lamc[r] - lamd[r])) <= 1e-8 * max(1.0, np.max(np.abs(lamd[r])))
    for t in np.nonzero(~cont)[0]:   # pass-through (CS2)
        r = slice(offs[t], offs[t + 1])
        assert np.array_equal(Xc[r], X[r]) and np.array_equal(Uc[r], U[r]) and np.array_equal(lamc[r], lam[r])
        assert stc[t].tobytes() == st[t].tobytes()
    return out["status"], oc["status"]


@pytest.mark.parametrize("pair,quat", [(0, 0), (1, 0), (2, 1)])
def test_continuation_matches_oracle_and_direct_solve(engine, slews, pair, quat):
    """M1 = 9: every slew continues and some converge after M1.  M1 = 12: the slews that converged before M1 pass
    through, the others continue to the end.  Continued trials against the oracle's continuation (counters exact, J, X,
    U and multipliers to tolerance) and against the direct solve to M2 = 20."""
    s9, c9 = check_continuation(engine, slews, 9, 20, pair, quat)
    assert np.all(s9 == 1) and np.any(c9 == 0)
    s12, c12 = check_continuation(engine, slews, 12, 20, pair, quat)
    assert np.any(s12 != 1) and np.any(s12 == 1)


@pytest.mark.parametrize("generic", [0, 1])
def test_general_inertia_export_and_continuation(engine, generic):
    """A non-diagonal inertia matrix runs the general-inertia instantiations (as does k3_generic_inertia = 1 with a
    diagonal one): the exporting fresh solve is bit-identical to ts_alilqr_solve_batch, and export and continuation
    match the oracle."""
    J = np.array([[2e-3, 1e-4, 0], [1e-4, 3e-3, 2e-4], [0, 2e-4, 1e-3]]) if not generic else S.J_1P
    mk = lambda angle, tfin: S.build_slew([0, 6578, 96, 0, 0, 90], J, S.quat_axis_angle([1, 0, 1], angle), np.array([1.0, 0, 0, 0]),
                                          t_final=tfin)
    sl = [mk(5.0, 60.0), mk(20.0, 30.0), mk(8.0, 40.0), mk(2.0, 20.0)]
    a = args_of(sl)
    o = gpu_opts(9, equal_tols=False)
    o.k3_generic_inertia = generic
    X0, U0, K0, out0, offs = engine.alilqr_solve_batch(**a, opts=o)
    X1, U1, K1, out1, _, st, lam = engine.alilqr_solve_state_batch(**a, opts=o)
    assert np.array_equal(X0, X1) and np.array_equal(U0, U1) and np.array_equal(K0, K1) and out0.tobytes() == out1.tobytes()
    check_continuation(engine, sl, 9, 14, generic=generic)


def test_pass_through_host_device_and_argument_errors(engine, slews):
    """CS2 pass-through is bitwise (X, U, K rows, outcome, state, lam), host and device pointers give bit-identical
    results, and a bad state is TS_ERR_ARG with nothing written."""
    import torch
    p = AS.pack(slews)
    tot = int(p["offs"][-1])
    T = len(slews)
    o12, o20 = gpu_opts(12), gpu_opts(20)
    X, U, K = np.zeros((tot, 8)), np.zeros((tot, 3)), np.zeros((tot, 24))
    out, st, lam = np.zeros(T, dtype=orc.OUTCOME_DTYPE), np.zeros(T, dtype=AS.AL_STATE_DTYPE), np.zeros((tot, 6))
    assert raw_call(engine, p, o12, X, U, K, out, 0, state_out=st, lam_out=lam) == 0
    K_given = np.random.default_rng(5).normal(size=K.shape)
    # continuing to max_outer = M1: everything passes through, bit for bit
    Xp, Up, Kp = X.copy(), U.copy(), K_given.copy()
    outp, stp, lamp = np.zeros(T, dtype=orc.OUTCOME_DTYPE), np.zeros(T, dtype=AS.AL_STATE_DTYPE), np.zeros((tot, 6))
    assert raw_call(engine, p, o12, Xp, Up, Kp, outp, 0, st, lam, stp, lamp) == 0
    assert np.array_equal(Xp, X) and np.array_equal(Up, U) and np.array_equal(Kp, K_given)
    assert outp.tobytes() == out.tobytes() and stp.tobytes() == st.tobytes() and np.array_equal(lamp, lam)
    # host vs device pointers on a continuation
    Xh, Uh, Kh = X.copy(), U.copy(), K_given.copy()
    outh, sth, lamh = np.zeros(T, dtype=orc.OUTCOME_DTYPE), np.zeros(T, dtype=AS.AL_STATE_DTYPE), np.zeros((tot, 6))
    assert raw_call(engine, p, o20, Xh, Uh, Kh, outh, 0, st, lam, sth, lamh) == 0
    dv = lambda a: torch.tensor(a, dtype=torch.float64, device="cuda")
    Xd, Ud, Kd, lamd_in, lamd = dv(X), dv(U), dv(K_given), dv(lam), dv(np.zeros((tot, 6)))
    p["B_dev"] = dv(p["B_eci"])
    torch.cuda.synchronize()
    outd, std = np.zeros(T, dtype=orc.OUTCOME_DTYPE), np.zeros(T, dtype=AS.AL_STATE_DTYPE)
    assert raw_call(engine, p, o20, Xd, Ud, Kd, outd, 1, st, lamd_in, std, lamd) == 0
    assert np.array_equal(Xd.cpu().numpy(), Xh) and np.array_equal(Ud.cpu().numpy(), Uh) and np.array_equal(Kd.cpu().numpy(), Kh)
    assert np.array_equal(lamd.cpu().numpy(), lamh) and outd.tobytes() == outh.tobytes() and std.tobytes() == sth.tobytes()
    for t in np.nonzero(st["status"] != 1)[0]:
        r = slice(p["offs"][t], p["offs"][t + 1])
        assert np.array_equal(Kh[r], K_given[r]) and np.array_equal(Xh[r], X[r])
    # argument errors: nothing written
    bad = []
    s1 = st.copy()
    s1["status"][1] = 7
    s2 = st.copy()
    s2["outer_iters"][0] = 0
    for si, li in ((st, None), (s1, lam), (s2, lam)):
        Xb, Ub, Kb = X.copy(), U.copy(), K_given.copy()
        ob, sb, lb = np.zeros(T, dtype=orc.OUTCOME_DTYPE), np.zeros(T, dtype=AS.AL_STATE_DTYPE), np.full((tot, 6), 3.0)
        bad.append(raw_call(engine, p, o20, Xb, Ub, Kb, ob, 0, si, li, sb, lb))
        assert np.array_equal(Xb, X) and np.array_equal(Ub, U) and np.array_equal(Kb, K_given)
        assert not ob.tobytes().strip(b"\0") and not sb.tobytes().strip(b"\0") and np.all(lb == 3.0)
    assert bad == [-2, -2, -2]
