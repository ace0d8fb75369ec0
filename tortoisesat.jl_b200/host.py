"""ctypes binding of libtortoise_b200.so + reference-named host functions.

Reference interface mirrored here (file:line in /root/reference/src):
  igrf12(date, r, lat, lon)                       igrf.jl:67-274
  igrf_data(altitude, year)                       magnetic_toolbox.jl:108-127
  its cubic B-spline interpolant                  magnetic_toolbox.jl:124-125   (MagFieldMap.interpolant)
(more entry points are added with each kernel)
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

TS_OK = 0
TS_ERR_CUDA, TS_ERR_ARG, TS_ERR_DATE, TS_ERR_DOMAIN, TS_ERR_NOMEM = -1, -2, -3, -4, -5

c_double_p = C.POINTER(C.c_double)
c_int64_p = C.POINTER(C.c_int64)


FIELD_OPTS_DTYPE = np.dtype([("GM", "<f8"), ("mjd", "<f8"), ("igrf_date", "<f8"), ("field_radius_m", "<f8"), ("t0", "<f8"),
                             ("tf", "<f8"), ("N", "<i8")])
GM_EARTH = 3.986004418E14 * (1 / 1000) ** 3  # km^3/s^2 (input_parameters.jl:26)


OUTCOME_DTYPE = np.dtype([("status", "<i4"), ("outer_iters", "<i4"), ("inner_iters", "<i4"), ("ls_rollouts", "<i4"),
                          ("N", "<i8"), ("J", "<f8"), ("c_max", "<f8"), ("t_final", "<f8"), ("slew_time", "<f8"),
                          ("flops", "<f8")])


# ts_al_state: the exported AL-iLQR solver state of one trial (CS1-CS4, DESIGN.md section 4, K3)
AL_STATE_DTYPE = np.dtype([("mu", "<f8"), ("lam_goal", "<f8", (8,)), ("J", "<f8"), ("c_max", "<f8"), ("status", "<i4"),
                           ("outer_iters", "<i4"), ("inner_iters", "<i4"), ("ls_rollouts", "<i4")])


class AlState(C.Structure):
    """ts_al_state (include/tortoise_b200.h), 104 bytes."""
    _fields_ = [("mu", C.c_double), ("lam_goal", C.c_double * 8), ("J", C.c_double), ("c_max", C.c_double),
                ("status", C.c_int32), ("outer_iters", C.c_int32), ("inner_iters", C.c_int32), ("ls_rollouts", C.c_int32)]


class IlqrOpts(C.Structure):
    """ts_ilqr_opts (include/tortoise_b200.h)."""
    _fields_ = [(k, C.c_int32) for k in ("max_outer", "max_inner", "max_linesearch", "dJ_counter_limit", "stage_cost_dt",
                                         "goal_mask")] + \
               [(k, C.c_double) for k in ("cost_tol", "cost_tol_intermediate", "grad_tol", "grad_tol_intermediate",
                                          "constraint_tol", "penalty_initial", "penalty_scaling", "penalty_max", "dual_max",
                                          "ls_lower", "ls_upper", "bp_reg_increase", "bp_reg_max", "bp_reg_min", "bp_reg_fp",
                                          "max_cost_value", "max_state_value", "max_control_value", "u_max", "u_min")] + \
               [(k, C.c_int32) for k in ("a2_active_ge", "a3_grad_over_N", "a4_no_intermediate", "a5_dual_active_only",
                                         "a6_penalty_conditional", "a7_carry_cost")] + \
               [("constraint_decrease_ratio", C.c_double), ("k3_suspend_after", C.c_int32), ("k3_tail_share", C.c_int32),
                ("k3_early_factor", C.c_double), ("k3_pair", C.c_int32), ("k3_wide_occ", C.c_int32),
                ("quat_error", C.c_int32), ("k3_generic_inertia", C.c_int32)]


class TvlqrOpts(C.Structure):
    """ts_tvlqr_opts (include/tortoise_b200.h)."""
    _fields_ = [("dt", C.c_double), ("t0", C.c_double), ("tf", C.c_double), ("Qd", C.c_double * 6), ("Qfd", C.c_double * 6),
                ("Rd", C.c_double * 3), ("dt_squared", C.c_int32), ("noise_mode", C.c_int32), ("seed", C.c_uint64),
                ("w_limit", C.c_double), ("ang_limit", C.c_double), ("literal_postproc", C.c_int32), ("pad_", C.c_int32)]


class FieldOpts(C.Structure):
    _fields_ = [("GM", C.c_double), ("mjd", C.c_double), ("igrf_date", C.c_double), ("field_radius_m", C.c_double),
                ("t0", C.c_double), ("tf", C.c_double), ("N", C.c_int64)]


class McConfig(C.Structure):
    """ts_mc_config"""
    _fields_ = [("n_trials", C.c_int64), ("shared_orbit", C.c_int32), ("run_tvlqr", C.c_int32), ("t0", C.c_double),
                ("tf", C.c_double), ("N_scope", C.c_int64), ("cutoff", C.c_double), ("dt", C.c_double), ("alpha", C.c_double),
                ("beta", C.c_double), ("eigen_axis_fix", C.c_int32), ("keep_trajectories", C.c_int32), ("ilqr", IlqrOpts),
                ("tvlqr", TvlqrOpts)]


class McStats(C.Structure):
    """ts_mc_stats"""
    _fields_ = [(k, C.c_int64) for k in ("n_trials", "n_converged", "n_no_cutoff", "n_fail_slew")] + \
               [(k, C.c_double) for k in ("sum_slew_time", "sum_slew_time_sq", "sum_t_final", "sum_inner_iters",
                                          "sum_ls_rollouts", "sum_knots", "flops", "ms_field", "ms_prep", "ms_solve",
                                          "ms_tvlqr")] + [("n_status", C.c_int64 * 6)]


class ReplayEnsembleOpts(C.Structure):
    """ts_replay_ensemble_opts (include/tortoise_b200.h)."""
    _fields_ = [("n_real", C.c_int64), ("r_first", C.c_int64), ("q_noise_scale", C.c_double)]


Q_NOISE_SCALE = (np.pi / 180) ** 2   # initial attitude noise of monte_carlo.jl: randn(3)*(pi/180)^2


def default_tvlqr_opts():
    o = TvlqrOpts()
    load_library().ts_tvlqr_default_opts(C.byref(o))
    return o


def default_mc_config(n_trials, shared_orbit=True, run_tvlqr=True, t0=0.0, tf=2400.0, N_scope=5000, cutoff=30.0, dt=0.2,
                      alpha=0.1, beta=1e3):
    """Defaults = the constants of src/monte_carlo.jl:37-78,169-171,227 (R_lqr = 0.5e3 there; TortoiseSat.jl:260 uses
    7.5e3, which is what ts_tvlqr_default_opts returns)."""
    cfg = McConfig()
    cfg.n_trials, cfg.shared_orbit, cfg.run_tvlqr = n_trials, int(shared_orbit), int(run_tvlqr)
    cfg.t0, cfg.tf, cfg.N_scope, cfg.cutoff, cfg.dt, cfg.alpha, cfg.beta = t0, tf, N_scope, cutoff, dt, alpha, beta
    cfg.eigen_axis_fix, cfg.keep_trajectories = 0, 0
    cfg.ilqr = default_ilqr_opts()
    cfg.tvlqr = default_tvlqr_opts()
    for i in range(3):
        cfg.tvlqr.Rd[i] = 0.5e3                                      # monte_carlo.jl:227
    return cfg


def default_ilqr_opts():
    o = IlqrOpts()
    load_library().ts_ilqr_default_opts(C.byref(o))
    return o


class TortoiseError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("tortoise_b200 error %d: %s" % (code, msg))
        self.code = code


def lib_path():
    """The in-tree library; TS_B200_LIB selects another build of the same sources (A/B runs of compile-time variants)."""
    return os.environ.get("TS_B200_LIB") or os.path.join(_HERE, "libtortoise_b200.so")


def load_library():
    """Loads the CUDA library.  Fails loudly (no fallback) if it is not built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    p = lib_path()
    if not os.path.exists(p):
        raise RuntimeError(
            "libtortoise_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'`; "
            "there is no CPU fallback." % p)
    L = C.CDLL(p)
    L.ts_version.restype = C.c_int
    L.ts_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.ts_create.restype = C.c_int
    L.ts_destroy.argtypes = [C.c_void_p]
    L.ts_destroy.restype = None
    L.ts_last_error.argtypes = [C.c_void_p]
    L.ts_last_error.restype = C.c_char_p
    L.ts_device_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_char_p, C.c_int]
    L.ts_launch_count.argtypes = [C.c_void_p]
    L.ts_launch_count.restype = C.c_int64
    L.ts_synchronize.argtypes = [C.c_void_p]
    L.ts_last_kernel_ms.argtypes = [C.c_void_p]
    L.ts_last_kernel_ms.restype = C.c_double
    L.ts_k3_last_split.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    L.ts_k3_last_split.restype = C.c_int
    L.ts_k3_last_parked.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]
    L.ts_k3_last_parked.restype = C.c_int
    L.ts_k3_last_cycles.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    L.ts_fp64_peak_probe.argtypes = [C.c_void_p, c_double_p]
    L.ts_fp64_latency_probe.argtypes = [C.c_void_p, c_double_p]
    L.ts_mc_trajectory_layout.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.ts_mc_fetch_trajectories.argtypes = [C.c_void_p] + [C.c_void_p] * 5
    L.ts_mc_fetch_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.ts_mc_continue.argtypes = [C.c_void_p, C.c_int64, C.POINTER(IlqrOpts), C.c_void_p, C.POINTER(McStats)]
    L.ts_mc_replay_ensemble.argtypes = [C.c_void_p, C.c_int64, C.POINTER(ReplayEnsembleOpts), C.c_int64] + [C.c_void_p] * 3
    L.ts_mc_replay_ensemble_last_split.argtypes = [C.c_void_p, c_double_p, c_double_p]
    L.ts_igrf12syn_batch.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_int64] + [C.c_void_p] * 7 + [C.c_int]
    L.ts_psiaki_pd_batch.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 7 + [C.c_double] * 3 + [C.c_void_p] * 3
    L.ts_attitude_dynamics_linear_batch.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 6
    L.ts_create_multi.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.c_int]
    L.ts_destroy_multi.argtypes = [C.c_void_p]
    L.ts_destroy_multi.restype = None
    L.ts_multi_last_error.argtypes = [C.c_void_p]
    L.ts_multi_last_error.restype = C.c_char_p
    L.ts_multi_device_count.argtypes = [C.c_void_p]
    L.ts_multi_ctx.argtypes = [C.c_void_p, C.c_int]
    L.ts_multi_ctx.restype = C.c_void_p
    L.ts_multi_monte_carlo_run.argtypes = [C.c_void_p, C.POINTER(McConfig)] + [C.c_void_p] * 8 + [C.POINTER(McStats)]
    L.ts_multi_mc_continue.argtypes = [C.c_void_p, C.c_int64, C.POINTER(IlqrOpts), C.c_void_p, C.POINTER(McStats)]
    L.ts_multi_mc_replay_ensemble.argtypes = [C.c_void_p, C.c_int64, C.POINTER(ReplayEnsembleOpts), C.c_int64] + [C.c_void_p] * 3
    L.ts_igrf12_batch.argtypes = [C.c_void_p, C.c_double, C.c_int64] + [C.c_void_p] * 6 + [C.c_int]
    L.ts_field_map_prefilter.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int]
    L.ts_field_map_eval_batch.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64] + [C.c_void_p] * 3 + [C.c_int]
    L.ts_magnetic_simulation_batch.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 7 + [C.c_int]
    L.ts_magnetic_gramian_batch.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 5 + [C.c_int]
    L.ts_condition_based_time_batch.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 5 + [C.c_int]
    L.ts_condition_cutoff_batch.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 6 + [C.c_int]
    L.ts_ilqr_default_opts.argtypes = [C.POINTER(IlqrOpts)]
    L.ts_ilqr_default_opts.restype = None
    L.ts_kep_eci_batch.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
    L.ts_orbit_rhs_batch.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.ts_legendre_schmidt_batch.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.ts_dynamics_batch.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_double,
                                    C.c_double, C.c_void_p, C.c_void_p]
    L.ts_rk3_step_batch.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_double,
                                    C.c_void_p, C.c_double, C.c_void_p]
    L.ts_tvlqr_default_opts.argtypes = [C.POINTER(TvlqrOpts)]
    L.ts_tvlqr_default_opts.restype = None
    L.ts_slew_weights_batch.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 4 + [C.c_double] * 4 + [C.c_int] + [C.c_void_p] * 6
    L.ts_tvlqr_sim_batch.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 14 + [C.POINTER(TvlqrOpts)] + [C.c_void_p] * 7 + [C.c_int]
    L.ts_monte_carlo_run.argtypes = [C.c_void_p, C.POINTER(McConfig)] + [C.c_void_p] * 8 + [C.POINTER(McStats)]
    L.ts_alilqr_solve_batch.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 13 + [C.c_double, C.c_void_p,
                                                                                      C.POINTER(IlqrOpts)] + [C.c_void_p] * 4 + [C.c_int]
    L.ts_alilqr_solve_state_batch.argtypes = L.ts_alilqr_solve_batch.argtypes + [C.c_void_p] * 4
    _LIB = L
    return L


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    """host numpy array or torch CUDA tensor -> raw address"""
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()  # torch tensor


def _is_tensor(a):
    return not isinstance(a, np.ndarray) and hasattr(a, "data_ptr")


def _cuda_f64(t):
    """a torch CUDA float64 tensor, contiguous (device-pointer path)"""
    if not _is_tensor(t) or not t.is_cuda or str(t.dtype) != "torch.float64":
        raise ValueError("the device path takes torch CUDA float64 tensors")
    return t.contiguous()


def _wait_for_torch(t):
    """The library runs on its own non-blocking stream: work torch has queued on the tensors (a copy, a random fill)
    must be finished before the library reads them."""
    import torch
    torch.cuda.current_stream(t.device).synchronize()


def _check_out(out, count):
    """a caller-provided output must be contiguous float64 storage of `count` values"""
    if _is_tensor(out):
        ok = out.is_cuda and str(out.dtype) == "torch.float64" and out.is_contiguous() and out.numel() == count
    else:
        ok = isinstance(out, np.ndarray) and out.dtype == np.float64 and out.flags.c_contiguous and out.size == count
    if not ok:
        raise ValueError("out must be contiguous float64 storage of %d values on the input's side" % count)


def _field_map_grid_dims(shape):
    if len(shape) != 3 or shape[2] != 3 or shape[0] < 2 or shape[1] < 2:
        raise ValueError("the field map grid must be n0 x n1 x 3 with n0, n1 >= 2, got %s" % (tuple(shape),))
    return int(shape[0]), int(shape[1])


def _field_map_coef_dims(shape):
    if len(shape) != 3 or shape[2] != 3 or shape[0] < 4 or shape[1] < 4:
        raise ValueError("field map coefficients must be (n0+2) x (n1+2) x 3 with n0, n1 >= 2, got %s" % (tuple(shape),))
    return int(shape[0]) - 2, int(shape[1]) - 2


class Engine:
    """One context per GPU (ts_ctx).  Not re-entrant."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.ts_create(C.byref(h), int(device))
        if rc != TS_OK:
            raise TortoiseError(rc, "ts_create(device=%d) failed: no usable CUDA device (there is no CPU fallback)" % device)
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.ts_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != TS_OK:
            raise TortoiseError(rc, self.lib.ts_last_error(self.h).decode())

    # -- bookkeeping
    def device_info(self):
        sm = C.c_int()
        name = C.create_string_buffer(128)
        self._check(self.lib.ts_device_info(self.h, C.byref(sm), name, 128))
        return sm.value, name.value.decode()

    def launch_count(self):
        return int(self.lib.ts_launch_count(self.h))

    def last_kernel_ms(self):
        return float(self.lib.ts_last_kernel_ms(self.h))

    def k3_last_split(self):
        """(persistent-kernel ms, straggler-kernel ms, trials handed over) of the most recent AL-iLQR solve."""
        a, b, n = C.c_double(0), C.c_double(0), C.c_int64(0)
        self._check(self.lib.ts_k3_last_split(self.h, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, int(n.value)

    def synchronize(self):
        self._check(self.lib.ts_synchronize(self.h))

    def fp64_peak_tflops(self):
        v = C.c_double()
        self._check(self.lib.ts_fp64_peak_probe(self.h, C.byref(v)))
        return v.value

    # -- K1 ---------------------------------------------------------------
    def igrf12_batch(self, date, r_m, lat, lon, out=None):
        """Batched igrf12 (igrf.jl:67-274).  numpy in -> numpy out (host path), or
        torch CUDA float64 tensors in -> `out` tensors filled (device path)."""
        if isinstance(r_m, np.ndarray) or np.isscalar(r_m) or isinstance(r_m, (list, tuple)):
            r_m, lat, lon = _f64(np.atleast_1d(r_m)), _f64(np.atleast_1d(lat)), _f64(np.atleast_1d(lon))
            n = r_m.shape[0]
            if not (lat.shape[0] == n and lon.shape[0] == n):
                raise ValueError("r, lat, lon must have the same length")
            if out is not None:   # caller-provided host outputs (e.g. views of pinned memory)
                Bn, Be, Bd = out
            else:
                Bn, Be, Bd = np.empty(n), np.empty(n), np.empty(n)
            rc = self.lib.ts_igrf12_batch(self.h, float(date), n, _ptr(r_m), _ptr(lat), _ptr(lon), _ptr(Bn), _ptr(Be),
                                          _ptr(Bd), 0)
            if rc == TS_ERR_DOMAIN:
                raise TortoiseError(rc, self.lib.ts_last_error(self.h).decode())
            self._check(rc)
            return Bn, Be, Bd
        n = r_m.numel()
        Bn, Be, Bd = out
        self._check(self.lib.ts_igrf12_batch(self.h, float(date), n, _ptr(r_m), _ptr(lat), _ptr(lon), _ptr(Bn), _ptr(Be),
                                             _ptr(Bd), 1))
        return Bn, Be, Bd

    # -- K8 ---------------------------------------------------------------
    def field_map_prefilter(self, grid, out=None):
        """FM1 (DESIGN section 4, K8) of the cubic B-spline of magnetic_toolbox.jl:124-125: n0 x n1 x 3 grid ->
        (n0+2) x (n1+2) x 3 coefficients.  numpy in -> numpy out (host path), or a torch CUDA float64 tensor in ->
        a tensor out (device path; `out` is allocated when not given)."""
        if _is_tensor(grid):
            n0, n1 = _field_map_grid_dims(grid.shape)
            grid = _cuda_f64(grid)
            if out is None:
                import torch
                out = torch.empty((n0 + 2, n1 + 2, 3), dtype=torch.float64, device=grid.device)
            _check_out(out, (n0 + 2) * (n1 + 2) * 3)
            _wait_for_torch(grid)
            self._check(self.lib.ts_field_map_prefilter(self.h, n0, n1, _ptr(grid), _ptr(out), 1))
            return out
        grid = _f64(grid)
        n0, n1 = _field_map_grid_dims(grid.shape)
        out = np.empty((n0 + 2, n1 + 2, 3)) if out is None else out
        _check_out(out, (n0 + 2) * (n1 + 2) * 3)
        self._check(self.lib.ts_field_map_prefilter(self.h, n0, n1, _ptr(grid), _ptr(out), 0))
        return out

    def field_map_eval_batch(self, coefs, x0, x1, out=None):
        """FM2 + FM3: the spline with coefficients `coefs` ((n0+2) x (n1+2) x 3) at the 1-based fractional indices
        (x0[p], x1[p]) -> n x 3 (all three components).  Host arrays -> numpy out; torch CUDA float64 tensors (coefs,
        x0, x1) -> a tensor out.  A non-finite index raises TortoiseError (code TS_ERR_DOMAIN) after the other rows of
        `out` (if given) have been written; the offending rows are NaN."""
        if _is_tensor(coefs):
            n0, n1 = _field_map_coef_dims(coefs.shape)
            coefs, x0, x1 = _cuda_f64(coefs), _cuda_f64(x0).reshape(-1), _cuda_f64(x1).reshape(-1)
            n = x0.numel()
            if x1.numel() != n:
                raise ValueError("x0 and x1 must have the same length")
            if out is None:
                import torch
                out = torch.empty((n, 3), dtype=torch.float64, device=coefs.device)
            _check_out(out, n * 3)
            _wait_for_torch(coefs)
            self._check(self.lib.ts_field_map_eval_batch(self.h, n0, n1, _ptr(coefs), n, _ptr(x0), _ptr(x1), _ptr(out), 1))
            return out
        coefs = _f64(coefs)
        n0, n1 = _field_map_coef_dims(coefs.shape)
        x0, x1 = _f64(np.atleast_1d(x0)).reshape(-1), _f64(np.atleast_1d(x1)).reshape(-1)
        if x0.shape != x1.shape:
            raise ValueError("x0 and x1 must have the same length")
        out = np.empty((x0.shape[0], 3)) if out is None else out
        _check_out(out, x0.shape[0] * 3)
        self._check(self.lib.ts_field_map_eval_batch(self.h, n0, n1, _ptr(coefs), x0.shape[0], _ptr(x0), _ptr(x1), _ptr(out), 0))
        return out

    # -- K2 ---------------------------------------------------------------
    def magnetic_simulation_batch(self, kep6, opts, rows_limit=None, want_pos=False):
        """Batched magnetic_simulation (magnetic_toolbox.jl:33-106).  kep6: (T,6); opts:
        structured array FIELD_OPTS_DTYPE of length T.  Returns (B_eci, B_offs[, pos, vel])
        with B_eci rows concatenated per trial (2N_t rows each)."""
        kep6 = _f64(np.atleast_2d(kep6))
        T = kep6.shape[0]
        opts = np.ascontiguousarray(opts, dtype=FIELD_OPTS_DTYPE)
        offs = np.zeros(T + 1, dtype=np.int64)
        offs[1:] = np.cumsum(2 * opts["N"])
        B = np.empty((int(offs[-1]), 3))
        pos = np.empty((int(offs[-1]) + T, 3)) if want_pos else None
        vel = np.empty((int(offs[-1]) + T, 3)) if want_pos else None
        lim = None if rows_limit is None else np.ascontiguousarray(rows_limit, dtype=np.int64)
        self._check(self.lib.ts_magnetic_simulation_batch(
            self.h, T, _ptr(kep6), opts.ctypes.data, _ptr(offs), None if lim is None else _ptr(lim), _ptr(B),
            None if pos is None else _ptr(pos), None if vel is None else _ptr(vel), 0))
        if want_pos:
            return B, offs, pos, vel
        return B, offs

    def magnetic_gramian_batch(self, B, offs, rows, dt):
        B = _f64(B)
        offs = np.ascontiguousarray(offs, dtype=np.int64)
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        dt = _f64(dt)
        G = np.empty((B.shape[0], 3, 3))
        self._check(self.lib.ts_magnetic_gramian_batch(self.h, rows.shape[0], _ptr(B), _ptr(offs), _ptr(rows), _ptr(dt), _ptr(G), 0))
        return G

    def condition_based_time_batch(self, G, offs, rows, cutoff):
        G = _f64(G)
        offs = np.ascontiguousarray(offs, dtype=np.int64)
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        cutoff = _f64(cutoff)
        idx = np.zeros(rows.shape[0], dtype=np.int64)
        self._check(self.lib.ts_condition_based_time_batch(self.h, rows.shape[0], _ptr(G), _ptr(offs), _ptr(rows), _ptr(cutoff),
                                                           _ptr(idx), 0))
        return idx

    def condition_cutoff_batch(self, B, offs, rows, dt, cutoff):
        B = _f64(B)
        offs = np.ascontiguousarray(offs, dtype=np.int64)
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        dt, cutoff = _f64(dt), _f64(cutoff)
        idx = np.zeros(rows.shape[0], dtype=np.int64)
        self._check(self.lib.ts_condition_cutoff_batch(self.h, rows.shape[0], _ptr(B), _ptr(offs), _ptr(rows), _ptr(dt),
                                                       _ptr(cutoff), _ptr(idx), 0))
        return idx


    # -- K3 ---------------------------------------------------------------
    @staticmethod
    def _alilqr_inputs(N_i, x0, xf, Jmat, Qd, Qfd, Rd, B_eci, B_offs, B_rows, index_scale, clock_rate, dt, U0, opts):
        """The host arrays of ts_alilqr_solve_batch / ts_alilqr_solve_state_batch up to U0 and opts, in order, plus
        (T, offs).  The arrays are kept referenced by the returned tuple for the duration of the call."""
        N_i = np.ascontiguousarray(N_i, dtype=np.int64)
        T = N_i.shape[0]
        offs = np.zeros(T + 1, dtype=np.int64)
        offs[1:] = np.cumsum(N_i)
        arr = lambda a, w: _f64(np.asarray(a, dtype=np.float64).reshape(T, w))
        keep = [N_i, offs, arr(x0, 8), arr(xf, 8), arr(Jmat, 9), arr(Qd, 8), arr(Qfd, 8), arr(Rd, 3), _f64(B_eci),
                np.ascontiguousarray(B_offs, dtype=np.int64), np.ascontiguousarray(B_rows, dtype=np.int64), _f64(index_scale),
                _f64(clock_rate)]
        U0a = None if U0 is None else _f64(U0)
        o = opts if opts is not None else default_ilqr_opts()
        args = [T] + [_ptr(a) for a in keep] + [float(dt), None if U0a is None else _ptr(U0a), C.byref(o)]
        return T, offs, args, (keep, U0a, o)

    def alilqr_solve_batch(self, N_i, x0, xf, Jmat, Qd, Qfd, Rd, B_eci, B_offs, B_rows, index_scale, clock_rate, dt,
                           U0=None, opts=None, want_K=True):
        """Batched AL-iLQR solve (TortoiseSat.jl:145-146,169,178-199).  Per-trial rows in
        x0/xf (T,8), Jmat (T,9), Qd/Qfd (T,8), Rd (T,3); ragged knots addressed through
        offs = cumsum(N_i).  Returns (X, U, K, outcomes, offs): X (sum N, 8), U (sum N, 3)
        [row offs[t]+N_t-1 unused], K (sum N, 3, 8) or None."""
        T, offs, args, _keep = self._alilqr_inputs(N_i, x0, xf, Jmat, Qd, Qfd, Rd, B_eci, B_offs, B_rows, index_scale, clock_rate,
                                                   dt, U0, opts)
        tot = int(offs[-1])
        X = np.zeros((tot, 8))
        U = np.zeros((tot, 3))
        K = np.zeros((tot, 3, 8)) if want_K else None
        out = np.zeros(T, dtype=OUTCOME_DTYPE)
        self._check(self.lib.ts_alilqr_solve_batch(self.h, *args, _ptr(X), _ptr(U), None if K is None else _ptr(K), out.ctypes.data, 0))
        return X, U, K, out, offs

    def alilqr_solve_state_batch(self, N_i, x0, xf, Jmat, Qd, Qfd, Rd, B_eci, B_offs, B_rows, index_scale, clock_rate, dt,
                                 U0=None, opts=None, want_K=True, state=None, lam=None, X=None, U=None):
        """alilqr_solve_batch that also returns each trial's solver state and bound multipliers, and continues from them.
        state=None: a fresh solve (the same results as alilqr_solve_batch).  With `state` (AL_STATE_DTYPE, T records)
        and `lam` ((sum N, 6)) from an earlier call, plus that call's X and U: the trials that ended at max_outer with
        outer_iters < opts.max_outer continue (CS2, CS3); the others pass through (their K rows stay zero here).  Returns
        (X, U, K, out, offs, state, lam), state as AL_STATE_DTYPE records, lam (sum N, 6) [row offs[t]+N_t-1 zero]."""
        T, offs, args, _keep = self._alilqr_inputs(N_i, x0, xf, Jmat, Qd, Qfd, Rd, B_eci, B_offs, B_rows, index_scale, clock_rate,
                                                   dt, U0, opts)
        tot = int(offs[-1])
        if state is not None:
            if lam is None or X is None or U is None:
                raise ValueError("continuing from a state needs the lam, X and U it was exported with")
            state = np.ascontiguousarray(state, dtype=AL_STATE_DTYPE)
            if state.shape != (T,):
                raise ValueError("state must hold one record per trial")
            lam_in = np.ascontiguousarray(lam, dtype=np.float64).reshape(tot, 6)
            X = np.array(X, dtype=np.float64, order="C").reshape(tot, 8)     # copies: the call writes X and U in place
            U = np.array(U, dtype=np.float64, order="C").reshape(tot, 3)
        else:
            lam_in = None
            X, U = np.zeros((tot, 8)), np.zeros((tot, 3))
        K = np.zeros((tot, 3, 8)) if want_K else None
        out = np.zeros(T, dtype=OUTCOME_DTYPE)
        st_out = np.zeros(T, dtype=AL_STATE_DTYPE)
        lam_out = np.zeros((tot, 6))
        self._check(self.lib.ts_alilqr_solve_state_batch(
            self.h, *args, _ptr(X), _ptr(U), None if K is None else _ptr(K), out.ctypes.data, 0,
            None if state is None else state.ctypes.data, None if lam_in is None else _ptr(lam_in), st_out.ctypes.data,
            _ptr(lam_out)))
        return X, U, K, out, offs, st_out, lam_out


    # -- element-wise building blocks --------------------------------------
    def kep_eci_batch(self, kep6, t0=None, GM=GM_EARTH):
        kep6 = _f64(np.atleast_2d(kep6))
        n = kep6.shape[0]
        t0a = None if t0 is None else _f64(np.broadcast_to(np.asarray(t0, dtype=float), (n,)))
        rv = np.zeros((n, 6))
        self._check(self.lib.ts_kep_eci_batch(self.h, n, _ptr(kep6), None if t0a is None else _ptr(t0a), GM, _ptr(rv)))
        return rv

    def orbit_rhs_batch(self, x6):
        x6 = _f64(np.atleast_2d(x6))
        dx = np.zeros_like(x6)
        self._check(self.lib.ts_orbit_rhs_batch(self.h, x6.shape[0], _ptr(x6), _ptr(dx)))
        return dx

    def legendre_schmidt_batch(self, theta, n_max=13, want_dP=True):
        theta = _f64(np.atleast_1d(theta))
        n = theta.shape[0]
        P = np.zeros((n, n_max + 1, n_max + 1))
        dP = np.zeros_like(P) if want_dP else None
        self._check(self.lib.ts_legendre_schmidt_batch(self.h, n, _ptr(theta), n_max, _ptr(P), None if dP is None else _ptr(dP)))
        return (P, dP) if want_dP else P

    def dynamics_batch(self, mode, x, u, B, Jmat, index_scale=1.0, clock_rate=0.0):
        """mode 0 DerivFunction, 1 gain_simulator (x n x 8, B = field table), 2 attitude_dynamics (x n x 7, B = n x 3 body field)."""
        x, u, B, Jmat = _f64(np.atleast_2d(x)), _f64(np.atleast_2d(u)), _f64(np.atleast_2d(B)), _f64(np.asarray(Jmat).reshape(9))
        dx = np.zeros_like(x)
        self._check(self.lib.ts_dynamics_batch(self.h, mode, x.shape[0], _ptr(x), _ptr(u), _ptr(B), B.shape[0], float(index_scale),
                                               float(clock_rate), _ptr(Jmat), _ptr(dx)))
        return dx

    def rk3_step_batch(self, x, u, B, Jmat, index_scale, clock_rate, dt):
        x, u, B, Jmat = _f64(np.atleast_2d(x)), _f64(np.atleast_2d(u)), _f64(np.atleast_2d(B)), _f64(np.asarray(Jmat).reshape(9))
        xn = np.zeros_like(x)
        self._check(self.lib.ts_rk3_step_batch(self.h, x.shape[0], _ptr(x), _ptr(u), _ptr(B), B.shape[0], float(index_scale),
                                               float(clock_rate), _ptr(Jmat), float(dt), _ptr(xn)))
        return xn

    # -- prep / K4 / fused MC ----------------------------------------------
    def slew_weights_batch(self, x0, xf, Jmat, t_final, t0=0.0, dt=0.2, alpha=10.0, beta=1e3, want_guess=False, eigen_axis_fix=False):
        """eigen_axis_slew + Bryson weights (eigen_axis_slew.jl:1-38, TortoiseSat.jl:157-168).  eigen_axis_fix=False
        reproduces the reference's literal error quaternion qmult(q_f, q_0) (eigen_axis_slew.jl:16); True uses
        conj(q_f) (x) q_0."""
        x0 = _f64(np.atleast_2d(x0))
        T = x0.shape[0]
        xf, Jmat, t_final = _f64(np.asarray(xf).reshape(T, 8)), _f64(np.asarray(Jmat).reshape(T, 9)), _f64(np.asarray(t_final).reshape(T))
        Qd, Qfd, Rd = np.zeros((T, 8)), np.zeros((T, 8)), np.zeros((T, 3))
        goffs = wg = qg = None
        if want_guess:
            nt = np.array([int(np.floor((tf_ - t0) / dt + 1e-9)) + 1 for tf_ in t_final], dtype=np.int64)
            goffs = np.concatenate([[0], np.cumsum(nt)]).astype(np.int64)
            wg, qg = np.zeros((int(goffs[-1]), 3)), np.zeros((int(goffs[-1]), 4))
        self._check(self.lib.ts_slew_weights_batch(self.h, T, _ptr(x0), _ptr(xf), _ptr(Jmat), _ptr(t_final), t0, dt, alpha, beta,
                                                   int(bool(eigen_axis_fix)), _ptr(Qd), _ptr(Qfd), _ptr(Rd), None if goffs is None else _ptr(goffs),
                                                   None if wg is None else _ptr(wg), None if qg is None else _ptr(qg)))
        if want_guess:
            return Qd, Qfd, Rd, wg, qg, goffs
        return Qd, Qfd, Rd

    def tvlqr_sim_batch(self, N_i, X_lqr, U_lqr, x0_lqr, Jmat, B_eci, B_offs, B_rows, index_scale, clock_rate, t_final, q_final,
                        opts=None, noise=None, stream_id=None, want_traj=True):
        """Batched attitude_simulation (attitude_controller.jl:1-48) + slew-time rule.  X_lqr (sum N, 8),
        U_lqr (sum N, 3) ragged by offs = cumsum(N_i)."""
        N_i = np.ascontiguousarray(N_i, dtype=np.int64)
        T = N_i.shape[0]
        offs = np.zeros(T + 1, dtype=np.int64)
        offs[1:] = np.cumsum(N_i)
        tot = int(offs[-1])
        X_lqr, U_lqr = _f64(X_lqr), _f64(U_lqr)
        arr = lambda a, w: _f64(np.asarray(a, dtype=np.float64).reshape(T, w))
        x0_lqr, Jmat, q_final = arr(x0_lqr, 8), arr(Jmat, 9), arr(q_final, 4)
        B_eci = _f64(B_eci)
        B_offs = np.ascontiguousarray(B_offs, dtype=np.int64)
        B_rows = np.ascontiguousarray(B_rows, dtype=np.int64)
        index_scale, clock_rate, t_final = _f64(index_scale), _f64(clock_rate), _f64(t_final)
        o = opts if opts is not None else default_tvlqr_opts()
        nz = None if noise is None else _f64(noise)
        sid = None if stream_id is None else np.ascontiguousarray(stream_id, dtype=np.uint32)
        Xs = np.zeros((tot, 8)) if want_traj else None
        Us = np.zeros((tot, 3)) if want_traj else None
        dX = np.zeros((tot, 6)) if want_traj else None
        K = np.zeros((tot, 3, 6)) if want_traj else None
        nsim = np.zeros(T, dtype=np.int64)
        slew = np.zeros(T)
        pp = lambda a: None if a is None else _ptr(a)
        self._check(self.lib.ts_tvlqr_sim_batch(self.h, T, _ptr(N_i), _ptr(offs), _ptr(X_lqr), _ptr(U_lqr), _ptr(x0_lqr), _ptr(Jmat),
                                                _ptr(B_eci), _ptr(B_offs), _ptr(B_rows), _ptr(index_scale), _ptr(clock_rate),
                                                _ptr(t_final), _ptr(q_final), pp(sid), C.byref(o), pp(nz), pp(Xs), pp(Us), pp(dX),
                                                pp(K), _ptr(nsim), _ptr(slew), 0))
        return Xs, Us, dX, K, nsim, slew, offs

    def monte_carlo_run(self, cfg, kep6, fopts, x0, xf, Jmat, q_noise0=None, stream_id=None):
        """Fused Monte-Carlo (monte_carlo.jl:118-262 with the solver block of TortoiseSat.jl:178-199).
        fopts: structured array FIELD_OPTS_DTYPE (only GM, mjd, igrf_date, field_radius_m are read)."""
        n = int(cfg.n_trials)
        kep6 = _f64(np.atleast_2d(kep6))
        fopts = np.ascontiguousarray(fopts, dtype=FIELD_OPTS_DTYPE)
        x0, xf, Jmat = _f64(np.asarray(x0).reshape(n, 8)), _f64(np.asarray(xf).reshape(n, 8)), _f64(np.asarray(Jmat).reshape(n, 9))
        qn = None if q_noise0 is None else _f64(np.asarray(q_noise0).reshape(n, 3))
        sid = None if stream_id is None else np.ascontiguousarray(stream_id, dtype=np.uint32)
        out = np.zeros(n, dtype=OUTCOME_DTYPE)
        st = McStats()
        self._check(self.lib.ts_monte_carlo_run(self.h, C.byref(cfg), _ptr(kep6), fopts.ctypes.data, _ptr(x0), _ptr(xf), _ptr(Jmat),
                                                None if qn is None else _ptr(qn), None if sid is None else _ptr(sid),
                                                out.ctypes.data, C.byref(st)))
        return out, st

    def fp64_latency_cycles(self):
        """SM cycles per dependent DFMA, DADD/DMUL, rsqrt+DADD, and shared-memory round trip (ts_fp64_latency_probe)."""
        v = (C.c_double * 4)()
        self._check(self.lib.ts_fp64_latency_probe(self.h, v))
        return dict(zip(("dfma", "dadd_dmul", "rsqrt_dadd", "smem_roundtrip"), [float(x) for x in v]))

    def k3_last_cycles(self, n_trials):
        """(n_trials, 3) SM cycles of the last AL-iLQR solve: backward pass, forward pass, linearisation share."""
        cyc = np.zeros((int(n_trials), 3))
        self._check(self.lib.ts_k3_last_cycles(self.h, int(n_trials), _ptr(cyc)))
        return cyc

    def k3_last_parked(self, cap):
        """Trials the last AL-iLQR solve handed to its second launch: (trial index, outer count, inner count at parking)."""
        cap = int(cap)
        tr, ou, inn = np.zeros(cap, dtype=np.int64), np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.int32)
        n = C.c_int64(0)
        self._check(self.lib.ts_k3_last_parked(self.h, cap, _ptr(tr), _ptr(ou), _ptr(inn), C.byref(n)))
        return tr[:n.value], ou[:n.value], inn[:n.value]

    def mc_trajectories(self, n_trials, want=("X", "U", "X_sim", "U_sim", "B_eci")):
        """Trajectories of the last monte_carlo_run with cfg.keep_trajectories = 1: dict with knot_offs, row_offs and the
        requested arrays (`states`, `control_inputs`, `sim_states`, `sim_control_inputs`, `B_ECI_total` of
        monte_carlo.jl:52-66, ragged by knot_offs / row_offs)."""
        n = int(n_trials)
        ko, ro = np.zeros(n + 1, dtype=np.int64), np.zeros(n + 1, dtype=np.int64)
        self._check(self.lib.ts_mc_trajectory_layout(self.h, n, _ptr(ko), _ptr(ro)))
        K, R = int(ko[-1]), int(ro[-1])
        res = {"knot_offs": ko, "row_offs": ro}
        shapes = {"X": (K, 8), "U": (K, 3), "X_sim": (K, 8), "U_sim": (K, 3), "B_eci": (R, 3)}
        for k in want:
            res[k] = np.zeros(shapes[k])
        g = lambda k: _ptr(res[k]) if k in res else None
        self._check(self.lib.ts_mc_fetch_trajectories(self.h, g("X"), g("U"), g("X_sim"), g("U_sim"), g("B_eci")))
        return res

    def mc_state(self, n_trials):
        """The kept solver state of the last monte_carlo_run with cfg.keep_trajectories = 2 (ts_mc_fetch_state): (state,
        lam), state as AL_STATE_DTYPE records (a NO_CUTOFF trial: zero record with status 5), lam (sum N, 6) ragged by the
        knot_offs of mc_trajectories."""
        n = int(n_trials)
        ko = np.zeros(n + 1, dtype=np.int64)
        self._check(self.lib.ts_mc_trajectory_layout(self.h, n, _ptr(ko), None))
        state = np.zeros(n, dtype=AL_STATE_DTYPE)
        lam = np.zeros((int(ko[-1]), 6))
        self._check(self.lib.ts_mc_fetch_state(self.h, state.ctypes.data, _ptr(lam)))
        return state, lam

    def mc_continue(self, n_trials, opts):
        """Continues the max-outer trials of the last monte_carlo_run with cfg.keep_trajectories = 2 under `opts` (an
        IlqrOpts with a larger max_outer; rules MC1-MC4 of ts_mc_continue).  Returns (out, stats) for the whole ensemble;
        the kept run is updated in place, so mc_trajectories / mc_state return the continued run."""
        n = int(n_trials)
        out = np.zeros(n, dtype=OUTCOME_DTYPE)
        st = McStats()
        self._check(self.lib.ts_mc_continue(self.h, n, C.byref(opts), out.ctypes.data, C.byref(st)))
        return out, st

    def mc_replay_ensemble(self, n_trials, n_real, r_first=0, trials=None, q_noise_scale=Q_NOISE_SCALE, want_x_final=False):
        """The kept run's slews (last monte_carlo_run with cfg.keep_trajectories >= 1) replayed under n_real independent
        disturbance draws each (ts_mc_replay_ensemble, rules RE1-RE5): realisations r_first .. r_first + n_real - 1 of the
        selected trials (caller indices, repeats allowed; None = all).  Returns (slew_time (n_sel, n_real), x_final
        (n_sel, n_real, 8) or None); a NO_CUTOFF trial gets NaN rows."""
        return _replay_ensemble(self.lib.ts_mc_replay_ensemble, self.h, n_trials, n_real, r_first, trials, q_noise_scale,
                                want_x_final, self._check)

    def mc_replay_ensemble_split(self):
        """Device ms of the last mc_replay_ensemble: (gains, ensemble replay)."""
        g, r = C.c_double(), C.c_double()
        self._check(self.lib.ts_mc_replay_ensemble_last_split(self.h, C.byref(g), C.byref(r)))
        return g.value, r.value

    def igrf12syn_batch(self, isv, date, itype, alt, colat, elong):
        """igrf12syn (igrf.jl:335-534) at n points: alt km, colat/elong degrees -> x, y, z, f (nT)."""
        alt, colat, elong = _f64(np.atleast_1d(alt)), _f64(np.atleast_1d(colat)), _f64(np.atleast_1d(elong))
        n = alt.shape[0]
        o = [np.zeros(n) for _ in range(4)]
        self._check(self.lib.ts_igrf12syn_batch(self.h, int(isv), float(date), int(itype), n, _ptr(alt), _ptr(colat), _ptr(elong),
                                                _ptr(o[0]), _ptr(o[1]), _ptr(o[2]), _ptr(o[3]), 0))
        return tuple(o)


    def psiaki_pd_batch(self, N_i, x0, w_guess, q_guess, B_eci, Jmat, dt, C_1, C_2):
        """Batched Psiaki-style PD closed loop (comparison/psiaki2005.jl:116-164).  Ragged by offs = cumsum(N_i): w_guess
        (sum N, 3), q_guess (sum N, 4), B_eci (sum N, 3); x0 (T, 7), Jmat (T, 9).  Returns X (sum N, 7), M (sum N, 3),
        q_err (sum N, 4), offs."""
        N_i = np.ascontiguousarray(N_i, dtype=np.int64)
        T = N_i.shape[0]
        offs = np.zeros(T + 1, dtype=np.int64)
        offs[1:] = np.cumsum(N_i)
        tot = int(offs[-1])
        x0, Jmat = _f64(np.asarray(x0).reshape(T, 7)), _f64(np.asarray(Jmat).reshape(T, 9))
        wg, qg, B = _f64(np.asarray(w_guess).reshape(tot, 3)), _f64(np.asarray(q_guess).reshape(tot, 4)), _f64(np.asarray(B_eci).reshape(tot, 3))
        X, M, Qe = np.zeros((tot, 7)), np.zeros((tot, 3)), np.zeros((tot, 4))
        self._check(self.lib.ts_psiaki_pd_batch(self.h, T, _ptr(N_i), _ptr(offs), _ptr(x0), _ptr(wg), _ptr(qg), _ptr(B), _ptr(Jmat),
                                                float(dt), float(C_1), float(C_2), _ptr(X), _ptr(M), _ptr(Qe)))
        return X, M, Qe, offs

    def attitude_dynamics_linear_batch(self, x, u, x_linear, B_B, Jmat):
        x, u, xl, B = _f64(np.atleast_2d(x)), _f64(np.atleast_2d(u)), _f64(np.atleast_2d(x_linear)), _f64(np.atleast_2d(B_B))
        n = x.shape[0]
        dx = np.zeros((n, 7))
        J = _f64(np.asarray(Jmat).reshape(9))
        self._check(self.lib.ts_attitude_dynamics_linear_batch(self.h, n, _ptr(x), _ptr(u), _ptr(xl), _ptr(B), _ptr(J), _ptr(dx)))
        return dx


class MultiEngine:
    """Several GPUs of one node behind one handle (ts_create_multi): the library owns one context, one host thread and
    one NCCL communicator per device; trials are sharded round-robin."""

    def __init__(self, devices):
        self.lib = load_library()
        ids = (C.c_int * len(devices))(*[int(d) for d in devices])
        h = C.c_void_p()
        rc = self.lib.ts_create_multi(C.byref(h), ids, len(devices))
        if rc != 0 or not h.value:
            raise TortoiseError(rc, "ts_create_multi failed (no usable CUDA devices / NCCL?) -- there is no CPU fallback")
        self.h = h

    def close(self):
        if getattr(self, "h", None) is not None and self.h.value:
            self.lib.ts_destroy_multi(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def device_count(self):
        return int(self.lib.ts_multi_device_count(self.h))

    def monte_carlo_run(self, cfg, kep6, fopts, x0, xf, Jmat, q_noise0=None, stream_id=None):
        n = int(cfg.n_trials)
        kep6 = _f64(np.atleast_2d(kep6))
        fopts = np.ascontiguousarray(fopts, dtype=FIELD_OPTS_DTYPE)
        x0, xf, Jmat = _f64(np.asarray(x0).reshape(n, 8)), _f64(np.asarray(xf).reshape(n, 8)), _f64(np.asarray(Jmat).reshape(n, 9))
        qn = None if q_noise0 is None else _f64(np.asarray(q_noise0).reshape(n, 3))
        sid = None if stream_id is None else np.ascontiguousarray(stream_id, dtype=np.uint32)
        out = np.zeros(n, dtype=OUTCOME_DTYPE)
        st = McStats()
        rc = self.lib.ts_multi_monte_carlo_run(self.h, C.byref(cfg), _ptr(kep6), fopts.ctypes.data, _ptr(x0), _ptr(xf), _ptr(Jmat),
                                               None if qn is None else _ptr(qn), None if sid is None else _ptr(sid),
                                               out.ctypes.data, C.byref(st))
        if rc != 0:
            raise TortoiseError(rc, (self.lib.ts_multi_last_error(self.h) or b"").decode())
        return out, st

    def mc_continue(self, n_trials, opts):
        """Engine.mc_continue on every device's kept shard, records gathered and statistics reduced as after the run.
        (With one process per GPU, each rank calls Engine.mc_continue and then parallel.gather_outcomes / reduce_stats.)"""
        n = int(n_trials)
        out = np.zeros(n, dtype=OUTCOME_DTYPE)
        st = McStats()
        rc = self.lib.ts_multi_mc_continue(self.h, n, C.byref(opts), out.ctypes.data, C.byref(st))
        if rc != 0:
            raise TortoiseError(rc, (self.lib.ts_multi_last_error(self.h) or b"").decode())
        return out, st

    def mc_replay_ensemble(self, n_trials, n_real, r_first=0, trials=None, q_noise_scale=Q_NOISE_SCALE, want_x_final=False):
        """Engine.mc_replay_ensemble over the devices' kept shards: each trial on the device that holds it (t mod
        n_devices); the rows equal the single-device rows bit for bit (RE4)."""
        def check(rc):
            if rc != 0:
                raise TortoiseError(rc, (self.lib.ts_multi_last_error(self.h) or b"").decode())
        return _replay_ensemble(self.lib.ts_multi_mc_replay_ensemble, self.h, n_trials, n_real, r_first, trials, q_noise_scale,
                                want_x_final, check)


def _replay_ensemble(fn, h, n_trials, n_real, r_first, trials, q_noise_scale, want_x_final, check):
    n = int(n_trials)
    o = ReplayEnsembleOpts(int(n_real), int(r_first), float(q_noise_scale))
    sel = None if trials is None else np.ascontiguousarray(trials, dtype=np.int64).reshape(-1)
    ns = n if sel is None else sel.shape[0]
    R = max(int(n_real), 0)
    slew = np.zeros((ns, R))
    xf = np.zeros((ns, R, 8)) if want_x_final else None
    check(fn(h, n, C.byref(o), ns, None if sel is None else _ptr(sel), _ptr(slew), None if xf is None else _ptr(xf)))
    return slew, xf


# ---------------------------------------------------------------------------
# Reference-named free functions (scalar calls route to batch-of-1; correctness
# path, not the performance path).  A module-level default engine is created on
# first use.
_DEFAULT = None


def default_engine():
    global _DEFAULT
    if _DEFAULT is None:
        _DEFAULT = Engine(0)
    return _DEFAULT


def igrf12(date, r, lat, lon, show_warns=True):
    """igrf12(date, r, λ, Ω) -> [north, east, down] nT  (igrf.jl:67-274).
    Raises like the reference for date/lat/lon outside their ranges."""
    Bn, Be, Bd = default_engine().igrf12_batch(date, [r], [lat], [lon])
    return np.array([Bn[0], Be[0], Bd[0]])


class MagFieldMap:
    """What igrf_data returns in the reference: the n x n x 3 map (Tesla) behind a callable
    ``mag_field(i, j, c)`` with 1-based indices (monte_carlo.jl:90-96).  The reference wraps the
    array in a cubic B-spline interpolant with periodic extrapolation (magnetic_toolbox.jl:124-125)
    but only ever evaluates it at integer grid nodes, where an interpolating spline returns the
    data itself: this object returns the node values and wraps indices periodically (period n per
    axis, 3 for the component axis).  Non-integer arguments are rejected here; ``interpolant()``
    gives the spline itself, which takes fractional spatial indices."""

    def __init__(self, grid):
        self.grid = np.ascontiguousarray(grid, dtype=np.float64)

    def interpolant(self, engine=None):
        """The cubic B-spline of magnetic_toolbox.jl:124-125 over this map (FM1..FM4, DESIGN section 4, K8), prefiltered
        on the GPU and kept there."""
        return MagFieldInterpolant(self.grid, engine or default_engine())

    def __call__(self, i, j, c):
        for v in (i, j, c):
            if int(v) != v:
                raise ValueError("mag_field(i,j,c): only integer grid nodes are supported")
        n0, n1, n2 = self.grid.shape
        return float(self.grid[(int(i) - 1) % n0, (int(j) - 1) % n1, (int(c) - 1) % n2])

    def __array__(self, dtype=None, copy=None):
        return self.grid if dtype is None else self.grid.astype(dtype)

    @property
    def shape(self):
        return self.grid.shape

    def __getitem__(self, idx):
        return self.grid[idx]


class MagFieldInterpolant:
    """extrapolate(interpolate(A, BSpline(Cubic(Reflect(OnCell())))), Periodic()) of an n0 x n1 x 3 map
    (magnetic_toolbox.jl:124-125), rules FM1..FM4 of DESIGN section 4 (K8).  The coefficients stay on the GPU as a torch
    CUDA tensor (``coefs``, (n0+2) x (n1+2) x 3) and every evaluation runs through the device-pointer path.

    ``mag(i, j, c)``: real 1-based i, j (periodic, period n0 / n1), integer c (period 3; a fractional c is rejected,
    it would blend north, east and down) -> float.  ``mag.eval(i, j)``: arrays -> n x 3 (numpy for host inputs, a
    tensor for torch CUDA inputs).  A non-finite index raises TortoiseError."""

    def __init__(self, grid, engine):
        import torch
        self.engine = engine
        self.device = torch.device("cuda", engine.device)
        g = torch.as_tensor(np.ascontiguousarray(grid, dtype=np.float64)).to(self.device)
        self.coefs = engine.field_map_prefilter(g)
        self.shape = tuple(g.shape)

    def eval(self, i, j):
        import torch
        if _is_tensor(i):
            return self.engine.field_map_eval_batch(self.coefs, i, j)
        x0 = torch.as_tensor(_f64(np.atleast_1d(i)).reshape(-1)).to(self.device)
        x1 = torch.as_tensor(_f64(np.atleast_1d(j)).reshape(-1)).to(self.device)
        return self.engine.field_map_eval_batch(self.coefs, x0, x1).cpu().numpy()

    def __call__(self, i, j, c):
        if int(c) != c:
            raise ValueError("mag_field(i,j,c): the component index c must be an integer")
        return float(self.eval(float(i), float(j))[0, (int(c) - 1) % 3])


def igrf_data(altitude, year, n=1000):
    """igrf_data(altitude, year) (magnetic_toolbox.jl:108-127): the n x n x 3 lat/long map in Tesla
    (one K1 launch for the n^2 points) behind the reference's ``mag_field(i,j,c)`` call shape."""
    R_E = 6378
    lat = np.linspace(-np.pi / 2, np.pi / 2, n)
    lon = np.linspace(-np.pi, np.pi, n)
    LA, LO = np.meshgrid(lat, lon, indexing="ij")
    r = np.full(LA.size, (altitude + R_E) * 1000.0)
    Bn, Be, Bd = default_engine().igrf12_batch(year, r, LA.ravel(), LO.ravel())
    return MagFieldMap(np.stack([Bn, Be, Bd], axis=-1).reshape(n, n, 3) / 1.0e9)


class params:
    """struct params (input_parameters.jl:4-16)."""

    def __init__(self, type, mass, J, BC, alt, Kep, MJD, GM, R_E, T, w_0):
        self.type, self.mass, self.J, self.BC, self.alt = type, mass, J, BC, alt
        self.Kep, self.MJD, self.GM, self.R_E, self.T, self.w_0 = Kep, MJD, GM, R_E, T, w_0


def input_parameters(type, Kep, MJD):
    """input_parameters(type, Kep, MJD) (input_parameters.jl:24-66), including its
    quirks: alt forced to 400 (:58) and MJD forced to 58155.0 (:63)."""
    GM = GM_EARTH
    R_E = 6371.0
    if type == "1U":
        mass = .75
        J = np.diag([0.00125, 0.00125, 0.00125])
    elif type == "1P":
        mass = .25
        J = np.diag([0.0001041667, 0.0001041667, 0.0001041667])
    elif type == "3U":
        mass = 2.5
        J = np.diag([0.020833, 0.020833, 0.0041666])
    else:
        raise ValueError("Type not recognized")
    BC = mass / 2.2 / (J[0, 0] * J[1, 1])
    Kep = np.array(Kep, dtype=np.float64).reshape(-1)
    alt = 400.0
    T = 2 * np.pi * np.sqrt(Kep[1] ** 3 / GM)
    w_0 = np.sqrt(GM / Kep[1] ** 3)
    return params(type, mass, J, BC, alt, Kep, 58155.0, GM, R_E, T, w_0)


def magnetic_simulation(p, t0, tf, N, mag_field=None, alt=None, igrf_date=2019.0):
    """magnetic_simulation(p,t0,tf,N,mag_field) -> (B (2N x 3), pos (3 x 2N+1), vel)
    (magnetic_toolbox.jl:33-106).  `alt` stands for the reference's *global* alt used in
    the field radius (alt+R_E)*1000 (:81, quirk Q3); default p.alt."""
    alt = p.alt if alt is None else alt
    o = np.zeros(1, dtype=FIELD_OPTS_DTYPE)
    o[0] = (p.GM, p.MJD, igrf_date, (alt + p.R_E) * 1000.0, t0, tf, int(N))
    B, offs, pos, vel = default_engine().magnetic_simulation_batch(p.Kep.reshape(1, 6), o, want_pos=True)
    return B, pos.T.copy(), vel.T.copy()


def magnetic_gramian(B_N, dt):
    """magnetic_gramian(B_N,dt) -> 3 x 3 x rows (magnetic_toolbox.jl:1-12)."""
    B_N = _f64(B_N)
    G = default_engine().magnetic_gramian_batch(B_N, [0], [B_N.shape[0]], [dt])
    return np.transpose(G, (1, 2, 0)).copy()


def condition_based_time(B_gram, cutoff):
    """condition_based_time(B_gram,cutoff) (magnetic_toolbox.jl:14-31); B_gram 3 x 3 x rows."""
    G = np.ascontiguousarray(np.transpose(_f64(B_gram), (2, 0, 1)))
    return int(default_engine().condition_based_time_batch(G, [0], [G.shape[0]], [cutoff])[0])


def eigen_axis_slew(x0, xf, t):
    """eigen_axis_slew(x0,xf,t) -> (w_guess (nt x 3), q_guess (nt x 4))  (eigen_axis_slew.jl:1-38).
    t must be a uniform range t0:dt:t_end, as in the reference."""
    t = _f64(t)
    x0p = np.concatenate([np.asarray(x0, dtype=float)[:7], [0.0]])
    xfp = np.concatenate([np.asarray(xf, dtype=float)[:7], [0.0]])
    dt = float(t[1] - t[0])
    _, _, _, wg, qg, _ = default_engine().slew_weights_batch([x0p], [xfp], np.eye(3).reshape(1, 9), [float(t[-1])], t0=float(t[0]),
                                                            dt=dt, want_guess=True)
    return wg[:len(t)], qg[:len(t)]


def kep_ECI(kep_elements, t0, GM):
    """kep_ECI(kep,t0,GM) -> [r'; v'] (2 x 3)  (kep_ECI.jl:1-35); like the reference it also mutates
    kep_elements[5] (kep_ECI.jl:7-8)."""
    k = np.asarray(kep_elements, dtype=np.float64).reshape(-1)
    rv = default_engine().kep_eci_batch(k.reshape(1, 6), [t0], GM)[0]
    try:
        kep_elements[5] = np.fmod(k[5] + t0 * np.sqrt(GM / k[1] ** 3), 360.0)
    except Exception:
        pass
    return rv.reshape(2, 3)


def OrbitPlotter(x, p=None, t=None):
    """OrbitPlotter(x,p,t) -> [v; a]  (OrbitPlotter.jl:1-52)."""
    return default_engine().orbit_rhs_batch(np.asarray(x, dtype=float).reshape(1, 6))[0]


def legendre(phi, n_max, ph_term=False):
    """legendre(Val{:schmidt}, phi, n_max, false)  (legendre.jl:254-292)."""
    if ph_term:
        raise NotImplementedError("only ph_term = false is on the IGRF path (igrf.jl:124)")
    return default_engine().legendre_schmidt_batch([phi], n_max, want_dP=False)[0]


def dlegendre(phi, n_max, ph_term=False):
    """dlegendre(Val{:schmidt}, phi, n_max, false)  (dlegendre.jl:221-309, via :411-419)."""
    if ph_term:
        raise NotImplementedError("only ph_term = false is on the IGRF path (igrf.jl:125)")
    return default_engine().legendre_schmidt_batch([phi], n_max, want_dP=True)[1][0]


def attitude_dynamics(x, u, B_B, J):
    """attitude_dynamics(x,u,B_B,J) -> xdot (7)  (attitude_dynamics.jl:2-24)."""
    return default_engine().dynamics_batch(2, np.asarray(x, dtype=float).reshape(1, 7), np.asarray(u, dtype=float).reshape(1, 3),
                                           np.asarray(B_B, dtype=float).reshape(1, 3), J)[0]


def qmult(q1, q2):
    """qmult.jl:1-3 (host helper)."""
    q1, q2 = np.asarray(q1, dtype=float), np.asarray(q2, dtype=float)
    return np.concatenate([[q1[0] * q2[0] - q1[1:] @ q2[1:]], q1[0] * q2[1:] + q2[0] * q1[1:] + np.cross(q1[1:], q2[1:])])


def qrot(q, r):
    """qrot.jl:1-3 (host helper)."""
    q, r = np.asarray(q, dtype=float), np.asarray(r, dtype=float)
    return r + 2 * np.cross(q[1:], np.cross(q[1:], r) + q[0] * r)


def q_inv(q):
    """q_inv (attitude_controller.jl:164-166)."""
    q = np.asarray(q, dtype=float)
    return np.concatenate([[q[0]], -q[1:4]])


def hat(x):
    """hat (magnetic_toolbox.jl:142-146)."""
    x = np.asarray(x, dtype=float)
    return np.array([[0, -x[2], x[1]], [x[2], 0, -x[0]], [-x[1], x[0], 0]])


def DerivFunction(x, u, B_ECI, J, N, tf, t0=0.0):
    """DerivFunction(dx,x,u) (DerivFunction.jl:1-56) as a function: returns dx (8).  B_ECI, J, N, tf, t0 are
    the globals the reference's version reads (field row floor(x[8]*N+1), clock rate 1/(tf-t0), u*1e-2)."""
    return default_engine().dynamics_batch(0, np.asarray(x, dtype=float).reshape(1, 8), np.asarray(u, dtype=float).reshape(1, 3),
                                           B_ECI, J, index_scale=float(N), clock_rate=1.0 / (tf - t0))[0]


def gain_simulator(x, u, B_ECI, J, N, tf, t0=0.0):
    """gain_simulator(dx,x,u) (gain_simulator.jl:1-53) as a function: the noise-free simulator (u/100)."""
    return default_engine().dynamics_batch(1, np.asarray(x, dtype=float).reshape(1, 8), np.asarray(u, dtype=float).reshape(1, 3),
                                           B_ECI, J, index_scale=float(N), clock_rate=1.0 / (tf - t0))[0]


def bryson_weights(x0, xf, J, t_final, t0=0.0, dt=0.2, alpha=10.0, beta=1e3):
    """Bryson-rule LQR weights from the eigen-axis guess (TortoiseSat.jl:157-168): returns (Q, R, Qf) 8x8, 3x3, 8x8."""
    Qd, Qfd, Rd = default_engine().slew_weights_batch(np.asarray(x0, dtype=float).reshape(1, 8), np.asarray(xf, dtype=float).reshape(1, 8),
                                                      np.asarray(J, dtype=float).reshape(1, 9), [t_final], t0=t0, dt=dt, alpha=alpha,
                                                      beta=beta)
    return np.diag(Qd[0]), np.diag(Rd[0]), np.diag(Qfd[0])


def solve_slew(x0, xf, J, Q, R, Qf, B_ECI, N, dt, N_field=None, tf_scope=5400.0, t0=0.0, U0=None, opts=None):
    """The TrajectoryOptimization.jl block of TortoiseSat.jl:145-146,169,178-199 for ONE slew (batch of 1):
    rk3(Model(DerivFunction,8,3)), LQRObjective(Q,R,Qf,xf,N), BoundConstraint(u in [-1,1]), goal_constraint(xf),
    AugmentedLagrangianSolver, solve!.  B_ECI (rows x 3) is the field table the reference keeps in a global; N_field and
    tf_scope are the globals N and tf that DerivFunction reads.  Returns X (8 x N), U (3 x N-1), K (3 x 8 x N-1) in the
    reference's column-per-knot shapes, and the outcome record."""
    B = np.ascontiguousarray(B_ECI, dtype=float).reshape(-1, 3)
    N = int(N)
    X, U, K, out, offs = default_engine().alilqr_solve_batch(
        [N], np.asarray(x0, dtype=float).reshape(1, 8), np.asarray(xf, dtype=float).reshape(1, 8),
        np.asarray(J, dtype=float).reshape(1, 9), np.diag(np.asarray(Q, dtype=float)).reshape(1, 8),
        np.diag(np.asarray(Qf, dtype=float)).reshape(1, 8), np.diag(np.asarray(R, dtype=float)).reshape(1, 3), B, [0], [B.shape[0]],
        [float(N if N_field is None else N_field)], [1.0 / (tf_scope - t0)], dt, U0=U0, opts=opts, want_K=True)
    return X.T.copy(), U[:N - 1].T.copy(), np.transpose(K[:N - 1], (1, 2, 0)).copy(), out[0]


def attitude_simulation(f, f_gains, integration, X_lqr, U_lqr, dt_lqr, x0_lqr, t0, tf, Q_lqr, R_lqr, Qf_lqr, *, B_ECI, J,
                        N_field=None, tf_scope=5400.0, noise_mode=2, seed=0, q_final=(1.0, 0.0, 0.0, 0.0)):
    """attitude_simulation(f!,f_gains!,integration,X_lqr,U_lqr,dt_lqr,x0_lqr,t0,tf,Q_lqr,R_lqr,Qf_lqr) -> (X_sim,U_sim,dX,K)
    (attitude_controller.jl:1-48).  f, f_gains and integration are accepted for signature compatibility: the library
    implements simulator / gain_simulator / rk4 (simulator.jl, gain_simulator.jl, attitude_controller.jl:122-145).
    X_lqr is 8 x N, U_lqr 3 x (N-1) as in the reference; the noise is Philox(seed) instead of Julia's global RNG."""
    X_lqr = np.asarray(X_lqr, dtype=float)
    N = X_lqr.shape[1]
    o = default_tvlqr_opts()
    o.dt, o.t0, o.noise_mode, o.seed = float(dt_lqr), float(t0), int(noise_mode), int(seed)
    for i in range(6):
        o.Qd[i], o.Qfd[i] = float(np.asarray(Q_lqr)[i, i]), float(np.asarray(Qf_lqr)[i, i])
    for i in range(3):
        o.Rd[i] = float(np.asarray(R_lqr)[i, i])
    Up = np.zeros((N, 3))
    Ul = np.asarray(U_lqr, dtype=float)
    Up[:Ul.shape[1]] = Ul.T
    B = np.ascontiguousarray(B_ECI, dtype=float).reshape(-1, 3)
    Xs, Us, dX, K, nsim, slew, offs = default_engine().tvlqr_sim_batch(
        [N], X_lqr.T.copy(), Up, np.asarray(x0_lqr, dtype=float).reshape(1, 8), np.asarray(J, dtype=float).reshape(1, 9), B, [0],
        [B.shape[0]], [float(N if N_field is None else N_field)], [1.0 / (tf_scope - t0)], [float(tf)], np.asarray(q_final, dtype=float),
        opts=o)
    n = int(nsim[0])
    return Xs[:n].T.copy(), Us[:n].T.copy(), dX[:n].T.copy(), np.transpose(K[:N - 1], (1, 2, 0)).copy()


def monte_carlo(number_sims=100, alt=400.0, R_E=6371.0, inclination=96.6, MJD_0=58155.0, igrf_date=2019.0, t0=0.0, tf=60 * 40.0,
                cutoff=30.0, N=5000, J=None, q_0=None, q_final=(np.sqrt(2) / 2, np.sqrt(2) / 2, 0.0, 0.0), alpha=1.0e-1, beta=1.0e3,
                seed=0, run_tvlqr=True, ilqr=None, rng=None, random_attitudes=False, trajectories=True, eigen_axis_fix=False,
                sat_att=False, resumable=False):
    """The loop of monte_carlo.jl:118-262 (solver block of TortoiseSat.jl:178-199) for number_sims trials in ONE
    library call.  Returns the arrays the script leaves in globals (monte_carlo.jl:52-66,237-240): A (number_sims x 6),
    t_final, slew_time, fails, and -- with trajectories=True -- the per-trial lists `states` (8 x N_i), `control_inputs`
    (3 x N_i-1), `sim_states` (8 x N_sim_i), `sim_control_inputs` (3 x N_sim_i), `B_ECI_total` (2N_i x 3), `t_total`, plus
    the outcome records and the statistics block.  Randomisation as in monte_carlo.jl:122-127,207 (RAAN and anomaly
    uniform in [0,360); q_0 = [1,0,0,0] for every trial as at monte_carlo.jl:108-111 unless random_attitudes=True, which
    draws q_0 uniformly on S^3 -- the BASELINE configs[2] ensemble; initial attitude noise randn(3)*(pi/180)^2), from
    numpy's generator instead of Julia's global RNG.  sat_att=True selects the quaternion-aware solver the script asks of
    its forked TrajectoryOptimization (monte_carlo.jl:158 Model(DerivFunction, n, m, quaternion_error,
    quaternion_expansion), :192 solver.opts.sat_att = true): ts_ilqr_opts.quat_error.  resumable=True keeps the solver
    state on the default engine (keep_trajectories = 2) so that continue_monte_carlo can give the max-outer trials more
    outer iterations; the result then also holds the run's solver options as `ilqr`."""
    rng = np.random.default_rng(seed) if rng is None else rng
    n = int(number_sims)
    J = np.diag([0.00125, 0.00125, 0.00125]) if J is None else np.asarray(J, dtype=float)
    A = np.zeros((n, 6))
    alt_i = np.broadcast_to(np.asarray(alt, dtype=float), (n,))          # scalars as in monte_carlo.jl, or one value per trial
    A[:, 1], A[:, 2] = alt_i + R_E, np.broadcast_to(np.asarray(inclination, dtype=float), (n,))
    A[:, 3], A[:, 5] = rng.random(n) * 360, rng.random(n) * 360
    fo = np.zeros(n, dtype=FIELD_OPTS_DTYPE)
    for i in range(n):
        fo[i] = (GM_EARTH, MJD_0, igrf_date, (alt_i[i] + R_E) * 1000.0, 0.0, 0.0, 0)
    x0, xf = np.zeros((n, 8)), np.zeros((n, 8))
    if random_attitudes:
        q = rng.normal(size=(n, 4))
        x0[:, 3:7] = q / np.linalg.norm(q, axis=1, keepdims=True)
    else:
        x0[:, 3:7] = np.asarray((1.0, 0.0, 0.0, 0.0) if q_0 is None else q_0, dtype=float)
    xf[:, 3:7], xf[:, 7] = np.asarray(q_final, dtype=float), 1.0
    qn = rng.normal(size=(n, 3)) * (np.pi / 180) ** 2
    cfg = default_mc_config(n, shared_orbit=False, run_tvlqr=run_tvlqr, t0=t0, tf=tf, N_scope=int(N), cutoff=cutoff, dt=0.2,
                            alpha=alpha, beta=beta)
    if ilqr is not None:
        cfg.ilqr = ilqr
    if sat_att:
        cfg.ilqr.quat_error = 1
    cfg.tvlqr.noise_mode, cfg.tvlqr.seed = 2, int(seed)
    for i in range(6):                                   # monte_carlo.jl:69-71,216-226
        cfg.tvlqr.Qd[i], cfg.tvlqr.Qfd[i] = 10.0, 1000.0
    for i in range(3):
        cfg.tvlqr.Rd[i] = 0.5e3
    cfg.eigen_axis_fix, cfg.keep_trajectories = int(bool(eigen_axis_fix)), 2 if resumable else int(bool(trajectories))
    eng = default_engine()
    out, st = eng.monte_carlo_run(cfg, A, fo, x0, xf, np.tile(J.reshape(-1), (n, 1)), q_noise0=qn)
    fails = (out["slew_time"] == out["t_final"]).astype(float)     # monte_carlo.jl:257-261
    res = dict(A=A, t_final=out["t_final"].copy(), slew_time=out["slew_time"].copy(), fails=fails, outcomes=out, stats=st)
    if resumable:
        res["ilqr"] = IlqrOpts.from_buffer_copy(cfg.ilqr)
    if trajectories:
        tr = eng.mc_trajectories(n, want=("X", "U", "X_sim", "U_sim", "B_eci") if run_tvlqr else ("X", "U", "B_eci"))
        ko, ro = tr["knot_offs"], tr["row_offs"]
        sl = lambda a, t, last=0: a[ko[t]:ko[t + 1] - last].T.copy()
        res["states"] = [sl(tr["X"], t) for t in range(n)]                       # monte_carlo.jl:200
        res["control_inputs"] = [sl(tr["U"], t, 1) for t in range(n)]            # :201
        res["B_ECI_total"] = [tr["B_eci"][ro[t]:ro[t] + 2 * (ko[t + 1] - ko[t])].copy() for t in range(n)]   # :149
        res["t_total"] = [t0 + 0.2 * np.arange(ko[t + 1] - ko[t] + 1) for t in range(n)]                      # :144
        if run_tvlqr:
            res["sim_states"] = [sl(tr["X_sim"], t) for t in range(n)]           # :232
            res["sim_control_inputs"] = [sl(tr["U_sim"], t) for t in range(n)]   # :233
    return res


def continue_monte_carlo(res, max_outer=30, ilqr=None):
    """Gives the trials of a monte_carlo(..., resumable=True) result that ended at max_outer more outer iterations, up to
    `max_outer` in all (ts_mc_continue on the default engine, which must not have run another Monte-Carlo call since),
    and updates `res` in place as retry_failed does: outcomes, slew_time, fails (monte_carlo.jl:257-261) and the trajectory
    lists of the continued trials.  `ilqr` (default: the run's options) supplies the other solver options.  Returns the
    0-based indices of the continued trials."""
    if "ilqr" not in res:
        raise ValueError("continue_monte_carlo needs a monte_carlo(..., resumable=True) result")
    o = IlqrOpts.from_buffer_copy(res["ilqr"] if ilqr is None else ilqr)
    o.max_outer = int(max_outer)
    prev = res["outcomes"]
    n = prev.shape[0]
    idx = np.nonzero((prev["status"] == 1) & (prev["outer_iters"] < o.max_outer))[0]   # MC1
    eng = default_engine()
    out, st = eng.mc_continue(n, o)
    res["outcomes"], res["stats"], res["ilqr"] = out, st, o
    res["slew_time"] = out["slew_time"].copy()
    res["fails"] = (out["slew_time"] == out["t_final"]).astype(float)
    if idx.size and "states" in res:
        run_tvlqr = "sim_states" in res
        tr = eng.mc_trajectories(n, want=("X", "U", "X_sim", "U_sim") if run_tvlqr else ("X", "U"))
        ko = tr["knot_offs"]
        sl = lambda a, t, last=0: a[ko[t]:ko[t + 1] - last].T.copy()
        for t in idx:
            res["states"][t] = sl(tr["X"], t)
            res["control_inputs"][t] = sl(tr["U"], t, 1)
            if run_tvlqr:
                res["sim_states"][t] = sl(tr["X_sim"], t)
                res["sim_control_inputs"][t] = sl(tr["U_sim"], t)
    return idx


def replay_ensemble(res, n_real=100, trials=None, r_first=0, q_noise_scale=Q_NOISE_SCALE):
    """The slew-time distribution of the optimised slews of a monte_carlo() result under the simulator's disturbances:
    every selected trial (None = all) replayed n_real times with independent draws (ts_mc_replay_ensemble on the default
    engine, which must not have run another Monte-Carlo call since; the result must come from monte_carlo with
    trajectories=True, the default, or resumable=True).  Realisation 0 repeats the run's own replay (RE3).  Returns a dict:
    slew_time (n_sel, n_real), fails (slew_time == t_final, monte_carlo.jl:257-261), fail_rate (n_sel: the share of failing
    draws), slew_mean / slew_std (n_sel: over the non-failing draws, NaN if none) and trials (the selected indices).  A
    NO_CUTOFF trial has NaN slew times, no fails and a NaN fail_rate."""
    if "states" not in res and "ilqr" not in res:
        raise ValueError("replay_ensemble needs a monte_carlo(..., trajectories=True) or monte_carlo(..., resumable=True) result")
    out = res["outcomes"]
    n = out.shape[0]
    sel = np.arange(n, dtype=np.int64) if trials is None else np.ascontiguousarray(trials, dtype=np.int64).reshape(-1)
    slew, _ = default_engine().mc_replay_ensemble(n, n_real, r_first=r_first, trials=sel, q_noise_scale=q_noise_scale)
    tf = out["t_final"][sel][:, None]
    fails = slew == tf
    valid = ~np.isnan(slew)
    ok = valid & ~fails
    with np.errstate(invalid="ignore", divide="ignore"):
        nv = valid.sum(axis=1)
        fail_rate = np.where(nv > 0, fails.sum(axis=1) / np.maximum(nv, 1), np.nan)
        k = ok.sum(axis=1)
        s = np.where(ok, slew, 0.0)
        mean = np.where(k > 0, s.sum(axis=1) / np.maximum(k, 1), np.nan)
        var = np.where(k > 0, (np.where(ok, slew - mean[:, None], 0.0) ** 2).sum(axis=1) / np.maximum(k, 1), np.nan)
    return dict(slew_time=slew, fails=fails, fail_rate=fail_rate, slew_mean=mean, slew_std=np.sqrt(var), trials=sel)


# ---------------------------------------------------------------------------
# Result persistence + retry of failed trials (SURVEY 8f row 3; monte_carlo.jl:269,334-343, heatmap.jl:114-123)
def save_monte_carlo(res, directory, prefix="100"):
    """Writes the result of monte_carlo() in the layout of monte_carlo.jl:334-343: one container per array and per trial,
    `<prefix>_A`, `<prefix>_states_<i>` (datasets `one_state`, `states` = sim_states[i], as the script writes them),
    `<prefix>_control_<i>` (`control` = sim_control_inputs[i]), `<prefix>_B_N_<i>` (`B_ECI`), `<prefix>_t_total_<i>`
    (`t_total`), i = 1..number_sims.  The reference uses HDF5 (`h5write`); this image has no HDF5 library, so each container
    is a NumPy .npz archive holding the SAME dataset names (np.load(path)["states"] replaces h5read(path, "states")).
    A `<prefix>_summary` container adds what the script keeps in globals: t_final, slew_time, fails, retry, outcomes."""
    import os
    os.makedirs(directory, exist_ok=True)
    p = lambda name: os.path.join(directory, "%s_%s.npz" % (prefix, name))
    n = res["A"].shape[0]
    np.savez(p("A"), A=res["A"])
    for i in range(n):
        if "sim_states" in res:
            np.savez(p("states_%d" % (i + 1)), one_state=res["sim_states"][i], states=res["sim_states"][i])
            np.savez(p("control_%d" % (i + 1)), control=res["sim_control_inputs"][i])
        if "B_ECI_total" in res:
            np.savez(p("B_N_%d" % (i + 1)), B_ECI=res["B_ECI_total"][i])
            np.savez(p("t_total_%d" % (i + 1)), t_total=res["t_total"][i])
    retry = np.nonzero(res["fails"] == 1.0)[0] + 1                      # monte_carlo.jl:269 (1-based, like findall)
    np.savez(p("summary"), t_final=res["t_final"], slew_time=res["slew_time"], fails=res["fails"], retry=retry,
             outcomes=res["outcomes"])
    return retry


def load_monte_carlo(directory, prefix="100"):
    """Inverse of save_monte_carlo: the arrays a resumed script needs (A, t_final, slew_time, fails, retry, and the
    per-trial lists when they were written)."""
    import os
    p = lambda name: os.path.join(directory, "%s_%s.npz" % (prefix, name))
    s = np.load(p("summary"))
    res = dict(A=np.load(p("A"))["A"], t_final=s["t_final"], slew_time=s["slew_time"], fails=s["fails"], retry=s["retry"],
               outcomes=s["outcomes"])
    n = res["A"].shape[0]
    if os.path.exists(p("states_1")):
        res["sim_states"] = [np.load(p("states_%d" % (i + 1)))["states"] for i in range(n)]
        res["sim_control_inputs"] = [np.load(p("control_%d" % (i + 1)))["control"] for i in range(n)]
    if os.path.exists(p("B_N_1")):
        res["B_ECI_total"] = [np.load(p("B_N_%d" % (i + 1)))["B_ECI"] for i in range(n)]
        res["t_total"] = [np.load(p("t_total_%d" % (i + 1)))["t_total"] for i in range(n)]
    return res


def retry_failed(res, max_rounds=3, inclination=None, seed=1, **mc_kwargs):
    """Re-runs the trials listed in `retry` (fails == 1) with fresh orbit draws, as paper_images/heatmap.jl:114-123 does
    (`for i in retry`: new RAAN and anomaly, and -- when `inclination` is None, the heat-map variant -- a new inclination
    rand*90, for those rows of A only), merging the new outcomes into `res` in place.  One library call per round; stops
    when nothing fails.  Returns the 1-based indices still failing."""
    rng = np.random.default_rng(seed)
    for _ in range(max_rounds):
        retry = np.nonzero(res["fails"] == 1.0)[0]
        if retry.size == 0:
            break
        inc = rng.random(retry.size) * 90 if inclination is None else inclination          # heatmap.jl:120
        sub = monte_carlo(number_sims=retry.size, rng=rng, inclination=inc, **mc_kwargs)
        for k, i in enumerate(retry):
            res["A"][i] = sub["A"][k]
            for f in ("t_final", "slew_time", "fails"):
                res[f][i] = sub[f][k]
            res["outcomes"][i] = sub["outcomes"][k]
            for f in ("states", "control_inputs", "sim_states", "sim_control_inputs", "B_ECI_total", "t_total"):
                if f in res and f in sub:
                    res[f][i] = sub[f][k]
    return np.nonzero(res["fails"] == 1.0)[0] + 1


# ---------------------------------------------------------------------------
# Comparison controller (SURVEY 8f row 4; src/comparison/psiaki_dynamics.jl, psiaki2005.jl, attitude_dynamics.jl:26-48)
def attitude_dynamics_linear(x, u, x_linear, B_B, J):
    """attitude_dynamics_linear(x,u,x_linear,B_B,J) -> xdot (7)  (attitude_dynamics.jl:26-48)."""
    return default_engine().attitude_dynamics_linear_batch(np.asarray(x, dtype=float).reshape(1, 7), np.asarray(u, dtype=float).reshape(1, 3),
                                                           np.asarray(x_linear, dtype=float).reshape(1, 7),
                                                           np.asarray(B_B, dtype=float).reshape(1, 3), J)[0]


def psiaki_controller(C_1, C_2, J, q, w_bar, B_meas, m_limit=None):
    """psiaki_controller (comparison/psiaki_dynamics.jl:1-26; host helper -- the batched loop evaluates it on the GPU).  The
    m_limit clamp is commented out in the reference and is not applied."""
    q, w_bar, B_meas = np.asarray(q, dtype=float), np.asarray(w_bar, dtype=float), np.asarray(B_meas, dtype=float)
    T_req = -(C_1 * w_bar + C_2 * np.linalg.inv(np.asarray(J, dtype=float)) @ q[1:4])
    return np.cross(B_meas, T_req) / (np.linalg.norm(B_meas) ** 2)


def psiaki_pd_simulation(x0, w_guess, q_guess, B_ECI, J, dt, C_1=1e-6, C_2=1e-9):
    """The closed loop of comparison/psiaki2005.jl:116-164 for ONE slew (batch of 1): w_guess 3 x N, q_guess 4 x N, B_ECI
    3 x N as in the script.  Returns x (7 x N), the moments (3 x N) and the error quaternions q_bar (4 x N)."""
    w_guess, q_guess, B_ECI = np.asarray(w_guess, dtype=float), np.asarray(q_guess, dtype=float), np.asarray(B_ECI, dtype=float)
    N = w_guess.shape[1]
    X, M, Qe, _ = default_engine().psiaki_pd_batch([N], np.asarray(x0, dtype=float).reshape(1, 7), w_guess.T.copy(), q_guess.T.copy(),
                                                   B_ECI.T.copy(), np.asarray(J, dtype=float).reshape(1, 9), dt, C_1, C_2)
    return X.T.copy(), M.T.copy(), Qe.T.copy()
