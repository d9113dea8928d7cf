"""carnd-mpc-project_b200 -- B200-native batched nonlinear-MPC solve (host-side Python binding).

The product is ``libmpc_b200.so`` (C-ABI in ``include/mpc_b200.h`` over hand-written sm_100a
kernels in ``csrc/``).  This module is a thin ctypes view of that C-ABI for tests, ``bench.py`` and
multi-GPU orchestration; PyTorch is used only for device memory, streams and torch.distributed.

There is NO CPU fallback: importing works without a GPU (so the symbol table can be checked), but
every compute call raises ``MpcError`` unless the CUDA library loaded and a device is present.

Boundary mirrored: ``MPC::solve`` (/root/reference/src/control/MPC.cpp:183-325) and ``Config::load``
(/root/reference/src/utils/Config.cpp:31-87).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MPC_B200_LIB") or os.path.join(_HERE, "libmpc_b200.so")   # override: A/B builds of the kernels
CSRC = os.path.join(_HERE, "csrc")

NCOEF, NTAB, NWEIGHTS, NMAX = 5, 16, 12, 64
KERNEL_AUTO, KERNEL_LANE, KERNEL_COOP = 0, 2, 3
LANE_MIN_BATCH = 9216

STATUS_SUCCESS = 1
STATUS_NAMES = {0: "not_defined", 1: "success", 2: "maxiter_exceeded", 3: "stop_at_tiny_step",
                4: "stop_at_acceptable_point", 5: "local_infeasibility", 9: "restoration_failure",
                10: "error_in_step_computation", 11: "invalid_number_detected", 13: "internal_error"}

EXPORTS = ["mpc_config_defaults", "mpc_config_load_json", "mpc_config_parse_json", "mpc_create",
           "mpc_destroy", "mpc_set_config", "mpc_solve_batch", "mpc_solve_batch_host", "mpc_solve_one",
           "mpc_launch_count", "mpc_last_error", "mpc_version", "mpc_measure_fp64_peak", "mpc_set_kernel",
           "mpc_run_prepare", "mpc_run_finish", "mpc_compute_throttle", "mpc_vehicle_move", "mpc_run_batch",
           "mpc_rollout", "mpc_set_handoff", "mpc_set_tail", "mpc_tail_counts", "mpc_measure_solve_latency", "mpc_set_dual_outputs", "mpc_config_from_cli",
           "mpc_telemetry_parse", "mpc_telemetry_step", "mpc_create_multi", "mpc_destroy_multi", "mpc_multi_device_count",
           "mpc_multi_handle", "mpc_solve_batch_multi", "mpc_set_rollout_mode", "mpc_set_warm_start", "mpc_warm_start_shift",
           "mpc_set_warm_start_one", "mpc_solution_sensitivity"]


class MpcError(RuntimeError):
    pass


class MpcConfig(C.Structure):
    """``mpc_config`` of include/mpc_b200.h (field order must match)."""
    _fields_ = [
        ("N", C.c_int), ("n_steers", C.c_int), ("n_steer_speeds", C.c_int), ("max_iter", C.c_int),
        ("dt", C.c_double), ("Lf", C.c_double), ("cte_panic", C.c_double), ("epsi_panic", C.c_double),
        ("max_speed", C.c_double), ("max_steering", C.c_double), ("max_accel", C.c_double),
        ("max_decel", C.c_double), ("weights", C.c_double * NWEIGHTS), ("steers", C.c_double * NTAB),
        ("steer_speeds", C.c_double * NTAB), ("tol", C.c_double),
        ("watchdog_trigger", C.c_int), ("filter_reset_trigger", C.c_int), ("tiny_step_tol", C.c_double),
        ("max_fit_order", C.c_int), ("latency_ms", C.c_int), ("max_fit_error", C.c_double),
        ("lookahead", C.c_double), ("ipopt_timeout", C.c_double), ("steer_adjust_thresh", C.c_double),
        ("steer_adjust_ratio", C.c_double), ("n_yaw_changes", C.c_int), ("n_yaw_change_speeds", C.c_int),
        ("yaw_changes", C.c_double * NTAB), ("yaw_change_speeds", C.c_double * NTAB),
    ]

    def as_dict(self):
        """Same keys as oracle.pyoracle.load_config_dict (SI units)."""
        return {
            "N": self.N, "dt": self.dt, "Lf": self.Lf, "cte_panic": self.cte_panic,
            "epsi_panic": self.epsi_panic, "max_speed": self.max_speed, "max_steering": self.max_steering,
            "max_accel": self.max_accel, "max_decel": self.max_decel, "weights": list(self.weights),
            "steers": list(self.steers[: self.n_steers]),
            "steer_speeds": list(self.steer_speeds[: self.n_steer_speeds]),
            "max_fit_order": self.max_fit_order, "max_fit_error": self.max_fit_error,
            "latency": self.latency_ms, "lookahead": self.lookahead, "ipopt_timeout": self.ipopt_timeout,
            "steer_adjust_thresh": self.steer_adjust_thresh, "steer_adjust_ratio": self.steer_adjust_ratio,
            "yaw_changes": list(self.yaw_changes[: self.n_yaw_changes]),
            "yaw_change_speeds": list(self.yaw_change_speeds[: self.n_yaw_change_speeds]),
        }


class MpcTelemetry(C.Structure):
    """``mpc_telemetry`` of include/mpc_b200.h."""
    _fields_ = [("kind", C.c_int), ("npts", C.c_int), ("x", C.c_double), ("y", C.c_double), ("psi", C.c_double),
                ("speed_mph", C.c_double), ("steering_angle", C.c_double), ("ptsx", C.c_double * 16), ("ptsy", C.c_double * 16)]


class MpcRunAux(C.Structure):
    """``mpc_run_aux`` of include/mpc_b200.h."""
    _fields_ = [("max_yaw_change", C.c_double), ("max_speed", C.c_double), ("target_speed", C.c_double),
                ("fit_error", C.c_double), ("fit_order", C.c_int)]


def build(verbose=False):
    """Compile csrc/ for sm_100a with nvcc into libmpc_b200.so (in-tree)."""
    out = subprocess.run(["make", "-C", CSRC], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode != 0:
        raise MpcError("nvcc build of libmpc_b200.so failed")
    return LIB_PATH


_lib = None


def lib():
    """Load the C-ABI library; raises loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MpcError("libmpc_b200.so is missing (%s): run __graft_entry__.build() -- there is no "
                       "CPU fallback for the MPC solve" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    dp, ip, vp = C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_void_p
    cfgp = C.POINTER(MpcConfig)
    L.mpc_config_defaults.argtypes = [cfgp]
    L.mpc_config_load_json.argtypes = [C.c_char_p, cfgp]
    L.mpc_config_parse_json.argtypes = [C.c_char_p, cfgp]
    L.mpc_config_from_cli.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.c_char_p, cfgp, C.c_char_p, C.c_int]
    L.mpc_create.argtypes = [cfgp, C.c_int, C.POINTER(vp)]
    L.mpc_destroy.argtypes = [vp]
    L.mpc_destroy.restype = None
    L.mpc_set_config.argtypes = [vp, cfgp]
    L.mpc_set_kernel.argtypes = [vp, C.c_int, C.c_int, C.c_int]
    L.mpc_set_handoff.argtypes = [vp, C.c_int]
    L.mpc_set_rollout_mode.argtypes = [vp, C.c_int]
    L.mpc_set_tail.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int]
    L.mpc_tail_counts.argtypes = [vp, C.POINTER(C.c_int), C.c_int]
    L.mpc_measure_solve_latency.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.mpc_set_dual_outputs.argtypes = [vp, vp, vp, vp]
    L.mpc_set_warm_start.argtypes = [vp, vp, vp, vp, vp, C.c_double]
    L.mpc_set_warm_start_one.argtypes = [vp, C.c_int, C.c_double]
    L.mpc_warm_start_shift.argtypes = [vp, C.c_int] + [vp] * 8 + [vp]
    L.mpc_solution_sensitivity.argtypes = [vp, C.c_int] + [vp] * 13 + [vp]
    L.mpc_telemetry_parse.argtypes = [C.c_char_p, C.POINTER(MpcTelemetry)]
    L.mpc_telemetry_step.argtypes = [vp, C.c_char_p, dp, C.c_double, C.c_int, C.c_char_p, C.c_int]
    L.mpc_solve_batch.argtypes = [vp, C.c_int] + [vp] * 13 + [vp]
    L.mpc_solve_batch_host.argtypes = [vp, C.c_int] + [vp] * 13
    L.mpc_solve_one.argtypes = [vp, dp, dp, C.c_double, C.c_double, dp, dp, dp, ip, ip]
    L.mpc_create_multi.argtypes = [cfgp, ip, C.c_int, C.POINTER(vp)]
    L.mpc_destroy_multi.argtypes = [vp]
    L.mpc_destroy_multi.restype = None
    L.mpc_multi_device_count.argtypes = [vp]
    L.mpc_multi_handle.argtypes = [vp, C.c_int]
    L.mpc_multi_handle.restype = vp
    L.mpc_solve_batch_multi.argtypes = [vp, C.c_int] + [vp] * 13
    L.mpc_measure_fp64_peak.argtypes = [C.c_int, dp]
    L.mpc_run_prepare.argtypes = [cfgp, dp, C.c_double, dp, dp, C.c_int, dp, dp, dp, dp, C.POINTER(MpcRunAux)]
    L.mpc_run_finish.argtypes = [cfgp, C.POINTER(MpcRunAux), C.c_double, dp, dp]
    L.mpc_compute_throttle.argtypes = [cfgp, C.c_double, C.c_double]
    L.mpc_compute_throttle.restype = C.c_double
    L.mpc_vehicle_move.argtypes = [dp, C.c_double, C.c_double, C.c_double, C.c_double]
    L.mpc_vehicle_move.restype = None
    L.mpc_run_batch.argtypes = [vp, C.c_int, vp, vp, vp, vp, C.c_int] + [vp] * 8 + [vp]
    L.mpc_rollout.argtypes = [vp, C.c_int, C.c_int, vp, vp, C.c_int, vp, vp, vp, C.c_double, C.c_double, vp, vp]
    L.mpc_launch_count.argtypes = [vp]
    L.mpc_launch_count.restype = C.c_longlong
    L.mpc_last_error.restype = C.c_char_p
    L.mpc_version.restype = C.c_char_p
    _lib = L
    return L


def _check(rc, what):
    if rc != 0:
        names = {-1: "MPC_EINVAL", -2: "MPC_ENODEV", -3: "MPC_ECUDA", -4: "MPC_ENOMEM", -5: "MPC_EIO",
                 -6: "MPC_EPARSE"}
        raise MpcError("%s failed: %s (%d) %s" % (what, names.get(rc, "?"), rc,
                                                  lib().mpc_last_error().decode()))


class MultiSolver:
    """``mpc_create_multi`` / ``mpc_solve_batch_multi``: the C-ABI's own multi-GPU path (one host thread, one handle
    and stream per device, contiguous shards).  bench.py's --gpus N uses one process per GPU instead; this class exists
    for the tests and for the bench's report of what a C++ caller gets."""

    def __init__(self, cfg, devices):
        self.cfg = cfg
        self._m = C.c_void_p()
        dev = (C.c_int * len(devices))(*devices)
        _check(lib().mpc_create_multi(C.byref(cfg), dev, len(devices), C.byref(self._m)), "mpc_create_multi")

    def close(self):
        if self._m:
            lib().mpc_destroy_multi(self._m)
            self._m = C.c_void_p()

    @property
    def n_devices(self):
        return lib().mpc_multi_device_count(self._m)

    def solve_raw(self, B, state, coeffs, yaw_lo, yaw_hi, result, traj_x=None, traj_y=None, full=None, status=None,
                  iters=None, weights=None, N_per=None, dt_per=None):
        """Host arrays in the C layout ([k][B], batch index fastest); pinned memory lets the devices' copies overlap."""
        _check(lib().mpc_solve_batch_multi(self._m, B, _ptr(state), _ptr(coeffs), _ptr(yaw_lo), _ptr(yaw_hi), _ptr(weights),
                                           _ptr(N_per), _ptr(dt_per), _ptr(result), _ptr(traj_x), _ptr(traj_y), _ptr(full),
                                           _ptr(status), _ptr(iters)), "mpc_solve_batch_multi")

    def set_warm_start(self, g, x0=None, lam0=None, zl0=None, zu0=None, mu_init=0.0):
        """Warm start of shard g (problems [g*B/G, (g+1)*B/G)): device tensors on that shard's device, see
        Solver.set_warm_start."""
        self._warm = getattr(self, "_warm", {})
        self._warm[g] = (x0, lam0, zl0, zu0)   # keep them alive
        h = lib().mpc_multi_handle(self._m, int(g))
        _check(lib().mpc_set_warm_start(h, _ptr(x0), _ptr(lam0), _ptr(zl0), _ptr(zu0), float(mu_init)),
               "mpc_set_warm_start")

    def solve_batch_host(self, state, coeffs, yaw_lo, yaw_hi, weights=None, N_per=None, dt_per=None, want_full=False):
        B, N = state.shape[0], self.cfg.N
        st = np.ascontiguousarray(np.asarray(state, dtype=np.float64).T)
        co = np.ascontiguousarray(np.asarray(coeffs, dtype=np.float64).T)
        yl = np.ascontiguousarray(yaw_lo, dtype=np.float64)
        yh = np.ascontiguousarray(yaw_hi, dtype=np.float64)
        w = None if weights is None else np.ascontiguousarray(np.asarray(weights, dtype=np.float64).T)
        npp = None if N_per is None else np.ascontiguousarray(N_per, dtype=np.int32)
        dtp = None if dt_per is None else np.ascontiguousarray(dt_per, dtype=np.float64)
        res, tx, ty = np.zeros((9, B)), np.zeros((N, B)), np.zeros((N, B))
        full = np.zeros((8 * N - 2, B)) if want_full else None
        status, iters = np.zeros(B, dtype=np.int32), np.zeros(B, dtype=np.int32)
        self.solve_raw(B, st, co, yl, yh, res, tx, ty, full, status, iters, w, npp, dtp)
        out = {"result": res.T.copy(), "traj_x": tx.T.copy(), "traj_y": ty.T.copy(), "status": status, "iters": iters}
        if want_full:
            out["full"] = full.T.copy()
        return out


def config_defaults():
    cfg = MpcConfig()
    _check(lib().mpc_config_defaults(C.byref(cfg)), "mpc_config_defaults")
    return cfg


def config_from_json_file(path):
    """Config::load(path)."""
    cfg = MpcConfig()
    _check(lib().mpc_config_load_json(path.encode(), C.byref(cfg)), "mpc_config_load_json")
    return cfg


def config_from_json_text(text):
    cfg = MpcConfig()
    _check(lib().mpc_config_parse_json(text.encode(), C.byref(cfg)), "mpc_config_parse_json")
    return cfg


def config_from_cli(argv, config_dir):
    """mpc_main.cpp's command line (without the program name) -> (MpcConfig, chosen config file)."""
    cfg = MpcConfig()
    arr = (C.c_char_p * max(len(argv), 1))(*[a.encode() for a in argv])
    buf = C.create_string_buffer(1024)
    _check(lib().mpc_config_from_cli(len(argv), arr, config_dir.encode(), C.byref(cfg), buf, 1024), "mpc_config_from_cli")
    return cfg, buf.value.decode()


def telemetry_parse(msg):
    """hasData + parse of one SocketIO text (mpc_main.cpp:26-36, 92-124) -> MpcTelemetry."""
    t = MpcTelemetry()
    _check(lib().mpc_telemetry_parse(msg.encode(), C.byref(t)), "mpc_telemetry_parse")
    return t


def measure_fp64_peak(device=0):
    """Measured DFMA peak of the device in TFLOP/s (2 flop per FMA)."""
    v = C.c_double(0.0)
    _check(lib().mpc_measure_fp64_peak(device, C.byref(v)), "mpc_measure_fp64_peak")
    return v.value


def run_prepare(cfg, pose, ptsx, ptsy, steering=0.0):
    """MPC::run pre-processing (host): pose (x, y, psi, v) + global waypoints -> dict with the NLP
    inputs, the vehicle-frame waypoints and the ``mpc_run_aux`` needed by :func:`run_finish`."""
    dp = C.POINTER(C.c_double)
    po = np.ascontiguousarray(pose, dtype=np.float64)
    x = np.array(ptsx, dtype=np.float64)
    y = np.array(ptsy, dtype=np.float64)
    st, co = np.zeros(6), np.zeros(NCOEF)
    lo, hi = C.c_double(0), C.c_double(0)
    aux = MpcRunAux()
    _check(lib().mpc_run_prepare(C.byref(cfg), po.ctypes.data_as(dp), float(steering), x.ctypes.data_as(dp),
                                 y.ctypes.data_as(dp), len(x), st.ctypes.data_as(dp), co.ctypes.data_as(dp),
                                 C.byref(lo), C.byref(hi), C.byref(aux)), "mpc_run_prepare")
    return {"state": st, "coeffs": co, "yaw_lo": lo.value, "yaw_hi": hi.value, "aux": aux, "ptsx": x, "ptsy": y}


def run_finish(cfg, aux, v, result9):
    """MPC::run post-processing: -> {x1, y1, psi1, v1, steer in [-1, 1], accel, cte1, epsi1}."""
    dp = C.POINTER(C.c_double)
    r = np.ascontiguousarray(result9, dtype=np.float64)
    out = np.zeros(8)
    _check(lib().mpc_run_finish(C.byref(cfg), C.byref(aux), float(v), r.ctypes.data_as(dp), out.ctypes.data_as(dp)),
           "mpc_run_finish")
    return out


def compute_throttle(cfg, accel, target):
    """Vehicle::computeThrottle (Vehicle.cpp:81-103)."""
    return lib().mpc_compute_throttle(C.byref(cfg), float(accel), float(target))


def vehicle_move(pose4, steering, accel, length, dt):
    """Vehicle::move (Vehicle.cpp:145-168): (x, y, psi, v) -> moved copy."""
    p = np.array(pose4, dtype=np.float64)
    lib().mpc_vehicle_move(p.ctypes.data_as(C.POINTER(C.c_double)), float(steering), float(accel), float(length), float(dt))
    return p


def _ptr(t):
    """Device/host pointer of a torch tensor, numpy array or None."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


class Solver:
    """One ``mpc_handle``: the batched replacement of an ``MPC`` object (MPC.cpp:160-325)."""

    def __init__(self, cfg, device=0):
        self.cfg = cfg
        self.device = device
        h = C.c_void_p()
        _check(lib().mpc_create(C.byref(cfg), device, C.byref(h)), "mpc_create")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            lib().mpc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_config(self, cfg):
        _check(lib().mpc_set_config(self._h, C.byref(cfg)), "mpc_set_config")
        self.cfg = cfg

    def set_kernel(self, kind=KERNEL_AUTO, lane_threads=0, lane_ctas_per_sm=0):
        """Pick the kernel (auto / one problem per warp / one problem per lane) and the lane grid."""
        _check(lib().mpc_set_kernel(self._h, kind, lane_threads, lane_ctas_per_sm), "mpc_set_kernel")

    def set_rollout_mode(self, mode):
        """0 = automatic, 1 = three launches per control step, 2 = one persistent launch (mpc_set_rollout_mode)."""
        _check(lib().mpc_set_rollout_mode(self._h, int(mode)), "mpc_set_rollout_mode")

    def set_tail(self, park_lanes, resume_launches, sort_ragged=True, resume_min=0, late_copy=False):
        """Tail packing of the lane kernel (mpc_set_tail): sparse-warp threshold, resume launches (each runs only if it
        finds more than resume_min records), ragged sort, copy-back timing."""
        _check(lib().mpc_set_tail(self._h, int(park_lanes), int(resume_launches), int(resume_min),
                                  (1 if sort_ragged else 0) | (4 if late_copy else 0)), "mpc_set_tail")

    def measure_solve_latency(self, state, coeffs, yaw_lo, yaw_hi, reps=1000, warmup=200):
        """(p50, p99) in microseconds of mpc_solve_one called from native code on the given problems ([n,6], [n,5], [n], [n])."""
        st = np.ascontiguousarray(state, dtype=np.float64); co = np.ascontiguousarray(coeffs, dtype=np.float64)
        yl = np.ascontiguousarray(yaw_lo, dtype=np.float64); yh = np.ascontiguousarray(yaw_hi, dtype=np.float64)
        assert co.shape[1] == NCOEF and st.shape[1] == 6
        p50, p99 = C.c_double(0), C.c_double(0)
        _check(lib().mpc_measure_solve_latency(self._h, st.shape[0], st.ctypes.data, co.ctypes.data, yl.ctypes.data, yh.ctypes.data,
                                               reps, warmup, C.byref(p50), C.byref(p99)), "mpc_measure_solve_latency")
        return p50.value, p99.value

    def tail_counts(self, n=4):
        """Problems parked by each launch of the last lane-kernel chain (mpc_tail_counts)."""
        out = (C.c_int * n)()
        _check(lib().mpc_tail_counts(self._h, out, n), "mpc_tail_counts")
        return list(out)

    def set_handoff(self, iterations):
        """Iteration count after which the lane kernel hands a problem to the coop kernel (0 = never)."""
        _check(lib().mpc_set_handoff(self._h, iterations), "mpc_set_handoff")

    def set_dual_outputs(self, lam=None, zl=None, zu=None):
        """Device tensors lam [6N][B], zl, zu [8N-2][B] receiving the multipliers of later solves (None = off)."""
        self._dual = (lam, zl, zu)   # keep them alive
        _check(lib().mpc_set_dual_outputs(self._h, _ptr(lam), _ptr(zl), _ptr(zu)), "mpc_set_dual_outputs")

    def set_warm_start(self, x0=None, lam0=None, zl0=None, zu0=None, mu_init=0.0):
        """Warm start of later batch solves (mpc_set_warm_start): device tensors x0 [8N-2][B] (as ``full``), lam0 [6N][B],
        zl0, zu0 [8N-2][B] (as the dual outputs; each may be None), unscaled; mu_init 0 = Ipopt's 0.1.  x0 None = off."""
        self._warm = (x0, lam0, zl0, zu0)   # keep them alive
        _check(lib().mpc_set_warm_start(self._h, _ptr(x0), _ptr(lam0), _ptr(zl0), _ptr(zu0), float(mu_init)),
               "mpc_set_warm_start")

    def set_warm_start_one(self, on, mu_init=0.0):
        """solve_one starts from its previous solution shifted by one stage (mpc_set_warm_start_one)."""
        _check(lib().mpc_set_warm_start_one(self._h, int(bool(on)), float(mu_init)), "mpc_set_warm_start_one")

    def warm_start_shift(self, B, x, x0, lam=None, lam0=None, zl=None, zl0=None, zu=None, zu0=None, stream=None):
        """Receding-horizon shift of a solution into the next step's start point (mpc_warm_start_shift), device
        tensors in the layouts of set_warm_start; asynchronous on ``stream`` (None = torch's current stream)."""
        if stream is None:
            import torch
            stream = torch.cuda.current_stream().cuda_stream
        _check(lib().mpc_warm_start_shift(self._h, int(B), _ptr(x), _ptr(lam), _ptr(zl), _ptr(zu), _ptr(x0), _ptr(lam0),
                                          _ptr(zl0), _ptr(zu0), stream), "mpc_warm_start_shift")

    def solution_sensitivity(self, B, state, coeffs, yaw_lo, yaw_hi, full, lam, zl, zu, dresult, dfull=None, status=None,
                             weights=None, dt_per=None, stream=None):
        """Derivatives of solutions with respect to the initial state (mpc_solution_sensitivity): DEVICE tensors in the
        [k][B] layout of solve_batch_device -- the problem arrays of the solve, its ``full``, the multipliers of
        set_dual_outputs and (optionally) its status -> dresult [6][9][B] and dfull [6][8N-2][B] (or None), slice k =
        d/d state_k.  Asynchronous on ``stream`` (None = torch's current stream)."""
        if stream is None:
            import torch
            stream = torch.cuda.current_stream().cuda_stream
        _check(lib().mpc_solution_sensitivity(self._h, int(B), _ptr(state), _ptr(coeffs), _ptr(yaw_lo), _ptr(yaw_hi),
                                              _ptr(weights), _ptr(dt_per), _ptr(full), _ptr(lam), _ptr(zl), _ptr(zu),
                                              _ptr(status), _ptr(dresult), _ptr(dfull), stream),
               "mpc_solution_sensitivity")

    @property
    def launches(self):
        return int(lib().mpc_launch_count(self._h))

    def solve_batch_device(self, B, state, coeffs, yaw_lo, yaw_hi, result, traj_x=None, traj_y=None,
                           full=None, status=None, iters=None, weights=None, N_per=None, dt_per=None,
                           stream=None):
        """Asynchronous solve; every array is a DEVICE tensor in the [k][B] layout of the header.

        ``stream`` is a raw cudaStream_t (int); None = torch's current stream."""
        if stream is None:
            import torch
            stream = torch.cuda.current_stream().cuda_stream
        _check(lib().mpc_solve_batch(self._h, B, _ptr(state), _ptr(coeffs), _ptr(yaw_lo), _ptr(yaw_hi),
                                     _ptr(weights), _ptr(N_per), _ptr(dt_per), _ptr(result), _ptr(traj_x),
                                     _ptr(traj_y), _ptr(full), _ptr(status), _ptr(iters), stream),
               "mpc_solve_batch")

    def solve_batch_host(self, state, coeffs, yaw_lo, yaw_hi, weights=None, N_per=None, dt_per=None,
                         want_traj=True, want_full=False):
        """Host numpy in ([B,6], [B,5], [B], [B]) -> dict of host numpy outputs ([B,...])."""
        B = state.shape[0]
        N = self.cfg.N
        st = np.ascontiguousarray(np.asarray(state, dtype=np.float64).T)
        co = np.ascontiguousarray(np.asarray(coeffs, dtype=np.float64).T)
        yl = np.ascontiguousarray(yaw_lo, dtype=np.float64)
        yh = np.ascontiguousarray(yaw_hi, dtype=np.float64)
        w = None if weights is None else np.ascontiguousarray(np.asarray(weights, dtype=np.float64).T)
        npp = None if N_per is None else np.ascontiguousarray(N_per, dtype=np.int32)
        dtp = None if dt_per is None else np.ascontiguousarray(dt_per, dtype=np.float64)
        res = np.zeros((9, B))
        tx = np.zeros((N, B)) if want_traj else None
        ty = np.zeros((N, B)) if want_traj else None
        full = np.zeros((8 * N - 2, B)) if want_full else None
        status = np.zeros(B, dtype=np.int32)
        iters = np.zeros(B, dtype=np.int32)
        _check(lib().mpc_solve_batch_host(self._h, B, _ptr(st), _ptr(co), _ptr(yl), _ptr(yh), _ptr(w),
                                          _ptr(npp), _ptr(dtp), _ptr(res), _ptr(tx), _ptr(ty), _ptr(full),
                                          _ptr(status), _ptr(iters)), "mpc_solve_batch_host")
        out = {"result": res.T.copy(), "status": status, "iters": iters}
        if want_traj:
            out["traj_x"], out["traj_y"] = tx.T.copy(), ty.T.copy()
        if want_full:
            out["full"] = full.T.copy()
        return out

    def run_batch_device(self, B, pose, ptsx, ptsy, npts, out8, steering=None, traj_x=None, traj_y=None,
                         coeffs_out=None, ptsx_v=None, ptsy_v=None, status=None, iters=None, stream=None):
        """MPC::run for a batch on the device; every array a DEVICE tensor ([k][B] layout)."""
        if stream is None:
            import torch
            stream = torch.cuda.current_stream().cuda_stream
        _check(lib().mpc_run_batch(self._h, B, _ptr(pose), _ptr(steering), _ptr(ptsx), _ptr(ptsy), npts, _ptr(out8),
                                   _ptr(traj_x), _ptr(traj_y), _ptr(coeffs_out), _ptr(ptsx_v), _ptr(ptsy_v),
                                   _ptr(status), _ptr(iters), stream), "mpc_run_batch")

    def rollout_device(self, V, T, track_x, track_y, veh, seg, pending, dt_ctrl=0.1, tau_solve=0.0, rec=None,
                       stream=None):
        """Closed loop, V vehicles x T control steps (BASELINE config 5); DEVICE tensors, asynchronous."""
        if stream is None:
            import torch
            stream = torch.cuda.current_stream().cuda_stream
        _check(lib().mpc_rollout(self._h, V, T, _ptr(track_x), _ptr(track_y), int(track_x.numel()), _ptr(veh),
                                 _ptr(seg), _ptr(pending), float(dt_ctrl), float(tau_solve), _ptr(rec), stream),
               "mpc_rollout")

    def telemetry_step(self, msg, throttle_prev, tau_solve=0.0, with_trajectory=False):
        """One simulator message through the controller -> (reply text, new throttle_prev)."""
        thr = C.c_double(throttle_prev)
        buf = C.create_string_buffer(8192)
        _check(lib().mpc_telemetry_step(self._h, msg.encode(), C.byref(thr), float(tau_solve), int(with_trajectory), buf, 8192),
               "mpc_telemetry_step")
        return buf.value.decode(), thr.value

    def solve_one(self, state, coeffs, yaw_lo, yaw_hi):
        N = self.cfg.N
        st = np.ascontiguousarray(state, dtype=np.float64)
        co = np.zeros(NCOEF)
        co[: len(coeffs)] = coeffs
        res, tx, ty = np.zeros(9), np.zeros(N), np.zeros(N)
        status, iters = C.c_int(0), C.c_int(0)
        dp = C.POINTER(C.c_double)
        _check(lib().mpc_solve_one(self._h, st.ctypes.data_as(dp), co.ctypes.data_as(dp), float(yaw_lo),
                                   float(yaw_hi), res.ctypes.data_as(dp), tx.ctypes.data_as(dp),
                                   ty.ctypes.data_as(dp), C.byref(status), C.byref(iters)), "mpc_solve_one")
        return {"result": res, "traj_x": tx, "traj_y": ty, "status": status.value, "iters": iters.value}
