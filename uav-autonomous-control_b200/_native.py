"""ctypes binding of libuavb.so (include/uavb.h) for PyTorch device tensors.

PyTorch is plumbing here: it owns device memory and streams; every computation happens in the
hand-written sm_100a kernels behind the C ABI.  There is NO fallback: if the library is missing, or
no CUDA device is visible, the calls raise.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_longlong, c_ulonglong, c_void_p

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libuavb.so")

N_GAINS = 11
N_METRICS = 8
ABI_VERSION = 210          # UAVB_VERSION of include/uavb.h this module's struct mirrors were written against
CARRY_WORDS = 52
STATE_DIM = 13
MAX_SPLINES = 64
SOLVE_OK, SOLVE_DEGENERATE, SOLVE_NONFINITE, SOLVE_TOO_MANY = range(4)
TARGET_ROW_BYTES = 56
PLAN_REPORT_INTS = 128
GAIN_NAMES = ("kp_xy", "kd_xy", "kp_z", "kd_z", "ki_z", "kp_roll", "kp_pitch", "kp_yaw", "kp_p", "kp_q", "kp_r")
M_FINAL_DIST, M_COLLISION, M_RMSE, M_MEAN_ERR, M_MAX_ERR, M_STATUS, M_FIRST_HIT, M_PERIODS = range(8)
(STAGE_OUTER, STAGE_INNER, STAGE_PHYSICS, STAGE_ALTITUDE, STAGE_LATERAL, STAGE_ROLL_PITCH, STAGE_YAW, STAGE_BODY_RATE, STAGE_ALLOCATE,
 STAGE_PROPELLER, STAGE_ATTITUDE) = range(1, 12)

# every symbol include/uavb.h declares (tests check the library exports all of them)
SYMBOLS = (
    "uavb_version", "uavb_last_error", "uavb_device_count", "uavb_device_info", "uavb_minsnap_solve_f64",
    "uavb_minsnap_solve_ragged_f64", "uavb_minsnap_table_meta_f64", "uavb_minsnap_sample_f64", "uavb_minsnap_yaw_profile_f64",
    "uavb_minsnap_table_hits_f64", "uavb_minsnap_correct_f64", "uavb_minsnap_pack_f64", "uavb_plan_shared_f64", "uavb_minsnap_constraints_f64",
    "uavb_rollout_targets_f64", "uavb_rollout_f32", "uavb_rollout_f64", "uavb_vehicle_defaults", "uavb_stage_f32", "uavb_mc_uniform_f32",
    "uavb_mc_missions_f64", "uavb_measure_fma_peak", "uavb_measure_fma_rates", "uavb_minsnap_solve_f64_host", "uavb_fly_mission_host", "uavb_rrt_workspace_bytes", "uavb_rrt_star_f64", "uavb_segments_hit_aabbs_f64",
    "uavb_table_targets_f64", "uavb_rollout_tables_f32",
)


class UavbError(RuntimeError):
    pass


class Vehicle(Structure):
    """struct uavb_vehicle (include/uavb.h); defaults = lab_course.xml + Quad.__init__ gains."""
    _fields_ = [
        ("g", c_double), ("dt", c_double), ("mass", c_double), ("inertia", c_double * 3),
        ("arm", c_double), ("kf", c_double), ("kappa", c_double), ("min_thrust", c_double), ("max_thrust", c_double),
        ("tau_rise", c_double), ("tau_fall", c_double), ("max_ascent", c_double), ("max_descent", c_double),
        ("max_speed_xy", c_double), ("max_horiz_accel", c_double), ("max_tilt", c_double),
        ("gains", c_double * N_GAINS), ("integral_limit", c_double),
    ]


class RolloutArgs(Structure):
    """struct uavb_rollout_args (include/uavb.h)."""
    _fields_ = [
        ("B", c_int), ("n_ticks", c_int), ("inner_per_outer", c_int), ("thrust_frame_lag", c_int), ("resume", c_int),
        ("log_stride", c_int), ("n_obs", c_int), ("n_obs_sets", c_int), ("index_base", c_longlong),
        ("veh", Vehicle),
        ("mc_mass", c_void_p), ("mc_inertia", c_void_p), ("mc_gains", c_void_p), ("mc_wind", c_void_p),
        ("seg_coeffs", c_void_p), ("seg_rows", c_void_p), ("seg_table", c_void_p), ("seg_yaw0", c_void_p),
        ("mission_seg_begin", c_void_p), ("mission_seg_count", c_void_p), ("n_seg_shared", c_int), ("dt_outer", c_double),
        ("shared_targets", c_void_p), ("n_target_rows", c_int), ("n_slices", c_int),
        ("start", c_void_p), ("start_stride", c_int), ("goal", c_void_p), ("goal_stride", c_int),
        ("aabbs", c_void_p), ("aabb_set", c_void_p),
        ("carry", c_void_p), ("state_out", c_void_p), ("metrics_out", c_void_p), ("log_out", c_void_p),
        ("traj_out", c_void_p), ("traj_count_out", c_void_p), ("traj_max_samples", c_int), ("traj_gate_z", c_double), ("traj_interval", c_double),
        ("ground_on", c_int), ("ground_z", c_double), ("pair_kernel_only", c_int), ("log_tma", c_int),
    ]


class TableSet(Structure):
    """struct uavb_table_set (include/uavb.h): caller trajectory tables for uavb_rollout_tables_f32."""
    _fields_ = [("rows", c_void_p), ("offsets", c_void_p), ("table_index", c_void_p), ("n_tables", c_int), ("shared_rows", c_int)]


class StageArgs(Structure):
    """struct uavb_stage_args (include/uavb.h)."""
    _fields_ = [
        ("B", c_int), ("stage", c_int), ("veh", Vehicle), ("dt_outer", c_double),
        ("mc_mass", c_void_p), ("mc_inertia", c_void_p), ("mc_gains", c_void_p), ("wind", c_void_p),
        ("X", c_void_p), ("target", c_void_p), ("rot", c_void_p), ("integral", c_void_p), ("thrust", c_void_p), ("bxy", c_void_p),
        ("pqr_cmd", c_void_p), ("moment", c_void_p), ("forces", c_void_p), ("omega", c_void_p), ("omega_cmd", c_void_p), ("zb", c_void_p),
        ("zb_out", c_void_p), ("aabbs", c_void_p), ("n_obs", c_int), ("collided", c_void_p), ("rot_out", c_void_p), ("euler_out", c_void_p),
    ]


class MissionHost(Structure):
    """struct uavb_mission_host (include/uavb.h): one mission, B drones, host buffers."""
    _fields_ = [
        ("B", c_int), ("n_waypoints", c_int), ("n_takeoff_waypoints", c_int), ("waypoints", c_void_p), ("velocity", c_double),
        ("start_end_time_factor", c_double), ("frequency", c_int), ("n_ticks", c_int), ("thrust_frame_lag", c_int), ("veh", Vehicle),
        ("mc_mass", c_void_p), ("mc_inertia", c_void_p), ("mc_gains", c_void_p), ("mc_wind", c_void_p), ("aabbs", c_void_p),
        ("n_obs", c_int), ("start", c_void_p), ("goal", c_void_p), ("plan_aabbs", c_void_p), ("no_correction", c_int),
    ]


_lib = None


def lib() -> ctypes.CDLL:
    """Load libuavb.so once.  Raises (no fallback) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise UavbError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(nvcc, sm_100a). There is no CPU or PyTorch fallback for this path.")
    L = ctypes.CDLL(LIB_PATH)
    L.uavb_version.restype = c_int
    if L.uavb_version() != ABI_VERSION:
        raise UavbError(f"libuavb.so reports ABI {L.uavb_version()}, this package expects {ABI_VERSION}: rebuild with uav-autonomous-control_b200/build.py")
    L.uavb_last_error.restype = c_char_p
    L.uavb_device_count.restype = c_int
    L.uavb_device_info.argtypes = [c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int)]
    L.uavb_minsnap_solve_f64.argtypes = [c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_void_p, c_void_p, c_void_p]
    L.uavb_minsnap_solve_ragged_f64.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_double, c_void_p, c_void_p, c_void_p, c_void_p]
    L.uavb_minsnap_table_meta_f64.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_double, c_void_p, c_void_p, c_void_p, c_void_p]
    L.uavb_minsnap_sample_f64.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_double, c_void_p, c_void_p]
    L.uavb_minsnap_yaw_profile_f64.argtypes = [c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_void_p]
    L.uavb_minsnap_table_hits_f64.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p]
    L.uavb_minsnap_correct_f64.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_double, c_void_p, c_int, c_longlong, c_void_p, c_void_p,
                                           c_void_p, POINTER(c_int), c_void_p]
    L.uavb_minsnap_pack_f64.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]
    L.uavb_minsnap_constraints_f64.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]
    L.uavb_plan_shared_f64.argtypes = [c_int, POINTER(c_void_p), POINTER(c_int), c_void_p, c_double, c_double, c_void_p, c_int, c_int, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int), c_void_p, c_void_p]
    L.uavb_rollout_targets_f64.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_double, c_void_p, c_int, c_void_p]
    L.uavb_rollout_f32.argtypes = [POINTER(RolloutArgs), c_void_p]
    L.uavb_rollout_f64.argtypes = [POINTER(RolloutArgs), c_void_p]
    L.uavb_table_targets_f64.argtypes = [c_void_p, c_longlong, c_void_p, c_void_p]
    L.uavb_rollout_tables_f32.argtypes = [POINTER(RolloutArgs), POINTER(TableSet), c_void_p]
    L.uavb_vehicle_defaults.argtypes = [POINTER(Vehicle)]
    L.uavb_vehicle_defaults.restype = None
    L.uavb_stage_f32.argtypes = [POINTER(StageArgs), c_void_p]
    L.uavb_mc_uniform_f32.argtypes = [c_ulonglong, c_longlong, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]
    L.uavb_mc_missions_f64.argtypes = [c_ulonglong, c_longlong, c_int, c_int, c_void_p, c_void_p, c_void_p]
    L.uavb_measure_fma_peak.argtypes = [c_int, POINTER(c_double), POINTER(c_double)]
    L.uavb_measure_fma_rates.argtypes = [c_int, POINTER(c_double), POINTER(c_double), POINTER(c_double)]
    L.uavb_minsnap_solve_f64_host.argtypes = [c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_void_p, c_void_p]
    L.uavb_rrt_workspace_bytes.argtypes = [c_int, c_int]
    L.uavb_rrt_star_f64.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_double, c_int, c_void_p, c_int, c_ulonglong, c_longlong, c_void_p,
                                    c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    L.uavb_segments_hit_aabbs_f64.argtypes = [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p]
    L.uavb_fly_mission_host.argtypes = [POINTER(MissionHost), c_void_p, c_void_p, POINTER(c_int)]
    for name in SYMBOLS:
        fn = getattr(L, name)
        if name not in ("uavb_last_error", "uavb_vehicle_defaults", "uavb_rrt_workspace_bytes"):
            fn.restype = c_int
    L.uavb_rrt_workspace_bytes.restype = c_longlong
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().uavb_last_error()
        raise UavbError(f"{what} failed with code {rc}: {msg.decode() if msg else ''}")


def default_vehicle() -> Vehicle:
    v = Vehicle()
    lib().uavb_vehicle_defaults(ctypes.byref(v))
    return v


def stream_ptr(device=None) -> c_void_p:
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


class _OnDevice:
    """``on(dev).uavb_xyz(args...)``: the library call with ``dev`` as the CURRENT device (the library sizes grids, picks its scratch
    pool and validates against cudaGetDevice()), return code checked."""

    def __init__(self, dev):
        self._dev = torch.device(dev)

    def __getattr__(self, name):
        fn = getattr(lib(), name)

        def call(*args):
            with torch.cuda.device(self._dev):
                check(fn(*args), name)
        return call


def on(dev) -> _OnDevice:
    return _OnDevice(dev)


def ptr(t: torch.Tensor | None, dtype: torch.dtype | None = None, name: str = "tensor") -> c_void_p:
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return c_void_p(None)
    if not t.is_cuda:
        raise UavbError(f"{name} must be a CUDA tensor (libuavb has no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise UavbError(f"{name} must have dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise UavbError(f"{name} must be contiguous")
    return c_void_p(t.data_ptr())


def device_info(dev: int = 0):
    sm, ma, mi = c_int(), c_int(), c_int()
    check(lib().uavb_device_info(dev, ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi)), "uavb_device_info")
    return sm.value, ma.value, mi.value


def measure_fma_peak(dev: int = 0):
    a, b = c_double(), c_double()
    check(lib().uavb_measure_fma_peak(dev, ctypes.byref(a), ctypes.byref(b)), "uavb_measure_fma_peak")
    return a.value, b.value


def measure_fma_rates(dev: int = 0):
    """(fp32, fp32 with three distinct register operands, fp64) FMA rates in TFLOP/s."""
    a, b, c = c_double(), c_double(), c_double()
    check(lib().uavb_measure_fma_rates(dev, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)), "uavb_measure_fma_rates")
    return a.value, b.value, c.value
