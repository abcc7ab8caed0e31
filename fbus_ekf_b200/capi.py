"""ctypes binding of the C ABI declared in include/fbus_ekf.h.

This is the stub a Python-side maintainer of the reference would add (see INTEGRATION.md); the
structures below are field-for-field mirrors of the C structs.  There is no CPU fallback: if the
shared library is missing, `lib()` raises, and if no CUDA device is usable `fbus_create` fails.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FBUS_EKF_LIB", os.path.join(HERE, "libfbus_ekf.so"))

FBUS_OK, FBUS_E_BADARG, FBUS_E_CUDA, FBUS_E_NOMEM, FBUS_E_STATE, FBUS_E_NCCL = 0, -1, -2, -3, -4, -5
FBUS_ABI_VERSION = 3  # include/fbus_ekf.h
FBUS_MEM_HOST = 0
FBUS_MEM_DEVICE = 1
FBUS_IMU_F64_SI = 0      # double, m/s^2 and rad/s (IMUData)
FBUS_IMU_F32_SENSOR = 1  # float, g and deg/s (the IMSEE SDK's ImuData; converted on the device as main.cpp:254 does)
# per-filter status bits (fbus_state_soa.status)
FBUS_ST_INIT_FAILED, FBUS_ST_RESET_SKIPPED, FBUS_ST_RESET_DONE, FBUS_ST_UPDATE_SKIPPED = 0x1, 0x2, 0x4, 0x8
FBUS_ST_NONFINITE, FBUS_ST_NO_DETECTION, FBUS_ST_MARKER_REJECTED = 0x10, 0x20, 0x40
FBUS_ST_UPDATE_REJECTED = 0x80  # rejected by the innovation gate (fbus_set_gate)
FBUS_FLAG_JOSEPH = 0x1
FBUS_FLAG_MATLAB = 0x2
FBUS_FLAG_ALL_MARKERS = 0x4  # every known marker of a frame updates the filter in turn (include/fbus_ekf.h)
FBUS_MAX_MARKERS = 16
FBUS_NSTATS = 8
# rows of a per-filter noise array (fbus_set_noise), in fbus_config order
NOISE_FIELDS = ("accel_n_cov", "gyro_n_cov", "accel_b_cov", "gyro_b_cov", "pos_n_cov", "quat_n_cov")
FBUS_NOISE_FIELDS = len(NOISE_FIELDS)

ST_INIT_FAILED = 0x1
ST_RESET_SKIPPED = 0x2
ST_RESET_DONE = 0x4
ST_UPDATE_SKIPPED = 0x8
ST_NONFINITE = 0x10
ST_NO_DETECTION = 0x20
ST_MARKER_REJECTED = 0x40

FLAG_JOSEPH = 0x1

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_float_p = C.POINTER(C.c_float)
c_uint32_p = C.POINTER(C.c_uint32)


class FbusConfig(C.Structure):
    _fields_ = [
        ("tsc_left", C.c_double * 16),
        ("tsc_right", C.c_double * 16),
        ("accel_n_cov", C.c_double), ("gyro_n_cov", C.c_double),
        ("accel_b_cov", C.c_double), ("gyro_b_cov", C.c_double),
        ("pos_n_cov", C.c_double), ("quat_n_cov", C.c_double),
        ("marker_max_dist", C.c_double), ("marker_switch_thres", C.c_double),
        ("p0_diag", C.c_double * 6),
        ("reset_gap", C.c_double),
        ("n_air", C.c_double), ("n_glass", C.c_double), ("n_water", C.c_double),
        ("d_air", C.c_double), ("d_glass", C.c_double),
        ("normal", C.c_double * 3),
        ("marker_dect_dist_thres", C.c_double),
        ("marker_size", C.c_double),
        ("cam_k", (C.c_double * 4) * 2),
        ("cam_d", (C.c_double * 4) * 2),
        ("n_markers", C.c_int32),
        ("marker_id", C.c_int32 * FBUS_MAX_MARKERS),
        ("marker_pos", C.c_double * (FBUS_MAX_MARKERS * 3)),
        ("marker_rot", C.c_double * (FBUS_MAX_MARKERS * 9)),
        ("flags", C.c_int32),
        ("reserved", C.c_int32),
        ("imu_g", C.c_double),
        ("gn_tol", C.c_double),
    ]


class ImuStream(C.Structure):
    _fields_ = [("n_samples", C.c_size_t), ("batch", C.c_size_t), ("t", c_double_p), ("data", C.c_void_p),
                ("mem", C.c_int32), ("format", C.c_int32)]


class DetFrames(C.Structure):
    _fields_ = [("n_frames", C.c_size_t), ("max_markers", C.c_size_t), ("batch", C.c_size_t), ("t", c_double_p),
                ("id", C.c_void_p), ("pose", C.c_void_p), ("mem", C.c_int32), ("reserved", C.c_int32)]


class StateSoa(C.Structure):
    _fields_ = [("batch", C.c_size_t), ("t", c_double_p), ("q", c_double_p), ("R", c_double_p), ("p", c_double_p),
                ("v", c_double_p), ("ba", c_double_p), ("bg", c_double_p), ("g", c_double_p), ("pv", c_double_p),
                ("qv", c_double_p), ("P", c_double_p), ("prev_marker_id", c_int32_p), ("initialised", c_int32_p),
                ("status", c_int32_p)]


class SynthSpec(C.Structure):
    _fields_ = [("n_samples", C.c_size_t), ("n_frames", C.c_size_t), ("base_imu", c_double_p), ("base_pose", c_double_p),
                ("marker_id", C.c_int32), ("reserved", C.c_int32),
                ("sigma_acc", C.c_double), ("sigma_gyro", C.c_double), ("sigma_ba", C.c_double), ("sigma_bg", C.c_double),
                ("sigma_pos", C.c_double), ("sigma_quat", C.c_double), ("seed", C.c_uint64), ("filter_offset", C.c_uint64)]


class CornerSpec(C.Structure):
    """fbus_corner_spec (fbus_synth_corners)"""
    _fields_ = [("n_frames", C.c_size_t), ("max_markers", C.c_size_t), ("base_pose", c_double_p), ("base_id", c_int32_p),
                ("underwater", C.c_int32), ("reserved", C.c_int32), ("sigma_corner", C.c_double), ("p_drop", C.c_double),
                ("p_outlier", C.c_double), ("sigma_outlier", C.c_double), ("seed", C.c_uint64), ("filter_offset", C.c_uint64)]


STATE_FIELDS = (("t", 1, np.float64), ("q", 4, np.float64), ("R", 9, np.float64), ("p", 3, np.float64),
                ("v", 3, np.float64), ("ba", 3, np.float64), ("bg", 3, np.float64), ("g", 3, np.float64),
                ("pv", 3, np.float64), ("qv", 4, np.float64), ("P", 324, np.float64),
                ("prev_marker_id", 1, np.int32), ("initialised", 1, np.int32), ("status", 1, np.int32))


def alloc_state(batch: int, with_cov: bool = True) -> dict:
    """dict of C-contiguous numpy arrays [n][B] (or [B]) matching fbus_state_soa."""
    out = {}
    for name, n, dt in STATE_FIELDS:
        if name == "P" and not with_cov:
            continue
        out[name] = np.zeros((batch,) if n == 1 else (n, batch), dtype=dt)
    return out


def state_view(arrs: dict, batch: int) -> StateSoa:
    s = StateSoa()
    s.batch = batch
    for name, n, dt in STATE_FIELDS:
        a = arrs.get(name)
        if a is None:
            continue
        assert a.flags["C_CONTIGUOUS"] and a.dtype == dt and a.size == n * batch, name
        ptr_t = c_double_p if dt == np.float64 else c_int32_p
        setattr(s, name, a.ctypes.data_as(ptr_t))
    return s


_lib = None


def lib() -> C.CDLL:
    """Loads libfbus_ekf.so (built in-tree by __graft_entry__.build()).  Fails loudly when missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"fbus_ekf_b200: CUDA library {LIB_PATH} is missing -- run __graft_entry__.build(); "
                           "there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    H = C.c_void_p
    sig = {
        "fbus_config_default": (C.c_int, [C.POINTER(FbusConfig)]),
        "fbus_config_matlab": (C.c_int, [C.POINTER(FbusConfig)]),
        "fbus_create": (C.c_int, [C.POINTER(H), C.POINTER(FbusConfig), C.c_int, C.c_size_t]),
        "fbus_destroy": (C.c_int, [H]),
        "fbus_last_error": (C.c_char_p, [H]),
        "fbus_abi_version": (C.c_int, []),
        "fbus_synchronize": (C.c_int, [H]),
        "fbus_batch": (C.c_size_t, [H]),
        "fbus_stream": (C.c_void_p, [H]),
        "fbus_init_gravity_gyrobias": (C.c_int, [H, C.POINTER(ImuStream), C.c_size_t, C.c_size_t]),
        "fbus_iir_prefilter": (C.c_int, [H, C.POINTER(ImuStream), C.c_size_t, C.c_size_t, C.c_void_p, C.c_int32]),
        "fbus_init_position_quaternion": (C.c_int, [H, C.POINTER(DetFrames), C.c_size_t, C.c_size_t]),
        "fbus_propagate": (C.c_int, [H, C.POINTER(ImuStream), C.c_size_t, C.c_size_t, C.c_double]),
        "fbus_reset_state": (C.c_int, [H, C.POINTER(DetFrames), C.c_size_t]),
        "fbus_update": (C.c_int, [H, C.POINTER(DetFrames), C.c_size_t]),
        "fbus_step_windows": (C.c_int, [H, C.POINTER(ImuStream), C.POINTER(DetFrames), c_uint32_p, C.c_size_t,
                                        C.c_size_t, C.c_void_p, C.c_int32]),
        "fbus_refract_solve": (C.c_int, [H, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
        "fbus_marker_pose": (C.c_int, [H, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int32]),
        "fbus_solve_to_detections": (C.c_int, [H, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32]),
        "fbus_undistort_fisheye": (C.c_int, [H, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int32]),
        "fbus_inair_solve": (C.c_int, [H, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
        "fbus_refract_solve_gn": (C.c_int, [H, C.c_void_p, C.c_int32, C.c_size_t, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
        "fbus_get_state": (C.c_int, [H, C.POINTER(StateSoa)]),
        "fbus_set_state": (C.c_int, [H, C.POINTER(StateSoa)]),
        "fbus_clear_status": (C.c_int, [H]),
        "fbus_stats": (C.c_int, [H, C.c_void_p, C.c_void_p, C.c_int32, c_double_p, C.c_void_p]),
        "fbus_stats_combine": (C.c_int, [c_double_p, C.c_size_t, c_double_p]),
        "fbus_set_noise": (C.c_int, [H, C.c_void_p, C.c_int32]),
        "fbus_filter_errors": (C.c_int, [H, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]),
        "fbus_set_gate": (C.c_int, [H, C.c_void_p, C.c_int32]),
        "fbus_rejected_updates": (C.c_int, [H, C.c_void_p, C.c_int32]),
        "fbus_stats_allreduce": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p), c_double_p]),
        "fbus_stats_allreduce_comm": (C.c_int, [H, C.c_void_p, C.c_void_p, c_double_p]),
        "fbus_synth_streams": (C.c_int, [H, C.POINTER(SynthSpec), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
        "fbus_marker_project": (C.c_int, [H, C.c_void_p, C.c_size_t, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32]),
        "fbus_synth_corners": (C.c_int, [H, C.POINTER(CornerSpec), C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p]),
        "fbus_quat_from_rotmat": (None, [c_double_p, c_double_p]),
        "fbus_measure_fp64_peak": (C.c_int, [H, c_double_p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if L.fbus_abi_version() != FBUS_ABI_VERSION:
        raise RuntimeError(f"fbus_ekf_b200: {LIB_PATH} has ABI version {L.fbus_abi_version()}, this binding mirrors version "
                           f"{FBUS_ABI_VERSION} of include/fbus_ekf.h -- rebuild with __graft_entry__.build()")
    _lib = L
    return L


EXPORTED_SYMBOLS = (
    "fbus_config_default", "fbus_config_matlab", "fbus_create", "fbus_destroy", "fbus_last_error", "fbus_abi_version", "fbus_synchronize",
    "fbus_batch", "fbus_stream", "fbus_init_gravity_gyrobias", "fbus_iir_prefilter", "fbus_init_position_quaternion", "fbus_propagate",
    "fbus_reset_state", "fbus_update", "fbus_step_windows", "fbus_refract_solve", "fbus_inair_solve", "fbus_undistort_fisheye", "fbus_solve_to_detections", "fbus_refract_solve_gn", "fbus_marker_pose", "fbus_get_state",
    "fbus_set_state", "fbus_clear_status", "fbus_stats", "fbus_stats_combine", "fbus_stats_allreduce", "fbus_stats_allreduce_comm", "fbus_synth_streams", "fbus_quat_from_rotmat",
    "fbus_measure_fp64_peak", "fbus_set_noise", "fbus_filter_errors", "fbus_marker_project", "fbus_synth_corners",
    "fbus_set_gate", "fbus_rejected_updates")


def config_default() -> FbusConfig:
    cfg = FbusConfig()
    rc = lib().fbus_config_default(C.byref(cfg))
    if rc != 0:
        raise RuntimeError("fbus_config_default failed")
    return cfg


def config_matlab() -> FbusConfig:
    """the constants of matlab/FBUS_EKF.m (P0, measurement noise) with FBUS_FLAG_MATLAB set"""
    cfg = FbusConfig()
    if lib().fbus_config_matlab(C.byref(cfg)) != 0:
        raise RuntimeError("fbus_config_matlab failed")
    return cfg


def noise_from_config(cfg: FbusConfig, batch: int) -> np.ndarray:
    """float64 [FBUS_NOISE_FIELDS][batch] array (fbus_set_noise layout) giving every filter the config's values"""
    col = np.array([getattr(cfg, name) for name in NOISE_FIELDS], dtype=np.float64)
    return np.ascontiguousarray(np.repeat(col[:, None], int(batch), axis=1))


def dptr(a: np.ndarray, typ=c_double_p):
    return a.ctypes.data_as(typ)


def make_imu_stream(t: np.ndarray, data, batch: int, mem: int = FBUS_MEM_HOST, keep: list | None = None,
                    fmt: int | None = None) -> ImuStream:
    """t: [N] float64 host array; data: numpy [N,6,B] (host; float64 in SI units or float32 in sensor units) or an int
    device pointer (then `fmt` says what it points to, default FBUS_IMU_F64_SI)."""
    s = ImuStream()
    t = np.ascontiguousarray(t, dtype=np.float64)
    s.n_samples = t.shape[0]
    s.batch = batch
    s.t = dptr(t)
    if isinstance(data, np.ndarray):
        assert data.dtype in (np.float64, np.float32) and data.flags["C_CONTIGUOUS"] and data.shape == (t.shape[0], 6, batch)
        s.data = data.ctypes.data
        if fmt is None:
            fmt = FBUS_IMU_F32_SENSOR if data.dtype == np.float32 else FBUS_IMU_F64_SI
        assert (fmt == FBUS_IMU_F32_SENSOR) == (data.dtype == np.float32)
    else:
        s.data = int(data)
    s.mem = mem
    s.format = FBUS_IMU_F64_SI if fmt is None else fmt
    if keep is not None:
        keep.extend([t, data])
    s._keep = (t, data)
    return s


def make_det_frames(t: np.ndarray, ids, pose, batch: int, max_markers: int, mem: int = FBUS_MEM_HOST) -> DetFrames:
    """t: [W]; ids: int32 [W,m,B]; pose: float64 [W,m,7,B] (numpy host arrays or device pointers)."""
    d = DetFrames()
    t = np.ascontiguousarray(t, dtype=np.float64)
    d.n_frames = t.shape[0]
    d.max_markers = max_markers
    d.batch = batch
    d.t = dptr(t)
    if isinstance(ids, np.ndarray):
        assert ids.dtype == np.int32 and ids.flags["C_CONTIGUOUS"] and ids.shape == (t.shape[0], max_markers, batch)
        assert pose.dtype == np.float64 and pose.flags["C_CONTIGUOUS"] and pose.shape == (t.shape[0], max_markers, 7, batch)
        d.id = ids.ctypes.data
        d.pose = pose.ctypes.data
    else:
        d.id = int(ids)
        d.pose = int(pose)
    d.mem = mem
    d._keep = (t, ids, pose)
    return d


REF_M_PI = 3.1415926  # common.hpp:14


def sensor_to_si(raw: np.ndarray, imu_g: float) -> np.ndarray:
    """float32 sensor units [N,6,B] (accel in g, gyro in deg/s) -> float64 SI, operation by operation as main.cpp:254:
    accel = (double)a * g ; gyro = (double)(w / 180.f) * M_PI   (host mirror of the kernels' conversion, for tests/oracle)"""
    raw = np.asarray(raw, dtype=np.float32)
    out = np.empty(raw.shape, dtype=np.float64)
    out[:, 0:3] = raw[:, 0:3].astype(np.float64) * np.float64(imu_g)
    out[:, 3:6] = (raw[:, 3:6] / np.float32(180.0)).astype(np.float64) * np.float64(REF_M_PI)
    return out


def si_to_sensor(si: np.ndarray, imu_g: float) -> np.ndarray:
    """nearest float32 sensor-unit sample of an SI stream (what a simulated IMSEE IMU would deliver)"""
    si = np.asarray(si, dtype=np.float64)
    out = np.empty(si.shape, dtype=np.float32)
    out[:, 0:3] = (si[:, 0:3] / imu_g).astype(np.float32)
    out[:, 3:6] = (si[:, 3:6] * (180.0 / REF_M_PI)).astype(np.float32)
    return out
