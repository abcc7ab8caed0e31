"""Host-side mirror of the reference filter interface over the C ABI (batched).

Method names follow the MATLAB API that the reference publishes (matlab/*.m) and the C++ private methods
they correspond to (C++/src/filter.cpp); every method is one C-ABI call (include/fbus_ekf.h):

  InitGravityAndGyrobias   InitGravityAndGyrobias.m   == FILTER::InitializeGravityAndBias (filter.cpp:256-285)
  InitPositionAndQuaternion InitPositionAndQuaternion.m == FILTER::InitializePose         (filter.cpp:291-399)
  ImuUpdate                ImuUpdate.m loop            == FILTER::BatchImuProcessing      (filter.cpp:483-531)
  ResetState               ResetState.m                == FILTER::ResetSystemState        (filter.cpp:405-477)
  MeasureUpdate            MeasureUpdate.m             == FILTER::ObservationUpdate       (filter.cpp:622-739)
  StepWindows              FBUS_EKF.m main loop        == FILTER::FilterThreadFunction body (filter.cpp:207-235)
  RefractSolve / MarkerPose                            == VISION::RefractionTriangulation + ComputeMarkerPose
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi


class FbusError(RuntimeError):
    pass


class BatchFilter:
    """`batch` independent FBUS-EKF filters resident on one CUDA device."""

    def __init__(self, cfg: capi.FbusConfig | None = None, batch: int = 1, device: int = 0):
        self._lib = capi.lib()
        self.cfg = cfg if cfg is not None else capi.config_default()
        self.batch = int(batch)
        self.device = int(device)
        self._h = C.c_void_p()
        rc = self._lib.fbus_create(C.byref(self._h), C.byref(self.cfg), self.device, self.batch)
        if rc != 0:
            msg = self._lib.fbus_last_error(None)
            self._h = C.c_void_p()
            raise FbusError(f"fbus_create failed ({rc}): {msg.decode() if msg else ''}")

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.fbus_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc: int):
        if rc != 0:
            msg = self._lib.fbus_last_error(self._h)
            raise FbusError(f"fbus call failed ({rc}): {msg.decode() if msg else ''}")

    # ---- F6 ----
    def InitGravityAndGyrobias(self, imu: capi.ImuStream, first: int, count: int):
        self._ck(self._lib.fbus_init_gravity_gyrobias(self._h, C.byref(imu), first, count))

    def IirPrefilter(self, imu: capi.ImuStream, first: int, count: int, out=None, mem: int = capi.FBUS_MEM_HOST):
        """FILTER::SetImuData's 1-pole IIR (filter.cpp:36-48) over samples [first, first+count), restarted at `first`.
        -> float64 [count][6][B] in SI units: a new numpy array, the given numpy array, or the given device pointer"""
        if mem == capi.FBUS_MEM_HOST:
            if out is None:
                out = np.empty((count, 6, self.batch))
            assert out.dtype == np.float64 and out.flags["C_CONTIGUOUS"] and out.size == count * 6 * self.batch
            self._ck(self._lib.fbus_iir_prefilter(self._h, C.byref(imu), first, count, out.ctypes.data, mem))
        else:
            self._ck(self._lib.fbus_iir_prefilter(self._h, C.byref(imu), first, count, int(out), mem))
        return out

    def InitPositionAndQuaternion(self, det: capi.DetFrames, frame: int, n_imu_before: int = 1):
        self._ck(self._lib.fbus_init_position_quaternion(self._h, C.byref(det), frame, n_imu_before))

    # ---- F1-F5 ----
    def ImuUpdate(self, imu: capi.ImuStream, first: int, count: int, t_end: float = float("inf")):
        self._ck(self._lib.fbus_propagate(self._h, C.byref(imu), first, count, t_end))

    def ResetState(self, det: capi.DetFrames, frame: int):
        self._ck(self._lib.fbus_reset_state(self._h, C.byref(det), frame))

    def MeasureUpdate(self, det: capi.DetFrames, frame: int):
        self._ck(self._lib.fbus_update(self._h, C.byref(det), frame))

    def StepWindows(self, imu: capi.ImuStream, det: capi.DetFrames, win_off, w0: int, w1: int, trace: bool = False,
                    trace_dev_ptr: int | None = None):
        win_off = np.ascontiguousarray(win_off, dtype=np.uint32)
        tr = None
        if trace_dev_ptr is not None:
            self._ck(self._lib.fbus_step_windows(self._h, C.byref(imu), C.byref(det), capi.dptr(win_off, capi.c_uint32_p), w0, w1,
                                                 trace_dev_ptr, capi.FBUS_MEM_DEVICE))
            return None
        if trace:
            tr = np.zeros((w1 - w0, 17, self.batch))
        self._ck(self._lib.fbus_step_windows(self._h, C.byref(imu), C.byref(det), capi.dptr(win_off, capi.c_uint32_p), w0, w1,
                                             tr.ctypes.data if tr is not None else None, capi.FBUS_MEM_HOST))
        return tr

    # ---- R1-R2 ----
    def RefractSolve(self, corners: np.ndarray):
        """corners float32 [16][n] -> (pose [7][n], corners3d [12][n], valid [n])"""
        assert corners.dtype == np.float32 and corners.flags["C_CONTIGUOUS"] and corners.shape[0] == 16
        n = corners.shape[1]
        pose = np.zeros((7, n))
        c3 = np.zeros((12, n))
        valid = np.zeros(n, dtype=np.int32)
        self._ck(self._lib.fbus_refract_solve(self._h, corners.ctypes.data, n, pose.ctypes.data, c3.ctypes.data, valid.ctypes.data,
                                              capi.FBUS_MEM_HOST))
        return pose, c3, valid

    def RefractSolveDevice(self, corners_ptr: int, n: int, pose_ptr: int, c3_ptr: int | None, valid_ptr: int | None):
        self._ck(self._lib.fbus_refract_solve(self._h, corners_ptr, n, pose_ptr, c3_ptr, valid_ptr, capi.FBUS_MEM_DEVICE))

    def SolveToDetections(self, corners, marker_ids, n_frames: int, max_markers: int, underwater: bool = True, gn_iters: int = 0,
                          det_id=None, det_pose=None, mem: int = capi.FBUS_MEM_HOST):
        """corners float32 [16][W*m*B], marker_ids int32 [W][m][B] -> (det_id int32 [W][m][B], det_pose float64 [W][m][7][B]);
        numpy arrays (host) or device pointers with preallocated outputs"""
        if mem == capi.FBUS_MEM_HOST:
            n = n_frames * max_markers * self.batch
            assert corners.dtype == np.float32 and corners.shape == (16, n) and corners.flags["C_CONTIGUOUS"]
            assert marker_ids.dtype == np.int32 and marker_ids.size == n and marker_ids.flags["C_CONTIGUOUS"]
            det_id = np.zeros((n_frames, max_markers, self.batch), dtype=np.int32)
            det_pose = np.zeros((n_frames, max_markers, 7, self.batch))
            self._ck(self._lib.fbus_solve_to_detections(self._h, corners.ctypes.data, marker_ids.ctypes.data, n_frames, max_markers,
                                                        int(underwater), gn_iters, det_id.ctypes.data, det_pose.ctypes.data, mem))
            return det_id, det_pose
        self._ck(self._lib.fbus_solve_to_detections(self._h, int(corners), int(marker_ids), n_frames, max_markers, int(underwater),
                                                    gn_iters, int(det_id), int(det_pose), mem))
        return det_id, det_pose

    def UndistortFisheye(self, pixels: np.ndarray) -> np.ndarray:
        """cv::fisheye::undistortPoints as DetectArucoTag applies it: pixel corners float32 [16][n] -> normalised float32 [16][n]"""
        assert pixels.dtype == np.float32 and pixels.flags["C_CONTIGUOUS"] and pixels.shape[0] == 16
        out = np.zeros_like(pixels)
        self._ck(self._lib.fbus_undistort_fisheye(self._h, pixels.ctypes.data, pixels.shape[1], out.ctypes.data, capi.FBUS_MEM_HOST))
        return out

    def InAirSolve(self, corners: np.ndarray):
        """VISION::NormalTriangulation + ComputeMarkerPose (land mode).  corners float32 [16][n] -> (pose, corners3d, valid)"""
        assert corners.dtype == np.float32 and corners.flags["C_CONTIGUOUS"] and corners.shape[0] == 16
        n = corners.shape[1]
        pose, c3, valid = np.zeros((7, n)), np.zeros((12, n)), np.zeros(n, dtype=np.int32)
        self._ck(self._lib.fbus_inair_solve(self._h, corners.ctypes.data, n, pose.ctypes.data, c3.ctypes.data, valid.ctypes.data,
                                            capi.FBUS_MEM_HOST))
        return pose, c3, valid

    def RefractSolveGN(self, corners: np.ndarray, iters: int = 5):
        """closed-form solve + Gauss-Newton refinement (R3).  corners float32 or float64 [16][n] ->
        (pose [7][n], cost [n], valid [n])"""
        assert corners.dtype in (np.float32, np.float64) and corners.flags["C_CONTIGUOUS"] and corners.shape[0] == 16
        n = corners.shape[1]
        pose = np.zeros((7, n))
        cost = np.zeros(n)
        valid = np.zeros(n, dtype=np.int32)
        self._ck(self._lib.fbus_refract_solve_gn(self._h, corners.ctypes.data, 1 if corners.dtype == np.float64 else 0, n, iters,
                                                 pose.ctypes.data, cost.ctypes.data, valid.ctypes.data, capi.FBUS_MEM_HOST))
        return pose, cost, valid

    def MarkerPose(self, corners3d: np.ndarray):
        assert corners3d.dtype == np.float64 and corners3d.flags["C_CONTIGUOUS"] and corners3d.shape[0] == 12
        n = corners3d.shape[1]
        pose = np.zeros((7, n))
        self._ck(self._lib.fbus_marker_pose(self._h, corners3d.ctypes.data, n, pose.ctypes.data, capi.FBUS_MEM_HOST))
        return pose

    # ---- state ----
    def GetState(self, with_cov: bool = True) -> dict:
        arrs = capi.alloc_state(self.batch, with_cov)
        sv = capi.state_view(arrs, self.batch)
        self._ck(self._lib.fbus_get_state(self._h, C.byref(sv)))
        return arrs

    def SetState(self, arrs: dict):
        sv = capi.state_view(arrs, self.batch)
        self._ck(self._lib.fbus_set_state(self._h, C.byref(sv)))

    def ClearStatus(self):
        self._ck(self._lib.fbus_clear_status(self._h))

    def Synchronize(self):
        self._ck(self._lib.fbus_synchronize(self._h))

    @property
    def stream(self) -> int:
        return int(self._lib.fbus_stream(self._h) or 0)

    # ---- statistics / workload support ----
    def Stats(self, truth_p, truth_q, mem: int = capi.FBUS_MEM_HOST, out_dev_ptr: int | None = None, want_host: bool = True):
        out = np.zeros(capi.FBUS_NSTATS)
        tp = truth_p.ctypes.data if isinstance(truth_p, np.ndarray) else int(truth_p)
        tq = truth_q.ctypes.data if isinstance(truth_q, np.ndarray) else int(truth_q)
        self._ck(self._lib.fbus_stats(self._h, tp, tq, mem, capi.dptr(out) if want_host else None, out_dev_ptr))
        return out

    def SetNoise(self, noise=None, mem: int = capi.FBUS_MEM_HOST):
        """Per-filter noise covariances (fbus_set_noise): float64 [6][B] numpy array, rows in capi.NOISE_FIELDS order, or a
        device pointer (mem = FBUS_MEM_DEVICE) to such an array.  None returns the handle to the config's values."""
        if noise is None:
            self._ck(self._lib.fbus_set_noise(self._h, None, mem))
            return
        if mem == capi.FBUS_MEM_HOST:
            assert isinstance(noise, np.ndarray) and noise.dtype == np.float64 and noise.flags["C_CONTIGUOUS"], "float64 C-contiguous array"
            assert noise.shape == (capi.FBUS_NOISE_FIELDS, self.batch), noise.shape
            self._ck(self._lib.fbus_set_noise(self._h, noise.ctypes.data, mem))
        else:
            self._ck(self._lib.fbus_set_noise(self._h, int(noise), mem))

    def SetGate(self, gate=None, mem: int = capi.FBUS_MEM_HOST):
        """Innovation gate (fbus_set_gate): float64 [B] numpy array of per-filter NIS thresholds (<= 0: no gate for that filter),
        or a device pointer (mem = FBUS_MEM_DEVICE) to such an array.  Resets the rejection counts.  None turns the gate off."""
        if gate is None:
            self._ck(self._lib.fbus_set_gate(self._h, None, mem))
            return
        if mem == capi.FBUS_MEM_HOST:
            assert isinstance(gate, np.ndarray) and gate.dtype == np.float64 and gate.flags["C_CONTIGUOUS"], "float64 C-contiguous array"
            assert gate.shape == (self.batch,), gate.shape
            self._ck(self._lib.fbus_set_gate(self._h, gate.ctypes.data, mem))
        else:
            self._ck(self._lib.fbus_set_gate(self._h, int(gate), mem))

    def RejectedUpdates(self, out=None, out_mem: int = capi.FBUS_MEM_HOST):
        """Updates rejected per filter since the last SetGate with an array (fbus_rejected_updates) -> int32 [B]: a new numpy
        array, the given numpy array, or the given device pointer (out_mem = FBUS_MEM_DEVICE)."""
        if out_mem == capi.FBUS_MEM_HOST:
            if out is None:
                out = np.empty(self.batch, dtype=np.int32)
            assert out.dtype == np.int32 and out.flags["C_CONTIGUOUS"] and out.shape == (self.batch,)
            self._ck(self._lib.fbus_rejected_updates(self._h, out.ctypes.data, out_mem))
        else:
            self._ck(self._lib.fbus_rejected_updates(self._h, int(out), out_mem))
        return out

    def FilterErrors(self, truth_p, truth_q, mem: int = capi.FBUS_MEM_HOST, out=None, out_mem: int = capi.FBUS_MEM_HOST):
        """Per-filter error terms (fbus_filter_errors) -> [4][B]: |p - p_true|^2, |dtheta|^2, NEES (6 dof), finite flag.
        truth_p [3][B], truth_q [4][B] float64 numpy arrays (or device pointers with mem = FBUS_MEM_DEVICE).  Output: a new
        numpy array, the given numpy array, or the given device pointer (out_mem = FBUS_MEM_DEVICE)."""
        if mem == capi.FBUS_MEM_HOST:
            for a, n in ((truth_p, 3), (truth_q, 4)):
                assert isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"] and a.shape == (n, self.batch)
            tp, tq = truth_p.ctypes.data, truth_q.ctypes.data
        else:
            tp, tq = int(truth_p), int(truth_q)
        if out_mem == capi.FBUS_MEM_HOST:
            if out is None:
                out = np.empty((4, self.batch))
            assert out.dtype == np.float64 and out.flags["C_CONTIGUOUS"] and out.shape == (4, self.batch)
            self._ck(self._lib.fbus_filter_errors(self._h, tp, tq, mem, out.ctypes.data, out_mem))
        else:
            self._ck(self._lib.fbus_filter_errors(self._h, tp, tq, mem, int(out), out_mem))
        return out

    def SynthStreams(self, spec: capi.SynthSpec, imu_ptr: int, det_id_ptr: int, det_pose_ptr: int, bias_ptr: int | None = None):
        self._ck(self._lib.fbus_synth_streams(self._h, C.byref(spec), imu_ptr, det_id_ptr, det_pose_ptr, bias_ptr))

    def MarkerProject(self, pose, underwater: bool = True, n: int | None = None, corners=None, valid=None,
                      mem: int = capi.FBUS_MEM_HOST):
        """Forward model of the stereo front end (fbus_marker_project): marker poses float64 [7][n] (p xyz, q wxyz of corner 0,
        flipped left-camera frame) -> (corners float64 [16][n], valid int32 [n]) in the input layout of RefractSolve /
        InAirSolve; an invalid item's corners are NaN.  With mem = FBUS_MEM_DEVICE, pose, corners and valid (or None) are
        device pointers and n is required."""
        if mem == capi.FBUS_MEM_HOST:
            pose = np.ascontiguousarray(pose, dtype=np.float64)
            assert pose.ndim == 2 and pose.shape[0] == 7, pose.shape
            n = pose.shape[1]
            corners = np.empty((16, n))
            valid = np.empty(n, dtype=np.int32)
            self._ck(self._lib.fbus_marker_project(self._h, pose.ctypes.data, n, int(underwater), corners.ctypes.data,
                                                   valid.ctypes.data, mem))
            return corners, valid
        self._ck(self._lib.fbus_marker_project(self._h, int(pose), int(n), int(underwater), int(corners),
                                               int(valid) if valid is not None else None, mem))
        return corners, valid

    def SynthCorners(self, spec: capi.CornerSpec, w0: int, w1: int, corners_ptr: int, ids_ptr: int):
        """Per-filter stereo corner streams of frames [w0, w1) (fbus_synth_corners) into DEVICE buffers: corners float32
        [16][(w1-w0)*m*B], ids int32 [w1-w0][m][B], the input of SolveToDetections"""
        self._ck(self._lib.fbus_synth_corners(self._h, C.byref(spec), int(w0), int(w1), int(corners_ptr), int(ids_ptr)))

    def MeasureFp64Peak(self) -> float:
        v = C.c_double(0.0)
        self._ck(self._lib.fbus_measure_fp64_peak(self._h, C.byref(v)))
        return v.value
