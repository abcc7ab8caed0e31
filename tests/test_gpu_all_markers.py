"""FBUS_FLAG_ALL_MARKERS on the GPU (include/fbus_ekf.h): every known marker of a frame updates the filter in turn.  The mode runs on
the first-generation lanes-per-filter kernel at every batch size and is checked against the mode's restatement on the C++ oracle
(tests/all_markers_ref.py)."""
import copy
import os

import numpy as np
import pytest

from all_markers_ref import OrcAllMarkers
from helpers import cov_close, cov_whitened_err, state_close
from test_all_markers_host import _board

pytestmark = pytest.mark.gpu


def _flags(cfg, flags):
    c = copy.copy(cfg)
    c.flags = flags
    return c


def _oracle(bcfg, flags, traj, imu, det_id, det_pose):
    """all frames on the C++ oracle in this mode (flags: FBUS_FLAG_ALL_MARKERS, optionally with FBUS_FLAG_JOSEPH)"""
    o = OrcAllMarkers(_flags(bcfg, flags), imu.shape[2])
    o.step_windows(traj["t_imu"], imu, traj["t_frames"], det_id, det_pose, traj["win_off"], 0, len(traj["t_frames"]))
    return o.get_state()


def _gpu(bcfg, flags, traj, imu, det_id, det_pose, env=None, noise=None, trace=False):
    from fbus_ekf_b200 import BatchFilter, capi
    B, m = imu.shape[2], det_id.shape[1]
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        f = BatchFilter(_flags(bcfg, flags), batch=B)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    if noise is not None:
        f.SetNoise(noise)
    s = capi.make_imu_stream(traj["t_imu"], imu, B)
    d = capi.make_det_frames(traj["t_frames"], det_id, det_pose, B, m)
    tr = f.StepWindows(s, d, traj["win_off"], 0, len(traj["t_frames"]), trace=trace)
    return f.GetState(), tr


def _check(sg, so, idx=None, n_whitened=4):
    if idx is not None:
        sg = {k: v[..., idx] for k, v in sg.items()}
    assert state_close(sg, so, 1e-9)[0]
    assert cov_close(sg["P"], so["P"], 1e-9)[0]
    assert np.array_equal(sg["prev_marker_id"], so["prev_marker_id"]) and np.array_equal(sg["status"], so["status"])
    for b in range(min(n_whitened, so["P"].shape[1])):   # the (p, theta) block the NEES inverts (test_gpu_precision's gate)
        assert cov_whitened_err(sg["P"][:, b], so["P"][:, b]) <= 1e-9


@pytest.mark.parametrize("joseph", [False, True])
def test_board_pipeline(cfg, joseph):
    """fbus_solve_to_detections -> fbus_step_windows on the GPU against the oracle chain on the same detections"""
    from fbus_ekf_b200 import BatchFilter, capi, synth
    B, m = 48, 8
    bcfg = synth.board_config(cfg)
    traj = synth.truth_trajectory(bcfg, 0.6, standoff=1.0)
    W, N = len(traj["t_frames"]), len(traj["t_imu"])
    base, ids, _ = synth.board_base_corners(bcfg, traj)
    rng = np.random.default_rng(8)
    corners = np.ascontiguousarray((np.repeat(base, B, axis=1) + rng.normal(size=(16, W * m * B)) * 2e-4).astype(np.float32))
    mids = np.ascontiguousarray(np.repeat(ids[:, :, None], B, axis=2))
    mids[3, 5, ::4] = -1
    mids[6, 2, 1::3] = 11                                  # not on the board: skipped with FBUS_ST_UPDATE_SKIPPED
    flags = capi.FBUS_FLAG_ALL_MARKERS | (capi.FBUS_FLAG_JOSEPH if joseph else 0)
    f = BatchFilter(_flags(bcfg, flags), batch=B)
    det_id, det_pose = f.SolveToDetections(corners, mids, W, m, underwater=True, gn_iters=4)
    imu = np.ascontiguousarray(traj["base_imu"][:, :, None] + rng.normal(size=(N, 6, B)) * np.array([0.015] * 3 + [1e-3] * 3)[None, :, None])
    s = capi.make_imu_stream(traj["t_imu"], imu, B)
    d = capi.make_det_frames(traj["t_frames"], det_id, det_pose, B, m)
    f.StepWindows(s, d, traj["win_off"], 0, W)
    so = _oracle(bcfg, flags, traj, imu, det_id, det_pose)
    sg = f.GetState()
    _check(sg, so)
    assert (sg["status"][1::3] & capi.FBUS_ST_UPDATE_SKIPPED).all()


def _tiled_board(B, duration=0.4):
    """board detections and IMU for min(B, 256) distinct filters, tiled to B (filter b has the inputs of filter b % 256)"""
    bcfg, traj, imu, det_id, det_pose = _board(B=min(B, 256), duration=duration, seed=11)
    reps = (B + 255) // 256 if B > 256 else 1
    til = lambda a: np.ascontiguousarray(np.concatenate([a] * reps, axis=-1)[..., :B])
    return bcfg, traj, imu, det_id, det_pose, til


@pytest.mark.parametrize("B", [1, 33, 4096, 65536])
def test_any_batch_size(B):
    """the default mode picks different kernels at these sizes; the flag always runs the lanes-per-filter kernel"""
    from fbus_ekf_b200 import capi
    bcfg, traj, imu, det_id, det_pose, til = _tiled_board(B)
    so = _oracle(bcfg, capi.FBUS_FLAG_ALL_MARKERS, traj, imu, det_id, det_pose)
    sg, _ = _gpu(bcfg, capi.FBUS_FLAG_ALL_MARKERS, traj, til(imu), til(det_id), til(det_pose))
    nb = imu.shape[2]
    _check(sg, so, idx=slice(0, nb))
    if B > 256:   # a spot check of the last 256 filters, which repeat the inputs of the first 256
        _check(sg, so, idx=slice(B - 256, B), n_whitened=0)


def test_single_marker_bitwise_equals_default():
    """one detection per frame: bit for bit the default mode on the same kernel (FBUS_LANE=1 FBUS_LANE_GEN=1)"""
    from fbus_ekf_b200 import capi
    bcfg, traj, imu, det_id, det_pose = _board(B=40, seed=12)
    det1 = det_id.copy()
    det1[:, 1:, :] = -1
    det1 = np.ascontiguousarray(det1)
    env = {"FBUS_LANE": "1", "FBUS_LANE_GEN": "1"}
    s0, t0 = _gpu(bcfg, 0, traj, imu, det1, det_pose, env=env, trace=True)
    s1, t1 = _gpu(bcfg, capi.FBUS_FLAG_ALL_MARKERS, traj, imu, det1, det_pose, trace=True)
    for k in s0:
        assert np.array_equal(s0[k], s1[k]), k
    assert np.array_equal(t0, t1)


def test_unfused_calls():
    """fbus_propagate / fbus_update against orc_propagate / orc_update"""
    from fbus_ekf_b200 import BatchFilter, capi
    bcfg, traj, imu, det_id, det_pose = _board(B=35, seed=13)
    B, m, W = imu.shape[2], 8, 6
    flags = capi.FBUS_FLAG_ALL_MARKERS
    o = OrcAllMarkers(_flags(bcfg, flags), B)
    f = BatchFilter(_flags(bcfg, flags), batch=B)
    s = capi.make_imu_stream(traj["t_imu"], imu, B)
    d = capi.make_det_frames(traj["t_frames"], det_id, det_pose, B, m)
    o.step_windows(traj["t_imu"], imu, traj["t_frames"], det_id, det_pose, traj["win_off"], 0, 3)  # initialise on the oracle ...
    f.SetState(o.get_state())                             # ... and start both from that state
    off = traj["win_off"]
    for w in range(3, W):
        o.propagate(s, int(off[w]), int(off[w + 1] - off[w]), float(traj["t_frames"][w]))
        f.ImuUpdate(s, int(off[w]), int(off[w + 1] - off[w]), float(traj["t_frames"][w]))
        o.update(traj["t_frames"], det_id, det_pose, w)
        f.MeasureUpdate(d, w)
    _check(f.GetState(), o.get_state())


def test_continuation_bitwise():
    """frames split over two continued calls (device-resident streams) equal one call bit for bit"""
    import torch
    from fbus_ekf_b200 import BatchFilter, capi
    bcfg, traj, imu, det_id, det_pose = _board(B=64, seed=14)
    B, m, W = imu.shape[2], 8, len(traj["t_frames"])
    dev = [torch.from_numpy(a).cuda() for a in (imu, det_id, det_pose)]
    s = capi.make_imu_stream(traj["t_imu"], dev[0].data_ptr(), B, capi.FBUS_MEM_DEVICE)
    d = capi.make_det_frames(traj["t_frames"], dev[1].data_ptr(), dev[2].data_ptr(), B, m, capi.FBUS_MEM_DEVICE)
    out = []
    for split in (None, W // 2):
        f = BatchFilter(_flags(bcfg, capi.FBUS_FLAG_ALL_MARKERS), batch=B)
        if split is None:
            f.StepWindows(s, d, traj["win_off"], 0, W)
        else:
            f.StepWindows(s, d, traj["win_off"], 0, split)
            f.StepWindows(s, d, traj["win_off"], split, W)
        out.append(f.GetState())
    for k in out[0]:
        assert np.array_equal(out[0][k], out[1][k]), k


def test_imu_f32_bitwise():
    """FBUS_IMU_F32_SENSOR samples give the same bits as the same values given as FBUS_IMU_F64_SI"""
    from fbus_ekf_b200 import BatchFilter, capi
    bcfg, traj, imu, det_id, det_pose = _board(B=40, seed=15)
    B, m, W = imu.shape[2], 8, len(traj["t_frames"])
    raw = np.ascontiguousarray(capi.si_to_sensor(imu, bcfg.imu_g).astype(np.float32))   # what the sensor would deliver
    si = np.ascontiguousarray(capi.sensor_to_si(raw, bcfg.imu_g))
    d = capi.make_det_frames(traj["t_frames"], det_id, det_pose, B, m)
    outs = []
    for data in (si, raw):
        f = BatchFilter(_flags(bcfg, capi.FBUS_FLAG_ALL_MARKERS), batch=B)
        f.StepWindows(capi.make_imu_stream(traj["t_imu"], data, B), d, traj["win_off"], 0, W)
        outs.append(f.GetState())
    for k in outs[0]:
        assert np.array_equal(outs[0][k], outs[1][k]), k


def test_per_filter_noise():
    """fbus_set_noise: every filter updates with its own R (and Q), as the oracle run with that filter's values"""
    from fbus_ekf_b200 import capi
    bcfg, traj, imu, det_id, det_pose = _board(B=32, seed=16)
    B = imu.shape[2]
    settings = []
    for j in range(2):
        c = copy.copy(bcfg)
        c.pos_n_cov, c.quat_n_cov = (1e-4, 1e-4) if j == 0 else (1e-6, 1e-5)
        c.accel_n_cov = bcfg.accel_n_cov * (1 + j)
        settings.append(c)
    noise = np.ascontiguousarray(np.array([[getattr(settings[b % 2], n) for b in range(B)] for n in capi.NOISE_FIELDS], dtype=np.float64))
    sg, _ = _gpu(bcfg, capi.FBUS_FLAG_ALL_MARKERS, traj, imu, det_id, det_pose, noise=noise)
    for j in range(2):
        so = _oracle(settings[j], capi.FBUS_FLAG_ALL_MARKERS, traj, imu, det_id, det_pose)
        idx = np.arange(j, B, 2)
        _check({k: v[..., idx] for k, v in sg.items()}, {k: v[..., idx] for k, v in so.items()}, n_whitened=2)


def test_matlab_combination_refused():
    from fbus_ekf_b200 import BatchFilter, FbusError, capi
    cfg = capi.config_matlab()
    cfg.flags |= capi.FBUS_FLAG_ALL_MARKERS
    with pytest.raises(FbusError):
        BatchFilter(cfg, batch=1)


def test_more_than_32_slots_refused():
    from fbus_ekf_b200 import BatchFilter, FbusError, capi, synth
    bcfg = synth.board_config(capi.config_default())
    traj = synth.truth_trajectory(bcfg, 0.2)
    W, N, m = len(traj["t_frames"]), len(traj["t_imu"]), 33
    imu = np.ascontiguousarray(np.repeat(traj["base_imu"][:, :, None], 2, axis=2))
    ids = np.full((W, m, 2), -1, dtype=np.int32)
    pose = np.zeros((W, m, 7, 2))
    s = capi.make_imu_stream(traj["t_imu"], imu, 2)
    d = capi.make_det_frames(traj["t_frames"], ids, pose, 2, m)
    with pytest.raises(FbusError):
        BatchFilter(_flags(bcfg, capi.FBUS_FLAG_ALL_MARKERS), batch=2).StepWindows(s, d, traj["win_off"], 0, W)
    BatchFilter(bcfg, batch=2).StepWindows(s, d, traj["win_off"], 0, W)   # the default mode takes any number of slots


def test_accuracy_board_monte_carlo(cfg):
    """4 096 Monte-Carlo runs of 3 s on the marker board (noisy corners -> refractive solve + Gauss-Newton -> EKF), fixed seeds:
    the final-frame position and attitude RMSE are lower with every marker than with the nearest one, by at least 10 %.  Every
    run must stay finite; the share of runs inside the chi-square(6) 95 % bound is printed with the RMSEs (line ACCURACY).
    Measured on an NVIDIA B200 (1000 W power limit): position RMSE 1.71e-3 m nearest-only -> 6.06e-4 m every marker (-64 %),
    attitude RMSE 1.66e-3 -> 9.56e-4 (-42 %); chi-square(6) 95 % share 1.0 in both modes."""
    from fbus_ekf_b200 import BatchFilter, capi, synth
    B, m = 4096, 8
    bcfg = synth.board_config(cfg)
    traj = synth.truth_trajectory(bcfg, 3.0, standoff=1.0)
    W, N = len(traj["t_frames"]), len(traj["t_imu"])
    base, ids, _ = synth.board_base_corners(bcfg, traj)
    rng = np.random.default_rng(2024)
    corners = np.ascontiguousarray((np.repeat(base, B, axis=1) + rng.normal(size=(16, W * m * B)) * 5e-4).astype(np.float32))
    mids = np.ascontiguousarray(np.repeat(ids[:, :, None], B, axis=2))
    imu = np.ascontiguousarray(traj["base_imu"][:, :, None] + rng.normal(size=(N, 6, B)) * np.array([0.015] * 3 + [1e-3] * 3)[None, :, None])
    f0 = BatchFilter(bcfg, batch=B)
    det_id, det_pose = f0.SolveToDetections(corners, mids, W, m, underwater=True, gn_iters=4)
    tp = np.ascontiguousarray(np.repeat(traj["truth_p"][-1][:, None], B, axis=1))
    tq = np.ascontiguousarray(np.repeat(traj["truth_q"][-1][:, None], B, axis=1))
    res = {}
    for name, flags in (("nearest", 0), ("all", capi.FBUS_FLAG_ALL_MARKERS)):
        f = BatchFilter(_flags(bcfg, flags), batch=B)
        s = capi.make_imu_stream(traj["t_imu"], imu, B)
        d = capi.make_det_frames(traj["t_frames"], det_id, det_pose, B, m)
        f.StepWindows(s, d, traj["win_off"], 0, W)
        e = f.FilterErrors(tp, tq)
        assert (e[3] != 0).all(), f"{name}: non-finite runs"
        res[name] = (float(np.sqrt(e[0].mean())), float(np.sqrt(e[1].mean())), float((e[2] <= 12.5916).mean()))
    print("ACCURACY", {k: dict(pos_rmse=v[0], att_rmse=v[1], nees_chi2_95_share=v[2]) for k, v in res.items()})
    assert res["all"][0] <= 0.9 * res["nearest"][0]
    assert res["all"][1] <= 0.9 * res["nearest"][1]
