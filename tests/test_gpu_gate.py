"""The innovation gate of fbus_set_gate on the GPU (include/fbus_ekf.h).  The gate runs on the first-generation lanes-per-filter
kernel at every batch size and is checked against its restatement on the NumPy oracle (tests/gate_ref.py) on corner-level board
workloads with outliers: fbus_synth_corners -> fbus_solve_to_detections -> fbus_step_windows.  Rejection counts and the status bit
must match bit for bit, with every reference NIS at least 1e-6 relative away from its threshold; state and covariance must match
at the suite's 1e-9."""
import copy
import os

import numpy as np
import pytest

from gate_ref import GatedFilter, stream_frames, stream_rows
from helpers import cov_close, cov_whitened_err, random_states, state_close
from test_gate_host import assert_margin

pytestmark = pytest.mark.gpu

LANE1 = {"FBUS_LANE": "1", "FBUS_LANE_GEN": "1"}
GATES = (16.81, 0.0, 24.32, 12.59, -1.0, 50.0, 18.48)  # per-filter thresholds, cycled: gated and ungated filters in one batch


def _make(cfg, flags=0, B=1, env=None):
    from fbus_ekf_b200 import BatchFilter
    c = copy.copy(cfg)
    c.flags = flags
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        return BatchFilter(c, batch=B)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _workload(n, seed, duration=0.6, p_outlier=0.08, sigma_outlier=5e-3):
    """n distinct filters of the board workload: corners with outliers from fbus_synth_corners, solved on the device (refractive
    solve + 5 Gauss-Newton iterations) into detections, and noisy IMU samples (SI doubles)"""
    import torch
    from fbus_ekf_b200 import capi, synth
    bcfg = synth.board_config(capi.config_default())
    traj = synth.truth_trajectory(bcfg, duration, standoff=1.0)
    W, N = len(traj["t_frames"]), len(traj["t_imu"])
    mpose, mids = synth.base_marker_poses(bcfg, traj)
    m = mpose.shape[1]
    spec = synth.make_corner_spec(mpose, mids, seed=seed, underwater=True, p_drop=0.05, p_outlier=p_outlier, sigma_outlier=sigma_outlier)
    f = _make(bcfg, 0, n)
    c_d = torch.empty((16, W * m * n), dtype=torch.float32, device="cuda")
    cid_d = torch.empty((W, m, n), dtype=torch.int32, device="cuda")
    f.SynthCorners(spec, 0, W, c_d.data_ptr(), cid_d.data_ptr())
    f.Synchronize()
    det_id, det_pose = f.SolveToDetections(np.ascontiguousarray(c_d.cpu().numpy()), np.ascontiguousarray(cid_d.cpu().numpy()), W, m,
                                           underwater=True, gn_iters=5)
    rng = np.random.default_rng(seed)
    imu = np.ascontiguousarray(traj["base_imu"][:, :, None] + rng.normal(size=(N, 6, n)) * np.array([0.015] * 3 + [1e-3] * 3)[None, :, None])
    return bcfg, traj, imu, det_id, det_pose


def _np_consts(bcfg, noise=None, b=0):
    """the NumPy oracle's constants for a capi config, with filter b's column of a [6][n] noise array if given"""
    import fbus_oracle_np as onp
    from test_all_markers_host import _np_config
    c = _np_config(bcfg)
    c.accel_n_cov, c.gyro_n_cov, c.accel_b_cov, c.gyro_b_cov, c.pos_n_cov, c.quat_n_cov = (
        bcfg.accel_n_cov, bcfg.gyro_n_cov, bcfg.accel_b_cov, bcfg.gyro_b_cov, bcfg.pos_n_cov, bcfg.quat_n_cov)
    if noise is not None:
        c.accel_n_cov, c.gyro_n_cov, c.accel_b_cov, c.gyro_b_cov, c.pos_n_cov, c.quat_n_cov = (float(x) for x in noise[:, b])
    return onp.Consts(c)


def _reference(bcfg, traj, imu, det_id, det_pose, gates, joseph, all_markers, noise=None, w_split=None):
    """the restatement for every filter of the workload; w_split = (w, gates2): the thresholds change to gates2 before frame w"""
    W = len(traj["t_frames"])
    out = []
    for b in range(imu.shape[2]):
        g = GatedFilter(_np_consts(bcfg, noise, b), gates[b], joseph, all_markers)
        rows, frames = stream_rows(traj["t_imu"], imu, b), stream_frames(traj["t_frames"], det_id, det_pose, b)
        if w_split is None:
            g.step(rows, frames, traj["win_off"], 0, W)
        else:
            g.step(rows, frames, traj["win_off"], 0, w_split[0])
            g.rejected, g.gate = 0, w_split[1][b]
            g.step(rows, frames, traj["win_off"], w_split[0], W)
        assert_margin(g.log)
        out.append(g)
    return out


def _compare(sg, rej, refs, n_whitened=3):
    """device state sg / counts rej of B filters against the restatement of n distinct ones (filter b has the inputs of b % n)"""
    from fbus_ekf_b200 import capi
    n = len(refs)
    B = rej.shape[0]
    fields = ("t", "q", "p", "v", "ba", "bg", "g")
    ref = {"t": np.array([[g.f.t for g in refs]])}
    for k in fields[1:]:
        ref[k] = np.stack([getattr(g.f, k) for g in refs], axis=1)
    Pref = np.stack([g.f.P.reshape(324) for g in refs], axis=1)
    idx = np.arange(B) % n
    assert np.array_equal(rej, np.array([g.rejected for g in refs], dtype=np.int32)[idx])
    assert np.array_equal((sg["status"] & capi.FBUS_ST_UPDATE_REJECTED) != 0, np.array([g.flag for g in refs])[idx])
    assert np.array_equal(sg["prev_marker_id"], np.array([g.f.prev_marker_id for g in refs], dtype=np.int32)[idx])
    for part in range(0, B, n):
        sl = slice(part, min(part + n, B))
        k = sl.stop - sl.start
        ok, worst = state_close({f: sg[f][..., sl] for f in fields}, {f: ref[f][..., :k] for f in fields}, 1e-9, fields=fields)
        assert ok, worst
        ok, worst = cov_close(sg["P"][:, sl], Pref[:, :k], 1e-9)
        assert ok, worst
    for b in range(min(n_whitened, n)):
        assert cov_whitened_err(sg["P"][:, b], Pref[:, b]) <= 1e-9


@pytest.mark.parametrize("B, joseph, all_markers, imu32, noise", [
    (1, False, False, False, False),
    (33, True, True, False, True),
    (33, False, True, True, False),
    (33, True, False, True, True),
    (4096, False, False, False, True),
    (4096, True, True, True, False),
])
def test_corner_pipeline_against_restatement(B, joseph, all_markers, imu32, noise):
    from fbus_ekf_b200 import capi
    n = min(B, 40)
    bcfg, traj, imu, det_id, det_pose = _workload(n, seed=100 + B + 2 * joseph + 4 * all_markers)
    W, m = len(traj["t_frames"]), det_id.shape[1]
    # the corner sweep's consistent setting of each mode: with the default (1e-3, 1e-3) hardly an update fails a threshold
    bcfg.pos_n_cov, bcfg.quat_n_cov = 1e-6, (1e-6 if all_markers else 1e-3)
    gates = np.array([GATES[b % len(GATES)] for b in range(n)])
    nz = None
    if noise:  # pos_n_cov 1e-6 with two quat_n_cov values, alternating, and the config's IMU noise; every marker diverges with
        # quat_n_cov > pos_n_cov (DESIGN.md §7), so that mode gets 1e-7 in place of the nearest marker's consistent 1e-3
        nz = np.array([[bcfg.accel_n_cov] * n, [bcfg.gyro_n_cov] * n, [bcfg.accel_b_cov] * n, [bcfg.gyro_b_cov] * n, [1e-6] * n,
                       [(1e-7 if all_markers else 1e-3) if b % 2 else 1e-6 for b in range(n)]])
    if imu32:  # the filter and the restatement see the same SI doubles (capi.sensor_to_si is the kernels' conversion)
        raw = capi.si_to_sensor(imu, bcfg.imu_g)
        imu = np.ascontiguousarray(capi.sensor_to_si(raw, bcfg.imu_g))
    refs = _reference(bcfg, traj, imu, det_id, det_pose, gates, joseph, all_markers, nz)
    assert any(g.log for g in refs) and (n == 1 or sum(g.rejected for g in refs) > 0)
    reps = (B + n - 1) // n
    til = lambda a: np.ascontiguousarray(np.concatenate([a] * reps, axis=-1)[..., :B])
    flags = (capi.FBUS_FLAG_JOSEPH if joseph else 0) | (capi.FBUS_FLAG_ALL_MARKERS if all_markers else 0)
    f = _make(bcfg, flags, B)
    if nz is not None:
        f.SetNoise(til(nz))
    f.SetGate(til(gates))
    s = capi.make_imu_stream(traj["t_imu"], til(raw) if imu32 else til(imu), B)
    d = capi.make_det_frames(traj["t_frames"], til(det_id), til(det_pose), B, m)
    f.StepWindows(s, d, traj["win_off"], 0, W)
    sg = f.GetState()
    _compare(sg, f.RejectedUpdates(), refs)
    # every other status bit is the ungated run's
    f0 = _make(bcfg, flags, B, LANE1)
    if nz is not None:
        f0.SetNoise(til(nz))
    f0.StepWindows(s, d, traj["win_off"], 0, W)
    assert np.array_equal(sg["status"] & ~capi.FBUS_ST_UPDATE_REJECTED, f0.GetState(with_cov=False)["status"])


@pytest.mark.parametrize("all_markers", [False, True])
def test_zero_gates_bitwise_default_and_null_restores(all_markers):
    """all thresholds 0: bit for bit the default mode on the same kernel; fbus_set_gate(NULL) afterwards: bit for bit a handle
    that never had a gate"""
    from fbus_ekf_b200 import capi
    bcfg, traj, imu, det_id, det_pose = _workload(40, seed=7)
    B, W, m = 40, len(traj["t_frames"]), det_id.shape[1]
    flags = capi.FBUS_FLAG_ALL_MARKERS if all_markers else 0
    s = capi.make_imu_stream(traj["t_imu"], imu, B)
    d = capi.make_det_frames(traj["t_frames"], det_id, det_pose, B, m)
    ref = _make(bcfg, flags, B, LANE1)
    t_ref = ref.StepWindows(s, d, traj["win_off"], 0, W, trace=True)
    gated = _make(bcfg, flags, B, LANE1)
    gated.SetGate(np.zeros(B))
    t_g = gated.StepWindows(s, d, traj["win_off"], 0, W, trace=True)
    a, b = ref.GetState(), gated.GetState()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(t_ref, t_g) and not gated.RejectedUpdates().any()
    # a gate that rejects, then NULL: the second half runs as on a handle that never had a gate
    h1, h2 = _make(bcfg, flags, B, LANE1), _make(bcfg, flags, B, LANE1)
    h1.SetGate(np.full(B, 1e-30))
    h1.SetGate(None)
    h1.StepWindows(s, d, traj["win_off"], 0, W)
    h2.StepWindows(s, d, traj["win_off"], 0, W)
    a, b = h1.GetState(), h2.GetState()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert not h1.RejectedUpdates().any()  # the counts stay readable after NULL


def test_unfused_update_reject_all():
    """fbus_update with a threshold no update passes: state and covariance bitwise unchanged, the status bit, a count of 1 and
    prev_marker_id of the chosen marker"""
    from fbus_ekf_b200 import capi
    import fbus_oracle_np as onp
    from test_all_markers_host import _dets_at, _np_filter
    cfg = capi.config_default()
    B = 5
    st = random_states(B, np.random.default_rng(13))
    st["prev_marker_id"][:] = 7
    k = onp.Consts(onp.default_config())
    ids = np.zeros((1, 2, B), dtype=np.int32)
    pose = np.zeros((1, 2, 7, B))
    for b in range(B):
        dets = _dets_at(_np_filter(k, {n: v[..., b:b + 1] for n, v in st.items()}), [(1, 0.9), (3, 0.7)], seed=b)
        for sl, dd in enumerate(dets):
            ids[0, sl, b], pose[0, sl, :, b] = int(dd[0]), dd[1:8]
    f = _make(cfg, 0, B)
    f.SetState(st)
    f.SetGate(np.full(B, 1e-30))
    before = f.GetState()
    f.MeasureUpdate(capi.make_det_frames(np.array([st["t"][0]]), ids, pose, B, 2), 0)
    after = f.GetState()
    for n in ("t", "q", "R", "p", "v", "ba", "bg", "g", "P"):
        assert np.array_equal(before[n], after[n]), n
    assert (after["status"] & capi.FBUS_ST_UPDATE_REJECTED).all() and np.array_equal(f.RejectedUpdates(), np.ones(B, dtype=np.int32))
    assert (after["prev_marker_id"] == 3).all()  # the nearer marker, chosen before the gate


def test_continuation_and_count_reset():
    """device-resident streams stepped in two continued calls: the same as one call, thresholds changed between the calls take
    effect from the next call, and fbus_set_gate resets the counts"""
    import torch
    from fbus_ekf_b200 import capi
    n = 24
    bcfg, traj, imu, det_id, det_pose = _workload(n, seed=31, duration=0.8)
    W, m, a = len(traj["t_frames"]), det_id.shape[1], 9
    g1 = np.array([GATES[b % len(GATES)] for b in range(n)])
    g2 = np.roll(g1, 3)
    imu_d, id_d, pose_d = (torch.from_numpy(x).cuda() for x in (imu, det_id, det_pose))
    s = capi.make_imu_stream(traj["t_imu"], imu_d.data_ptr(), n, capi.FBUS_MEM_DEVICE)
    d = capi.make_det_frames(traj["t_frames"], id_d.data_ptr(), pose_d.data_ptr(), n, m, capi.FBUS_MEM_DEVICE)
    one, two = _make(bcfg, 0, n), _make(bcfg, 0, n)
    one.SetGate(g1)
    one.StepWindows(s, d, traj["win_off"], 0, W)
    two.SetGate(g1)
    two.StepWindows(s, d, traj["win_off"], 0, a)
    two.StepWindows(s, d, traj["win_off"], a, W)
    x, y = one.GetState(), two.GetState()
    for k in x:
        assert np.array_equal(x[k], y[k]), k
    assert np.array_equal(one.RejectedUpdates(), two.RejectedUpdates())
    _compare(x, one.RejectedUpdates(), _reference(bcfg, traj, imu, det_id, det_pose, g1, False, False))
    # new thresholds between two continued calls: counted from the call on, the state continues
    three = _make(bcfg, 0, n)
    three.SetGate(g1)
    three.StepWindows(s, d, traj["win_off"], 0, a)
    three.SetGate(g2)
    assert not three.RejectedUpdates().any()
    three.StepWindows(s, d, traj["win_off"], a, W)
    _compare(three.GetState(), three.RejectedUpdates(),
             _reference(bcfg, traj, imu, det_id, det_pose, g1, False, False, w_split=(a, g2)))


def test_bad_arguments():
    from fbus_ekf_b200 import FbusError, capi
    lib = capi.lib()
    cfg = capi.config_default()
    f = _make(cfg, 0, 4)
    gate = np.full(4, 16.81)
    out = np.zeros(4, dtype=np.int32)
    assert lib.fbus_rejected_updates(f._h, out.ctypes.data, capi.FBUS_MEM_HOST) == capi.FBUS_E_STATE
    for mem in (2, -1):
        assert lib.fbus_set_gate(f._h, gate.ctypes.data, mem) == capi.FBUS_E_BADARG
        assert b"memory kind" in lib.fbus_last_error(f._h)
        assert lib.fbus_rejected_updates(f._h, out.ctypes.data, capi.FBUS_MEM_HOST) == capi.FBUS_E_STATE  # no effect
    f.SetGate(gate)
    for mem in (2, -1):
        assert lib.fbus_rejected_updates(f._h, out.ctypes.data, mem) == capi.FBUS_E_BADARG
    assert lib.fbus_rejected_updates(f._h, out.ctypes.data, capi.FBUS_MEM_HOST) == capi.FBUS_OK and not out.any()
    mcfg = capi.config_matlab()
    fm = _make(mcfg, mcfg.flags, 4)
    with pytest.raises(FbusError):
        fm.SetGate(gate)
    assert lib.fbus_set_gate(fm._h, None, capi.FBUS_MEM_HOST) == capi.FBUS_E_BADARG


def _mc_rmse(all_markers, quat_n_cov, gates, p_outlier, B=4096, duration=3.0, seed=5):
    """final position RMSE of B board runs for each threshold in `gates` (0: no gate), all on the same streams: IMU from
    fbus_synth_streams, corners from fbus_synth_corners (sigma_outlier 25x the corner noise), solved on the device"""
    import torch
    from fbus_ekf_b200 import capi, synth
    cfg = synth.board_config(capi.config_default())
    cfg.pos_n_cov, cfg.quat_n_cov = 1e-6, quat_n_cov
    flags = capi.FBUS_FLAG_ALL_MARKERS if all_markers else 0
    traj = synth.truth_trajectory(cfg, duration, standoff=1.0)
    N, W = len(traj["t_imu"]), len(traj["t_frames"])
    mpose, mids = synth.base_marker_poses(cfg, traj)
    m = mpose.shape[1]
    f = _make(cfg, flags, B)
    imu_d = torch.empty((N, 6, B), dtype=torch.float64, device="cuda")
    tmp_id = torch.empty((W, 1, B), dtype=torch.int32, device="cuda")
    tmp_pose = torch.empty((W, 1, 7, B), dtype=torch.float64, device="cuda")
    f.SynthStreams(synth.make_synth_spec(traj, seed=seed), imu_d.data_ptr(), tmp_id.data_ptr(), tmp_pose.data_ptr())
    spec = synth.make_corner_spec(mpose, mids, seed=seed, p_outlier=p_outlier, sigma_outlier=25 * synth.DEFAULT_CORNER_NOISE)
    c_d = torch.empty((16, W * m * B), dtype=torch.float32, device="cuda")
    cid_d = torch.empty((W, m, B), dtype=torch.int32, device="cuda")
    f.SynthCorners(spec, 0, W, c_d.data_ptr(), cid_d.data_ptr())
    id_d = torch.empty((W, m, B), dtype=torch.int32, device="cuda")
    pose_d = torch.empty((W, m, 7, B), dtype=torch.float64, device="cuda")
    f.SolveToDetections(c_d.data_ptr(), cid_d.data_ptr(), W, m, True, 5, id_d.data_ptr(), pose_d.data_ptr(), capi.FBUS_MEM_DEVICE)
    f.Synchronize()
    s = capi.make_imu_stream(traj["t_imu"], imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE)
    d = capi.make_det_frames(traj["t_frames"], id_d.data_ptr(), pose_d.data_ptr(), B, m, capi.FBUS_MEM_DEVICE)
    tp = np.ascontiguousarray(np.repeat(traj["truth_p"][-1][:, None], B, axis=1))
    tq = np.ascontiguousarray(np.repeat(traj["truth_q"][-1][:, None], B, axis=1))
    out = {}
    for g in gates:
        h = _make(cfg, flags, B)
        if g > 0:
            h.SetGate(np.full(B, g))
        h.StepWindows(s, d, traj["win_off"], 0, W)
        e = h.FilterErrors(tp, tq)
        ok = e[3] == 1.0  # as the sweep scores: RMSE over the finite runs, and the count of the others
        out[g] = (float(np.sqrt(e[0][ok].mean())), int((~ok).sum()), float(h.RejectedUpdates().mean()) if g > 0 else 0.0)
    return out


@pytest.mark.parametrize("all_markers, quat_n_cov, gate", [(False, 1e-3, 50.0), (True, 1e-6, 1000.0)])
def test_monte_carlo_gate_lowers_rmse(all_markers, quat_n_cov, gate):
    """4,096 board runs of 3 s with corner outliers (p_outlier 0.05, sigma_outlier 25x the corner noise), at the corner sweep's
    consistent setting of each fusion mode, the same runs with and without the gate: the gate lowers the final position RMSE.
    The table's thresholds are printed too: a filter initialised from an outlier pose (init is not gated) can reject every later
    update, and such runs dominate the RMSE at the tighter thresholds."""
    res = _mc_rmse(all_markers, quat_n_cov, (0.0, 16.81, 24.32, 50.0, 1000.0), 0.05)
    clean = _mc_rmse(all_markers, quat_n_cov, (0.0,), 0.0)
    print(f"all_markers={all_markers}: outlier-free {clean[0.0][0]:.3e} m ({clean[0.0][1]} non-finite); " +
          ", ".join(f"gate {g}: {r:.3e} m ({nf} non-finite, {n:.2f} rejected per run)" for g, (r, nf, n) in res.items()))
    assert res[gate][0] < res[0.0][0] and res[gate][1] <= res[0.0][1] and res[gate][2] > 0
