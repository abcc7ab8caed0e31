"""The innovation gate of fbus_set_gate (include/fbus_ekf.h) in its reference restatement (tests/gate_ref.py), and the sweep's
gate_chi2 dimension.  No GPU: the restatement against the two oracles, the rules on hand-built frames, the gate's calibration on
outlier-free pose-level streams, and the sweep's argument parsing, layout and rows."""
import copy
import json
import math

import numpy as np
import pytest

from all_markers_ref import OrcAllMarkers, np_chosen_index, np_update_with
from gate_ref import GatedFilter, nis, rejects, replay_gated, stream_frames, stream_rows
from helpers import cov_close, state_close
from test_all_markers_host import _board, _dets_at, _hand_state, _np_config, _np_filter

pytestmark = pytest.mark.usefixtures("built")

CHI2_7_999 = 24.32  # the 0.999 quantile of chi-square(7), the loosest threshold of the header's table


def assert_margin(log, rel=1e-6):
    """every tested NIS is at least `rel` relative away from its threshold, so that a rounding-level difference between two
    evaluations of the NIS cannot flip a decision"""
    for v, g in log:
        assert not math.isfinite(v) or abs(v - g) >= rel * g, (v, g)


def _replay_inputs(duration=2.0, seed=3):
    """replay input (imu rows [t, accel, gyro], image rows [t, id, p, q]) of a noisy synthetic run in front of marker 0"""
    from fbus_ekf_b200 import capi, synth
    cfg = capi.config_default()
    traj = synth.truth_trajectory(cfg, duration)
    rng = np.random.default_rng(seed)
    imu = traj["base_imu"] + rng.normal(size=traj["base_imu"].shape) * np.array([0.015] * 3 + [1e-3] * 3)
    imu_rows = np.concatenate([traj["t_imu"][:, None], imu], axis=1)
    pose = traj["base_pose"] + rng.normal(size=traj["base_pose"].shape) * np.array([2.5e-4] * 3 + [1.5e-3] * 4)
    image_rows = np.concatenate([traj["t_frames"][:, None], np.full((len(pose), 1), float(traj["marker_id"])), pose], axis=1)
    return imu_rows, image_rows


@pytest.mark.parametrize("gate", [0.0, -1.0, float("nan")])
def test_no_gate_is_replay_bitwise(gate):
    """a threshold <= 0 or NaN gates nothing: the restatement is fbus_oracle_np.replay bit for bit"""
    import fbus_oracle_np as onp
    imu, image_rows = _replay_inputs()
    cfg = onp.default_config()
    ref = onp.replay(cfg, imu, image_rows, n_init=20)
    got = replay_gated(cfg, imu, image_rows, gate, n_init=20)
    assert np.array_equal(got["rows"], ref["rows"])
    assert np.array_equal(got["gated"].f.P, ref["filter"].P)
    assert got["gated"].rejected == 0 and got["gated"].log == []


@pytest.mark.parametrize("joseph, all_markers", [(False, False), (True, False), (False, True), (True, True)])
def test_accept_all_equals_cpp_oracle(joseph, all_markers):
    """a threshold every update passes: the restatement agrees with the C++ oracle (the suite's 1e-9)"""
    import orc
    import fbus_oracle_np as onp
    from fbus_ekf_b200 import capi
    bcfg, traj, imu, det_id, det_pose = _board()
    B, m, W = imu.shape[2], det_id.shape[1], len(traj["t_frames"])
    c = copy.copy(bcfg)
    c.flags = (capi.FBUS_FLAG_JOSEPH if joseph else 0) | (capi.FBUS_FLAG_ALL_MARKERS if all_markers else 0)
    if all_markers:
        o = OrcAllMarkers(c, B)
        o.step_windows(traj["t_imu"], imu, traj["t_frames"], det_id, det_pose, traj["win_off"], 0, W)
    else:
        o = orc.Oracle(c, B)
        o.step_windows(capi.make_imu_stream(traj["t_imu"], imu, B), capi.make_det_frames(traj["t_frames"], det_id, det_pose, B, m),
                       traj["win_off"], 0, W)
    so = o.get_state()
    k = onp.Consts(_np_config(bcfg))
    for b in range(B):
        g = GatedFilter(k, 1e6, joseph, all_markers)
        g.step(stream_rows(traj["t_imu"], imu, b), stream_frames(traj["t_frames"], det_id, det_pose, b), traj["win_off"], 0, W)
        assert g.rejected == 0 and len(g.log) >= W - 1
        assert_margin(g.log)
        f = g.f
        st = {"t": np.array([f.t]), "q": f.q, "p": f.p, "v": f.v, "ba": f.ba, "bg": f.bg, "g": f.g}
        assert state_close({n: so[n][..., b] for n in st}, st, 1e-9, fields=tuple(st))[0]
        assert cov_close(so["P"][:, b:b + 1], f.P.reshape(324, 1), 1e-9)[0]
        assert so["prev_marker_id"][b] == f.prev_marker_id


def _propagate_only(k, rows, frames, off):
    """the frame loop with every update rejected: init, reset and propagation, and the marker choice of each update"""
    import fbus_oracle_np as onp
    f = onp.Filter(k)
    cursor = int(off[0])
    for w, (t_det, dets) in enumerate(frames):
        hi = int(off[w + 1])
        if not dets:
            continue
        if not f.initialised:
            later = np.nonzero(rows[cursor:hi, 0] > t_det)[0]
            cnt = int(later[0]) if len(later) else hi - cursor
            if f.init_pose(dets, t_det, cnt):
                cursor += cnt
        else:
            f.reset_state(dets, t_det)
            cursor += f.batch_imu(rows[cursor:hi], t_det)
            d = dets[np_chosen_index(f, dets)]
            if int(d[0]) in k.markers:
                f.prev_marker_id = int(d[0])
    return f


@pytest.mark.parametrize("all_markers", [False, True])
def test_rejected_update_leaves_the_propagated_state(all_markers):
    """a threshold no update passes: the result is the propagated state bit for bit, every update counted"""
    import fbus_oracle_np as onp
    bcfg, traj, imu, det_id, det_pose = _board(B=2)
    k = onp.Consts(_np_config(bcfg))
    W = len(traj["t_frames"])
    for b in range(2):
        rows, frames = stream_rows(traj["t_imu"], imu, b), stream_frames(traj["t_frames"], det_id, det_pose, b)
        g = GatedFilter(k, 1e-30, False, all_markers)
        g.step(rows, frames, traj["win_off"], 0, W)
        ref = _propagate_only(k, rows, frames, traj["win_off"])
        for name in ("t", "q", "p", "v", "ba", "bg", "g", "P", "prev_marker_id"):
            assert np.array_equal(getattr(g.f, name), getattr(ref, name)), name
        n_updates = sum(len([d for d in dets if int(d[0]) in k.markers]) if all_markers else 1 for _, dets in frames[1:] if dets)
        assert g.flag and g.rejected == n_updates and len(g.log) == n_updates


def test_prev_marker_id_after_a_rejected_chosen_marker():
    """the marker choice comes before the gate: a rejected chosen marker still becomes prev_marker_id (here by hysteresis)"""
    cfg, k, st = _hand_state()
    st["prev_marker_id"][0] = 2
    f = _np_filter(k, st)
    dets = _dets_at(f, [(2, 1.0), (1, 0.8)])
    assert np_chosen_index(f, dets) == 0
    g = GatedFilter(k, 1e-30)
    g.f = f
    P0, p0 = f.P.copy(), f.p.copy()
    g.update(dets)
    assert f.prev_marker_id == 2 and g.rejected == 1 and np.array_equal(f.P, P0) and np.array_equal(f.p, p0)
    # without hysteresis the nearest marker is chosen, and becomes prev_marker_id although rejected
    f.prev_marker_id = 5
    g.update(dets)
    assert f.prev_marker_id == 1 and g.rejected == 2 and np.array_equal(f.P, P0)


def _predicted_dets(f, ids, seed):
    """detections of markers `ids` where filter f predicts them, with 1e-4 of noise"""
    rng = np.random.default_rng(seed)
    out = []
    for mid in ids:
        d = np.zeros(8)
        d[0] = mid
        hP, hQ, _ = f.measurement_model(d)
        q = hQ + rng.normal(size=4) * 1e-4
        d[1:4], d[4:8] = hP + rng.normal(size=3) * 1e-4, q / np.linalg.norm(q)
        out.append(d)
    return out


def test_all_markers_gates_each_update_in_order():
    """under FBUS_FLAG_ALL_MARKERS each update is gated on its own: a rejected chosen marker does not stop the further slots, which
    follow in slot order"""
    cfg, k, st = _hand_state(6)
    st["prev_marker_id"][0] = 5
    st["P"] *= 1e-4
    f = _np_filter(k, st)
    dets = _predicted_dets(f, [2, 1, 3], seed=2)
    dets[1][1:4] += 0.3  # the chosen (nearest) marker is a 30 cm outlier
    assert np_chosen_index(f, dets) == 1
    g = GatedFilter(k, CHI2_7_999, all_markers=True)
    g.f = f
    g.update(dets)
    assert_margin(g.log)
    assert g.rejected == 1 and len(g.log) == 3 and g.log[0][0] > CHI2_7_999 and all(v < CHI2_7_999 for v, _ in g.log[1:])
    ref = _np_filter(k, st)
    np_update_with(ref, dets[0])
    np_update_with(ref, dets[2])
    assert np.array_equal(f.p, ref.p) and np.array_equal(f.q, ref.q) and np.array_equal(f.P, ref.P)
    assert f.prev_marker_id == 1


def test_nan_nis_is_rejected():
    assert rejects(16.81, float("nan")) and rejects(16.81, float("inf"))
    assert not rejects(0.0, float("nan")) and not rejects(float("nan"), 1e9) and not rejects(-1.0, 1e9)
    assert not rejects(5.0, 5.0) and rejects(5.0, np.nextafter(5.0, 6.0))
    cfg, k, st = _hand_state(7)
    f = _np_filter(k, st)
    d = _dets_at(f, [(1, 0.9)])[0]
    d[5] = np.nan
    assert math.isnan(nis(f, d))
    g = GatedFilter(k, 16.81)
    g.f = f
    p0, P0 = f.p.copy(), f.P.copy()
    g.update([d])
    assert g.rejected == 1 and np.array_equal(f.p, p0) and np.array_equal(f.P, P0)


# The false rejections of the loosest threshold in the table on outlier-free pose-level streams (synth.DEFAULT_NOISE on the
# trajectory of the noise sweep) at the setting the pose-level sweep finds consistent by NEES, pos_n_cov = 1e-6, quat_n_cov = 1e-3.
# Measured: 0 of 1,184 updates (16 filters x 74 updates); mean NIS 0.037, 99th percentile 0.17, largest 0.54.  The NIS sits far
# below chi-square(7) because quat_n_cov = 1e-3 overstates the quaternion noise of these streams (1.5e-3 std, 2.25e-6
# variance) 400-fold, so at this setting the gate only meets gross errors.  The bounds keep 10x headroom.
def test_calibration_on_outlier_free_pose_streams():
    import fbus_oracle_np as onp
    from fbus_ekf_b200 import capi, synth
    cfg = capi.config_default()
    traj = synth.truth_trajectory(cfg, 3.0)
    ncfg = onp.default_config()
    ncfg.pos_n_cov, ncfg.quat_n_cov = 1e-6, 1e-3
    k = onp.Consts(ncfg)
    nz = synth.DEFAULT_NOISE
    rng = np.random.default_rng(21)
    W = len(traj["t_frames"])
    n_upd = n_rej = 0
    worst = 0.0
    for b in range(16):
        bias = np.concatenate([rng.normal(size=3) * nz["sigma_ba"], rng.normal(size=3) * nz["sigma_bg"]])
        imu = traj["base_imu"] + bias + rng.normal(size=traj["base_imu"].shape) * np.array([nz["sigma_acc"]] * 3 + [nz["sigma_gyro"]] * 3)
        pose = traj["base_pose"] + rng.normal(size=traj["base_pose"].shape) * np.array([nz["sigma_pos"]] * 3 + [nz["sigma_quat"]] * 4)
        frames = [(float(traj["t_frames"][w]), [np.concatenate([[traj["marker_id"]], pose[w]])]) for w in range(W)]
        g = GatedFilter(k, CHI2_7_999)
        g.step(np.concatenate([traj["t_imu"][:, None], imu], axis=1), frames, traj["win_off"], 0, W)
        n_upd += len(g.log)
        n_rej += g.rejected
        worst = max(worst, max(v for v, _ in g.log))
    assert n_upd == 16 * (W - 1)
    assert n_rej / n_upd <= 0.005 and worst <= 5.0, (n_rej, worst)


# ------------------------------------------------------------------------------------------------------------ the sweep
BASE = dict(zip(("accel_n_cov", "gyro_n_cov", "accel_b_cov", "gyro_b_cov", "pos_n_cov", "quat_n_cov"), (1e-3, 1e-4, 1e-3, 1e-4, 1e-3, 1e-3)))


def test_sweep_gate_dimension_and_layout():
    from fbus_ekf_b200 import capi, sweep
    sets = sweep.parse_sets(["pos_n_cov=1e-6,1e-5", "gate_chi2=0,16.81,24.32"])
    assert sets == [("pos_n_cov", [1e-6, 1e-5]), ("gate_chi2", [0.0, 16.81, 24.32])]
    grid = sweep.expand_grid(sets, BASE)
    assert len(grid) == 6 and [(s["pos_n_cov"], s["gate_chi2"]) for s in grid] == [
        (1e-6, 0.0), (1e-6, 16.81), (1e-6, 24.32), (1e-5, 0.0), (1e-5, 16.81), (1e-5, 24.32)]
    assert list(grid[0]) == list(capi.NOISE_FIELDS) + ["gate_chi2"]
    runs = 4
    gate = sweep.gate_array(grid, runs)
    assert gate.shape == (24,) and gate.dtype == np.float64 and gate.flags["C_CONTIGUOUS"]
    b = np.arange(24)
    assert np.array_equal(gate, np.array([s["gate_chi2"] for s in grid])[sweep.setting_of(b, runs)])
    # the noise array ignores the gate dimension
    assert np.array_equal(sweep.noise_array(grid, runs)[capi.NOISE_FIELDS.index("pos_n_cov")], np.repeat([1e-6] * 3 + [1e-5] * 3, runs))
    # without the dimension: no gate, and the settings are the six noise values only
    grid0 = sweep.expand_grid(sweep.parse_sets(["pos_n_cov=1e-6"]), BASE)
    assert sweep.gate_array(grid0, runs) is None and list(grid0[0]) == list(capi.NOISE_FIELDS)
    with pytest.raises(ValueError):
        sweep.parse_sets(["gate_chi2=1", "gate_chi2=2"])
    with pytest.raises(ValueError):
        sweep.parse_sets(["gate=16.81"])


def test_sweep_rows_without_gate_are_unchanged():
    """without gate_chi2 in --set the rows are byte for byte the format before the gate existed"""
    from fbus_ekf_b200 import sweep
    grid = sweep.expand_grid(sweep.parse_sets(["quat_n_cov=1e-3,1e-4"]), BASE)
    red = np.arange(2 * 5 * 2, dtype=np.float64).reshape(2, 5, 2) + 0.25
    rows = sweep._rows(grid, 8, red, [1.0, 2.0])
    expected = ('{"accel_n_cov": 0.001, "gyro_n_cov": 0.0001, "accel_b_cov": 0.001, "gyro_b_cov": 0.0001, "pos_n_cov": 0.001, '
                '"quat_n_cov": 0.001, "runs": 8, "rmse_pos_m": %r, "rmse_att_rad": %r, "t_eval": [1.0, 2.0], "nees6_mean": [4.25, 14.25], '
                '"frac_nees6_le_12.59": 16.25, "n_nonfinite": 18}' % (math.sqrt(10.25), math.sqrt(12.25)))
    assert json.dumps(rows[0]) == expected
    gated = sweep._rows(sweep.expand_grid(sweep.parse_sets(["quat_n_cov=1e-3,1e-4", "gate_chi2=24.32"]), BASE), 8, red, [1.0, 2.0],
                        np.array([0.5, 1.25]))
    assert list(gated[1])[-2:] == ["n_nonfinite", "rejected_per_run"] and gated[1]["rejected_per_run"] == 1.25
    assert gated[0]["gate_chi2"] == 24.32 and list(gated[0])[6] == "gate_chi2"


def test_sweep_help_names_the_gate():
    import subprocess
    import sys
    from test_sweep_host import ROOT
    r = subprocess.run([sys.executable, "-m", "fbus_ekf_b200.sweep", "--help"], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0 and "gate_chi2" in r.stdout
