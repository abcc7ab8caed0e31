"""FBUS_FLAG_ALL_MARKERS in the reference restatements of tests/all_markers_ref.py (include/fbus_ekf.h): every known marker of a
frame updates the filter in turn, the reference's chosen marker first, then the other slots in slot order.  The restatements on
the C++ oracle (orc) and on the NumPy oracle must agree on the marker-board workload; hand-built frames pin the order, the
unknown-id rules and the status bit."""
import copy

import numpy as np
import pytest

from all_markers_ref import OrcAllMarkers, np_observation_update_all, np_update_with
from helpers import random_states


def _np_config(bcfg):
    """the NumPy oracle's Config for a capi config (extrinsics, marker map; every other constant is the default in both)"""
    import fbus_oracle_np as onp
    markers = {int(bcfg.marker_id[m]): (np.array(bcfg.marker_pos[3 * m:3 * m + 3], dtype=np.float64),
                                        np.array(bcfg.marker_rot[9 * m:9 * m + 9], dtype=np.float64).reshape(3, 3))
               for m in range(bcfg.n_markers)}
    return onp.Config(tsc_left=np.array(bcfg.tsc_left).reshape(4, 4), tsc_right=np.array(bcfg.tsc_right).reshape(4, 4),
                      markers=markers)


def _np_step_windows(k, t_imu, imu, t_frames, det_id, det_pose, win_off, b, joseph, all_markers):
    """orc_step_windows for filter b, on the NumPy oracle (the loop of fbus_oracle_np.replay on detection frames)"""
    import fbus_oracle_np as onp
    f = onp.Filter(k)
    f.n_skipped = 0  # further updates skipped for an unknown id
    rows = np.concatenate([t_imu[:, None], imu[:, :, b]], axis=1)
    cursor = int(win_off[0])
    for w, t_det in enumerate(t_frames):
        hi = int(win_off[w + 1])
        dets = [np.concatenate([[det_id[w, s, b]], det_pose[w, s, :, b]]) for s in range(det_id.shape[1]) if det_id[w, s, b] >= 0]
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
            if all_markers:
                f.n_skipped += np_observation_update_all(f, dets, joseph)
            else:
                f.observation_update(dets, joseph=joseph)
    return f


def _board(B=3, duration=0.8, seed=5):
    """BASELINE configs[3] in small: noisy corners of the 8 board markers -> the oracle's refractive solve -> 8 slots per frame,
    some ids -1 and one id (9) that is not in the board's map"""
    import orc
    from fbus_ekf_b200 import capi, synth
    cfg = capi.config_default()
    bcfg = synth.board_config(cfg)
    traj = synth.truth_trajectory(bcfg, duration, standoff=1.0)
    W, N, m = len(traj["t_frames"]), len(traj["t_imu"]), 8
    base, ids, _ = synth.board_base_corners(bcfg, traj)
    rng = np.random.default_rng(seed)
    corners = np.ascontiguousarray((np.repeat(base, B, axis=1) + rng.normal(size=(16, W * m * B)) * 2e-4).astype(np.float32))
    po, _, vo = orc.refract_solve(bcfg, corners)
    det_pose = np.ascontiguousarray(po.reshape(7, W, m, B).transpose(1, 2, 0, 3))
    det_id = np.ascontiguousarray(np.where(vo.reshape(W, m, B) != 0, np.repeat(ids[:, :, None], B, axis=2), -1).astype(np.int32))
    det_id[2::3, 6, :] = -1          # undetected markers
    det_id[4::5, 1, ::2] = 9         # an id the map does not know
    imu = np.ascontiguousarray(traj["base_imu"][:, :, None] + rng.normal(size=(N, 6, B)) * np.array([0.015] * 3 + [1e-3] * 3)[None, :, None])
    return bcfg, traj, imu, det_id, det_pose


def _orc_run(bcfg, traj, imu, det_id, det_pose, flags):
    """the C++ oracle over all frames: as it stands, or through OrcAllMarkers when `flags` has FBUS_FLAG_ALL_MARKERS"""
    import orc
    from fbus_ekf_b200 import capi
    B, m = imu.shape[2], det_id.shape[1]
    c = copy.copy(bcfg)
    c.flags = flags
    W = len(traj["t_frames"])
    if flags & capi.FBUS_FLAG_ALL_MARKERS:
        o = OrcAllMarkers(c, B)
        o.step_windows(traj["t_imu"], imu, traj["t_frames"], det_id, det_pose, traj["win_off"], 0, W)
        return o.get_state()
    o = orc.Oracle(c, B)
    s = capi.make_imu_stream(traj["t_imu"], imu, B)
    d = capi.make_det_frames(traj["t_frames"], det_id, det_pose, B, m)
    o.step_windows(s, d, traj["win_off"], 0, len(traj["t_frames"]))
    return o.get_state()


@pytest.mark.parametrize("joseph", [False, True])
def test_board_cpp_vs_numpy(joseph):
    """the two restatements agree in this mode (tolerances of test_oracle_cross)"""
    import fbus_oracle_np as onp
    from fbus_ekf_b200 import capi
    bcfg, traj, imu, det_id, det_pose = _board()
    flags = capi.FBUS_FLAG_ALL_MARKERS | (capi.FBUS_FLAG_JOSEPH if joseph else 0)
    sc = _orc_run(bcfg, traj, imu, det_id, det_pose, flags)
    k = onp.Consts(_np_config(bcfg))
    for b in range(imu.shape[2]):
        f = _np_step_windows(k, traj["t_imu"], imu, traj["t_frames"], det_id, det_pose, traj["win_off"], b, joseph, True)
        assert f.initialised and sc["initialised"][b] == 1
        for name, v in (("p", f.p), ("q", f.q), ("v", f.v), ("ba", f.ba), ("bg", f.bg), ("g", f.g)):
            assert np.abs(sc[name][:, b] - v).max() <= 1e-10 * max(1.0, np.abs(v).max()), (b, name)
        assert sc["prev_marker_id"][b] == f.prev_marker_id
        Pc = sc["P"][:, b].reshape(18, 18)
        assert np.abs(Pc - f.P).max() <= 1e-9 * np.abs(f.P).max()
        big = np.abs(f.P) >= 1e-6 * np.abs(f.P).max()
        assert (np.abs(Pc - f.P)[big] <= 1e-9 * np.abs(f.P)[big]).all()
        # the unknown id 9 was seen by filters 0 and 2 and skipped with the status bit
        assert bool(sc["status"][b] & capi.FBUS_ST_UPDATE_SKIPPED) == (b % 2 == 0)
        assert f.n_skipped > 0 if b % 2 == 0 else f.n_skipped == 0


def test_board_differs_from_default():
    """with a second known marker in the frames the mode changes the result (the flag is not a no-op), and the extra updates
    pull the covariance of the pose down"""
    from fbus_ekf_b200 import capi
    bcfg, traj, imu, det_id, det_pose = _board()
    s0 = _orc_run(bcfg, traj, imu, det_id, det_pose, 0)
    s1 = _orc_run(bcfg, traj, imu, det_id, det_pose, capi.FBUS_FLAG_ALL_MARKERS)
    assert np.abs(s0["p"] - s1["p"]).min(axis=0).max() > 0 and not np.array_equal(s0["P"], s1["P"])
    tr = lambda s: s["P"].reshape(18, 18, -1)[[0, 1, 2], [0, 1, 2]].sum(axis=0)
    assert (tr(s1) < tr(s0)).all()
    assert np.array_equal(s0["prev_marker_id"], s1["prev_marker_id"])


def test_single_marker_stream_identical():
    """at most one known detection per frame: the flag changes nothing, in either oracle"""
    import fbus_oracle_np as onp
    from fbus_ekf_b200 import capi
    bcfg, traj, imu, det_id, det_pose = _board()
    det1 = det_id.copy()
    det1[:, 1:, :] = -1
    det1 = np.ascontiguousarray(det1)
    s0 = _orc_run(bcfg, traj, imu, det1, det_pose, 0)
    s1 = _orc_run(bcfg, traj, imu, det1, det_pose, capi.FBUS_FLAG_ALL_MARKERS)
    for key in s0:
        assert np.array_equal(s0[key], s1[key]), key
    k = onp.Consts(_np_config(bcfg))
    for b in range(imu.shape[2]):
        f0 = _np_step_windows(k, traj["t_imu"], imu, traj["t_frames"], det1, det_pose, traj["win_off"], b, False, False)
        f1 = _np_step_windows(k, traj["t_imu"], imu, traj["t_frames"], det1, det_pose, traj["win_off"], b, False, True)
        assert np.array_equal(f0.p, f1.p) and np.array_equal(f0.q, f1.q) and np.array_equal(f0.P, f1.P)


# ------------------------------------------------------------------------------------------------ rules on hand-built frames
def _hand_state(seed=3):
    """one random plausible state (both oracles) and the default configuration"""
    import fbus_oracle_np as onp
    from fbus_ekf_b200 import capi
    st = random_states(1, np.random.default_rng(seed))
    k = onp.Consts(onp.default_config())
    return capi.config_default(), k, st


def _np_filter(k, st):
    import fbus_oracle_np as onp
    f = onp.Filter(k)
    for name in ("q", "p", "v", "ba", "bg", "g"):
        setattr(f, name, st[name][:, 0].copy())
    f.R = st["R"][:, 0].reshape(3, 3).copy()
    f.P = st["P"][:, 0].reshape(18, 18).copy()
    f.t = float(st["t"][0])
    f.prev_marker_id = int(st["prev_marker_id"][0])
    f.initialised = True
    return f


def _dets_at(f, ids_dists, seed=0):
    """detections of markers `ids` near what the filter predicts, scaled to the given distances from the camera (the nearest
    marker rule reads only the distance); an id outside the map gets the pose of marker 0"""
    rng = np.random.default_rng(seed)
    out = []
    for mid, dist in ids_dists:
        d = np.zeros(8)
        d[0] = 0 if mid not in f.k.markers else mid
        hP, hQ, _ = f.measurement_model(d)
        hP = hP / np.linalg.norm(hP) * dist + rng.normal(size=3) * 1e-3
        hQ = hQ + rng.normal(size=4) * 1e-3
        d[0], d[1:4], d[4:8] = mid, hP, hQ / np.linalg.norm(hQ)
        out.append(d)
    return out


def _orc_update(cfg, st, dets, flags):
    """one un-fused update of a single filter on the C++ oracle, on one frame built from `dets` (slot order = list order)"""
    import orc
    from fbus_ekf_b200 import capi
    c = copy.copy(cfg)
    c.flags = flags
    m = len(dets)
    ids = np.ascontiguousarray(np.array([[int(d[0]) for d in dets]], dtype=np.int32)[:, :, None])
    pose = np.ascontiguousarray(np.array([[d[1:8] for d in dets]])[:, :, :, None])
    t = np.array([st["t"][0]])
    if flags & capi.FBUS_FLAG_ALL_MARKERS:
        o = OrcAllMarkers(c, 1)
        o.set_state(st)
        o.update(t, ids, pose, 0)
    else:
        o = orc.Oracle(c, 1)
        o.set_state(st)
        o.update(capi.make_det_frames(t, ids, pose, 1, m), 0)
    return o.get_state()


def _close(s, f):
    for name in ("p", "q", "v", "ba", "bg", "g"):
        assert np.abs(s[name][:, 0] - getattr(f, name)).max() <= 1e-10 * max(1.0, np.abs(getattr(f, name)).max()), name
    assert np.abs(s["P"][:, 0].reshape(18, 18) - f.P).max() <= 1e-9 * np.abs(f.P).max()


@pytest.mark.parametrize("prev, order", [
    (2, [0, 1, 2]),   # hysteresis: marker 2 (slot 0, 1.0 m) stays against the nearer marker 1 (slot 1, 0.8 m)
    (5, [1, 0, 2]),   # no hysteresis: the nearest (slot 1) first, then slots 0 and 2
])
def test_order_chosen_then_slots(prev, order):
    from fbus_ekf_b200 import capi
    cfg, k, st = _hand_state()
    st["prev_marker_id"][0] = prev
    f = _np_filter(k, st)
    dets = _dets_at(f, [(2, 1.0), (1, 0.8), (3, 1.2)])
    ref = _np_filter(k, st)
    for s in order:
        np_update_with(ref, dets[s])
    np_observation_update_all(f, dets)
    assert np.array_equal(f.p, ref.p) and np.array_equal(f.q, ref.q) and np.array_equal(f.P, ref.P)
    assert f.prev_marker_id == int(dets[order[0]][0])
    # a different order gives a different state: the check above pins the order
    alt = _np_filter(k, st)
    for s in sorted(order):
        np_update_with(alt, dets[s])
    assert sorted(order) == order or not np.array_equal(alt.p, ref.p)
    s = _orc_update(cfg, st, dets, capi.FBUS_FLAG_ALL_MARKERS)
    _close(s, ref)
    assert s["prev_marker_id"][0] == f.prev_marker_id and not (s["status"][0] & capi.FBUS_ST_UPDATE_SKIPPED)


def test_unknown_chosen_marker():
    """the chosen (nearest) marker is unknown: the other known ones are still applied in slot order, prev_marker_id stays"""
    from fbus_ekf_b200 import capi
    cfg, k, st = _hand_state(4)
    st["prev_marker_id"][0] = 5
    f = _np_filter(k, st)
    dets = _dets_at(f, [(1, 1.0), (99, 0.5), (3, 1.2)])
    ref = _np_filter(k, st)
    np_update_with(ref, dets[0])
    np_update_with(ref, dets[2])
    skipped = np_observation_update_all(f, dets)
    assert np.array_equal(f.p, ref.p) and np.array_equal(f.P, ref.P) and f.prev_marker_id == 5 and skipped == 1
    s = _orc_update(cfg, st, dets, capi.FBUS_FLAG_ALL_MARKERS)
    _close(s, ref)
    assert s["prev_marker_id"][0] == 5 and (s["status"][0] & capi.FBUS_ST_UPDATE_SKIPPED)
    # the default mode does nothing with this frame
    s0 = _orc_update(cfg, st, dets, 0)
    assert np.array_equal(s0["p"], st["p"]) and np.array_equal(s0["P"], st["P"])


@pytest.mark.parametrize("ids, skipped", [
    ([1, 2, 3], False),
    ([1, 99, 3], True),     # an unknown id in a further slot
    ([99, 2, 3], True),     # ... in the nearest slot
    ([1, -1, 3], False),    # an empty slot is not a skipped update
])
def test_status_update_skipped(ids, skipped):
    from fbus_ekf_b200 import capi
    cfg, k, st = _hand_state(5)
    f = _np_filter(k, st)
    dets = _dets_at(f, [(i, 0.7 + 0.2 * s) for s, i in enumerate(ids)])
    s = _orc_update(cfg, st, dets, capi.FBUS_FLAG_ALL_MARKERS)
    assert bool(s["status"][0] & capi.FBUS_ST_UPDATE_SKIPPED) == skipped
