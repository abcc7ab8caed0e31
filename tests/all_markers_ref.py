"""Reference restatement of FBUS_FLAG_ALL_MARKERS (include/fbus_ekf.h) on top of the two oracles, built from their unchanged calls
(test infrastructure).

The mode is "the reference's update with the marker it chooses, then every other known slot of the frame in slot order, each as
its own update at the state the previous one left".  Each further update is exactly the reference's ObservationUpdate on a
one-detection list: the chooser of a one-entry list picks that entry, so the oracle applies the reference's measurement model,
sign choice, gain and covariance form (standard or Joseph) to it.  Only two things of that call are undone, because the mode
departs from filter.cpp there (rules 1 and 3 of the flag's comment): prev_marker_id, which only the chosen marker sets, and the
FBUS_ST_NO_DETECTION bit that the C++ oracle's update sets for a filter without a detection in a round.

  np_observation_update_all  -- the NumPy oracle (fbus_oracle_np.Filter), one filter
  OrcAllMarkers              -- the C++ oracle (orc.Oracle), a batch: fused frames and the un-fused update
"""
from __future__ import annotations

import math

import numpy as np


# --------------------------------------------------------------------------------------------------------- NumPy oracle
def np_chosen_index(f, dets):
    """index into `dets` of the marker filter.cpp:639-664 updates with (fbus_oracle_np.Filter.observation_update's chooser)"""
    md, idx, prev_dist, prev_idx = 10.0, 0, 0.0, 0
    for c, d in enumerate(dets):
        dist = np.linalg.norm(d[1:4])
        if dist < md:
            md, idx = dist, c
        if int(d[0]) == f.prev_marker_id:
            prev_dist, prev_idx = dist, c
    if abs(prev_dist - md) < f.k.cfg.marker_switch_thres and prev_dist != 0:
        idx = prev_idx
    return idx


def np_update_with(f, d, joseph=False):
    """one further update with detection d (known marker): the reference's update of a one-detection list, prev_marker_id kept"""
    prev = f.prev_marker_id
    f.observation_update([d], joseph=joseph)
    f.prev_marker_id = prev


def np_observation_update_all(f, dets, joseph=False):
    """FBUS_FLAG_ALL_MARKERS on fbus_oracle_np.Filter f for the detection list `dets` (slot order, ids >= 0).
    Returns the number of updates skipped for an unknown id (the C++ side's FBUS_ST_UPDATE_SKIPPED)."""
    if len(dets) == 0:
        return 0
    idx = np_chosen_index(f, dets)
    skipped = 0 if int(dets[idx][0]) in f.k.markers else 1
    f.observation_update(dets, joseph=joseph)  # the chosen marker: the reference's update as it stands
    for c, d in enumerate(dets):
        if c == idx:
            continue
        if int(d[0]) in f.k.markers:
            np_update_with(f, d, joseph)
        else:
            skipped += 1
    return skipped


# ----------------------------------------------------------------------------------------------------------- C++ oracle
def orc_chosen_slot(ids, pose, prev_id, switch_thres):
    """slot (index into the frame's m slots) that oracle/fbus_oracle.cpp's ObservationUpdate chooses, -1 without detections.
    ids [m], pose [m][7] of one filter; the distance is evaluated as the oracle's norm3 does."""
    md, idx, prev_dist, prev_idx, n = 10.0, -1, 0.0, -1, 0
    for s in range(len(ids)):
        if ids[s] < 0:
            continue
        x, y, z = float(pose[s][0]), float(pose[s][1]), float(pose[s][2])
        dist = math.sqrt(x * x + y * y + z * z)
        if n == 0:
            idx = s  # the oracle's idx = 0 of the compacted list
        if dist < md:
            md, idx = dist, s
        if int(ids[s]) == prev_id:
            prev_dist, prev_idx = dist, s
        n += 1
    if n and abs(prev_dist - md) < switch_thres and prev_dist != 0:
        idx = prev_idx
    return idx


class OrcAllMarkers:
    """A batch of C++ oracle filters in FBUS_FLAG_ALL_MARKERS mode.  `cfg` is passed to orc.Oracle as is (FBUS_FLAG_JOSEPH selects
    the Joseph form; the oracle itself does not read FBUS_FLAG_ALL_MARKERS)."""

    def __init__(self, cfg, batch):
        import orc
        self.o = orc.Oracle(cfg, batch)
        self.B = batch
        self.thres = float(cfg.marker_switch_thres)

    def _further_updates(self, ids, pose, t, prev, upd):
        """the further updates of one frame.  ids [m][B], pose [m][7][B]; prev [B] prev_marker_id before the frame; upd [B] the
        filters whose frame got the reference's update"""
        from fbus_ekf_b200 import capi
        m = ids.shape[0]
        todo = []
        for b in range(self.B):
            lst = []
            if upd[b]:
                ch = orc_chosen_slot(ids[:, b], pose[:, :, b], int(prev[b]), self.thres)
                lst = [s for s in range(m) if s != ch and ids[s, b] >= 0]
            todo.append(lst)
        for r in range(max((len(x) for x in todo), default=0)):
            ids1 = np.full((1, 1, self.B), -1, dtype=np.int32)
            pose1 = np.zeros((1, 1, 7, self.B))
            has = np.zeros(self.B, dtype=bool)
            for b, lst in enumerate(todo):
                if r < len(lst):
                    ids1[0, 0, b] = ids[lst[r], b]
                    pose1[0, 0, :, b] = pose[lst[r], :, b]
                    has[b] = True
            before = self.o.get_state(with_cov=False)
            self.o.update(capi.make_det_frames(np.array([t]), ids1, pose1, self.B, 1), 0)
            after = self.o.get_state(with_cov=False)
            fix = {"prev_marker_id": np.ascontiguousarray(before["prev_marker_id"]),
                   "status": np.ascontiguousarray(np.where(has, after["status"], before["status"]).astype(np.int32))}
            self.o.set_state(fix)

    def step_windows(self, t_imu, imu, t_frames, det_id, det_pose, win_off, w0, w1):
        """fused frames [w0, w1) on host arrays (imu [N][6][B], det_id [W][m][B], det_pose [W][m][7][B]): frame by frame through
        orc_step_windows, continued from call to call, each followed by the frame's further updates"""
        from fbus_ekf_b200 import capi
        B, m = self.B, det_id.shape[1]
        self._s = capi.make_imu_stream(t_imu, imu, B)
        d = capi.make_det_frames(t_frames, det_id, det_pose, B, m)
        win_off = np.ascontiguousarray(win_off, dtype=np.uint32)
        for w in range(w0, w1):
            before = self.o.get_state(with_cov=False)
            self.o.step_windows(self._s, d, win_off, w, w + 1)
            # the reference's update runs for a filter initialised before the frame that has a detection (filter.cpp:207-235)
            upd = (before["initialised"] != 0) & (det_id[w] >= 0).any(axis=0)
            self._further_updates(det_id[w], det_pose[w], float(t_frames[w]), before["prev_marker_id"], upd)

    def update(self, t_frames, det_id, det_pose, w):
        """the un-fused update (orc_update / fbus_update) of frame w"""
        from fbus_ekf_b200 import capi
        B, m = self.B, det_id.shape[1]
        before = self.o.get_state(with_cov=False)
        self.o.update(capi.make_det_frames(t_frames, det_id, det_pose, B, m), w)
        self._further_updates(det_id[w], det_pose[w], float(t_frames[w]), before["prev_marker_id"], (det_id[w] >= 0).any(axis=0))

    def __getattr__(self, name):  # propagate, set_state, get_state, ... of the wrapped oracle
        return getattr(self.o, name)
