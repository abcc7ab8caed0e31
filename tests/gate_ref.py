"""Reference restatement of the innovation gate of fbus_set_gate (include/fbus_ekf.h) on the NumPy oracle (test infrastructure).

Every measurement update of the reference first forms NIS = r^T S^-1 r from the oracle's own measurement_model, the reference's
quaternion sign choice and S = H P H^T + R, solved with np.linalg.solve.  With threshold g the update is rejected iff
g > 0 and not NIS <= g; a rejected update leaves state and covariance as they are, but the marker choice (prev_marker_id) stands.
Accepted updates are the oracle's observation_update as it stands; under FBUS_FLAG_ALL_MARKERS the further slots follow in slot
order through tests/all_markers_ref.py, each gated on its own.  The frame loop is fbus_oracle_np.replay's; a frame without a
detection does nothing and leaves its IMU samples buffered for the next frame, as the kernel does.  The oracle is unchanged.

  GatedFilter    -- one filter: fused frames (continued from call to call) and the un-fused update
  replay_gated   -- fbus_oracle_np.replay with a gate
"""
from __future__ import annotations

import numpy as np

from all_markers_ref import np_chosen_index, np_update_with


def nis(f, d) -> float:
    """NIS of the reference's update of fbus_oracle_np.Filter f with detection d (a known marker)"""
    hP, hQ, H = f.measurement_model(d)
    yP, yQ = d[1:4], d[4:8]
    if np.sum((yQ - hQ) ** 2) > np.sum((yQ + hQ) ** 2):  # filter.cpp:702-706
        hQ = -hQ
        H[3:7, 6:9] = -H[3:7, 6:9]
    S = H @ f.P @ H.T + f.k.Rn
    r = np.concatenate([yP - hP, yQ - hQ])
    return float(r @ np.linalg.solve(S, r))


def rejects(g: float, v: float) -> bool:
    return bool(g > 0 and not (v <= g))


class GatedFilter:
    """one fbus_oracle_np.Filter with a gate threshold `gate`.  `rejected` counts the rejected updates, `flag` is set by the
    first one (FBUS_ST_UPDATE_REJECTED), `log` holds (NIS, threshold) of every update the gate tested with a threshold > 0"""

    def __init__(self, k, gate: float, joseph: bool = False, all_markers: bool = False):
        import fbus_oracle_np as onp
        self.f = onp.Filter(k)
        self.gate = float(gate)
        self.joseph, self.all_markers = joseph, all_markers
        self.rejected = 0
        self.flag = False
        self.log = []
        self.cursor = None  # first IMU row not consumed yet (fused frames)

    def _test(self, d) -> bool:
        """True when the update with detection d is accepted"""
        v = nis(self.f, d)
        if self.gate > 0:
            self.log.append((v, self.gate))
        if rejects(self.gate, v):
            self.rejected += 1
            self.flag = True
            return False
        return True

    def update(self, dets):
        """the reference's update of one frame (detections in slot order), gated"""
        f = self.f
        if len(dets) == 0:
            return
        idx = np_chosen_index(f, dets)
        d = dets[idx]
        if int(d[0]) in f.k.markers:
            if self._test(d):
                f.observation_update(dets, joseph=self.joseph)
            else:
                f.prev_marker_id = int(d[0])  # the choice stands
        if not self.all_markers:
            return
        for c, e in enumerate(dets):
            if c != idx and int(e[0]) in f.k.markers and self._test(e):
                np_update_with(f, e, self.joseph)

    def step(self, rows, frames, off, w0: int, w1: int):
        """fused frames [w0, w1): rows [N][7] (t, accel, gyro), frames [(t, dets)], off the window offsets; the IMU buffer
        continues from the previous call"""
        f = self.f
        if self.cursor is None:
            self.cursor = int(off[w0])
        for w in range(w0, w1):
            t_det, dets = frames[w]
            hi = int(off[w + 1])
            if not dets:
                continue
            if not f.initialised:
                later = np.nonzero(rows[self.cursor:hi, 0] > t_det)[0]
                cnt = int(later[0]) if len(later) else hi - self.cursor
                if f.init_pose(dets, t_det, cnt):
                    self.cursor += cnt
            else:
                f.reset_state(dets, t_det)
                self.cursor += f.batch_imu(rows[self.cursor:hi], t_det)
                self.update(dets)


def stream_frames(t_frames, det_id, det_pose, b: int):
    """[(t, dets)] of filter b from the fbus_det_frames arrays det_id [W][m][B], det_pose [W][m][7][B] (slots with id >= 0)"""
    return [(float(t_frames[w]), [np.concatenate([[det_id[w, s, b]], det_pose[w, s, :, b]]) for s in range(det_id.shape[1])
                                  if det_id[w, s, b] >= 0]) for w in range(len(t_frames))]


def stream_rows(t_imu, imu, b: int):
    """IMU rows [N][7] of filter b from an fbus_imu_stream array imu [N][6][B] (SI doubles)"""
    return np.concatenate([np.asarray(t_imu)[:, None], imu[:, :, b]], axis=1)


def replay_gated(cfg, imu, image_rows, gate: float, n_init: int = 500, joseph: bool = False, all_markers: bool = False):
    """fbus_oracle_np.replay (without the IIR and the covariance trace) with the gate; returns its rows and the GatedFilter"""
    import fbus_oracle_np as onp
    k = onp.Consts(cfg)
    g = GatedFilter(k, gate, joseph, all_markers)
    g.f.init_gravity_gyrobias(imu[:n_init])
    frames = onp.group_frames(image_rows)
    off = onp.window_offsets(imu[:, 0], [fr[0] for fr in frames], n_init)
    rows = []
    for w in range(len(frames)):
        g.step(imu, frames, off, w, w + 1)
        f = g.f
        rows.append(np.concatenate([[f.t], f.p, f.q, f.v, f.ba, f.bg]))
    return {"rows": np.array(rows), "gated": g}
