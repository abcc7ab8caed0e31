"""Synthetic workloads for the parity tests and the benchmark (SURVEY.md section 8d, configs 3-5).

Host-side NumPy only (small, shared, noise-free base data); the per-filter Monte-Carlo noise is added on the
GPU by fbus_synth_streams (Philox4x32-10).  Nothing here is on the timed path.

  truth_trajectory     smooth 6-DOF trajectory in front of marker 0 -> noise-free 200 Hz body accel/gyro, noise-free
                       25 Hz marker poses as the filter's own measurement model predicts them, per-frame truth, and the
                       per-frame IMU windows (win_off).
  forward_project      flat-port forward projection (air -> glass -> water) of 3-D points into normalised image
                       coordinates (SURVEY A.1-4); inverse of the ray trace of VISION::RefractionTriangulation.
  random_marker_corners  stereo corner observations of randomly posed square markers (config 4 input).
  base_marker_poses    noise-free pose of every map marker in every frame of a truth trajectory; with make_corner_spec the
                       input of fbus_synth_corners, which projects them and adds per-filter corner noise on the device.
"""
from __future__ import annotations

import numpy as np

from . import capi

# ---------------------------------------------------------------------------------------------- small rotation helpers


def _skew(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]], dtype=np.float64)


def _qmul(a, b):
    w = a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3]
    x = a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2]
    y = a[0] * b[2] + a[2] * b[0] + a[3] * b[1] - a[1] * b[3]
    z = a[0] * b[3] + a[3] * b[0] + a[1] * b[2] - a[2] * b[1]
    return np.array([w, x, y, z])


def _qconj(a):
    return np.array([a[0], -a[1], -a[2], -a[3]])


def _q2R(q):
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def _exp_q(phi):
    th = np.linalg.norm(phi)
    if th < 1e-12:
        return np.array([1.0, 0.5 * phi[0], 0.5 * phi[1], 0.5 * phi[2]])
    return np.concatenate([[np.cos(th / 2)], np.sin(th / 2) * phi / th])


def _right_jacobian(phi):
    th = np.linalg.norm(phi)
    K = _skew(phi)
    if th < 1e-8:
        return np.eye(3) - 0.5 * K
    return np.eye(3) - (1 - np.cos(th)) / th ** 2 * K + (th - np.sin(th)) / th ** 3 * K @ K


def quat_from_rotmat(R):
    """Eigen Quaterniond(Matrix3d) (main.cpp:201; SURVEY A.1-3): w,x,y,z, not normalised.  Host arithmetic of the workload
    generator only (the filter path derives its own constants on the device side of the C ABI); tests check it against the
    library helper fbus_quat_from_rotmat."""
    m = np.asarray(R, dtype=np.float64).reshape(3, 3)
    q = np.zeros(4)
    t = m[0, 0] + m[1, 1] + m[2, 2]
    if t > 0:
        t = np.sqrt(t + 1.0)
        q[0] = 0.5 * t
        t = 0.5 / t
        q[1], q[2], q[3] = (m[2, 1] - m[1, 2]) * t, (m[0, 2] - m[2, 0]) * t, (m[1, 0] - m[0, 1]) * t
    else:
        i = 0
        if m[1, 1] > m[0, 0]:
            i = 1
        if m[2, 2] > m[i, i]:
            i = 2
        j, k = (i + 1) % 3, (i + 2) % 3
        t = np.sqrt(m[i, i] - m[j, j] - m[k, k] + 1.0)
        q[1 + i] = 0.5 * t
        t = 0.5 / t
        q[0] = (m[k, j] - m[j, k]) * t
        q[1 + j] = (m[j, i] + m[i, j]) * t
        q[1 + k] = (m[k, i] + m[i, k]) * t
    return q


def filter_extrinsics(cfg: capi.FbusConfig):
    """R_IL, Q_IL (not normalised), P_IL as the filter derives them (filter.hpp:67-69, filter.cpp:369-372)."""
    T = np.diag([-1.0, -1.0, 1.0, 1.0]) @ np.array(cfg.tsc_left, dtype=np.float64).reshape(4, 4)
    R_IL = T[:3, :3].copy()
    return R_IL, quat_from_rotmat(R_IL), -R_IL.T @ T[:3, 3]


def stereo_extrinsics(cfg: capi.FbusConfig):
    """R_RL, P_LR as the vision path derives them from the raw T_SC (vision.cpp:476-481)."""
    TL = np.array(cfg.tsc_left, dtype=np.float64).reshape(4, 4)
    TR = np.array(cfg.tsc_right, dtype=np.float64).reshape(4, 4)
    R_RL = TL[:3, :3] @ TR[:3, :3].T
    return R_RL, TL[:3, 3] - R_RL @ TR[:3, 3]


# ---------------------------------------------------------------------------------------------- EKF workload


def truth_trajectory(cfg: capi.FbusConfig, duration: float, imu_rate: float = 200.0, frame_rate: float = 25.0, marker_id: int = 0,
                     seed: int = 20260117, periodic: bool = False, standoff: float = 0.50):
    """Smooth trajectory matching the envelope of the reference's logs (position extent < 0.8 m, |v| < 0.4 m/s, a few
    hundredths rad/s of rotation) in front of marker `marker_id`.  Gravity convention of the filter after
    InitializePose: g = (9.8, 0, 0) (filter.cpp:387), i.e. accel_body = R^T (p'' - g).
    periodic=True makes the motion exactly periodic in `duration` (all sinusoid frequencies are multiples of
    1/duration), so a stream of one period can be replayed with timestamps advanced by k*duration."""
    rng = np.random.default_rng(seed)
    n_frames = int(round(duration * frame_rate))
    per = int(round(imu_rate / frame_rate))
    n_samples = n_frames * per
    dt = 1.0 / imu_rate
    t_imu = dt * (1 + np.arange(n_samples))
    t_frames = t_imu[per - 1::per].copy()
    # sums of sinusoids
    nf = 4
    fp = rng.uniform(0.05, 0.45, size=(nf, 3))
    ap = rng.uniform(0.02, 0.06, size=(nf, 3))
    php = rng.uniform(0, 2 * np.pi, size=(nf, 3))
    fr = rng.uniform(0.05, 0.35, size=(nf, 3))
    ar = rng.uniform(0.01, 0.03, size=(nf, 3))
    phr = rng.uniform(0, 2 * np.pi, size=(nf, 3))
    if periodic:
        harm = np.array([1.0, 1.0, 2.0, 3.0])[:, None] / duration
        fp = np.repeat(harm, 3, axis=1)
        fr = np.repeat(harm, 3, axis=1)
        ap = ap * 0.25 / (harm * duration)
        ar = ar * 0.5 / (harm * duration)
    p0 = np.array([-0.10, 0.05, standoff])  # `standoff` = distance from the marker plane
    q0 = np.array([-0.0203, -0.7053, 0.7086, -0.0065])
    q0 /= np.linalg.norm(q0)

    def pos(t, d=0):
        w = 2 * np.pi * fp
        arg = w[None] * np.asarray(t)[:, None, None] + php[None]
        if d == 0:
            return p0 + (ap[None] * np.sin(arg)).sum(1)
        if d == 1:
            return (ap[None] * w[None] * np.cos(arg)).sum(1)
        return (-ap[None] * w[None] ** 2 * np.sin(arg)).sum(1)

    def rotvec(t, d=0):
        w = 2 * np.pi * fr
        arg = w[None] * np.asarray(t)[:, None, None] + phr[None]
        if d == 0:
            return (ar[None] * np.sin(arg)).sum(1)
        return (ar[None] * w[None] * np.cos(arg)).sum(1)

    g = np.array([9.8, 0.0, 0.0])
    tm = t_imu - 0.5 * dt  # the filter applies sample i over (t_{i-1}, t_i]: use mid-interval kinematics
    acc_w = pos(tm, 2)
    phi, dphi = rotvec(tm), rotvec(tm, 1)
    base_imu = np.zeros((n_samples, 6))
    for i in range(n_samples):
        R = _q2R(_qmul(q0, _exp_q(phi[i])))
        base_imu[i, 0:3] = R.T @ (acc_w[i] - g)
        base_imu[i, 3:6] = _right_jacobian(phi[i]) @ dphi[i]
    # per-frame truth and noise-free measurements hP = R_IL R^T (P_M - p - R P_IL), hQ = Q_IL * conj(q) * Q_M
    R_IL, Q_IL, P_IL = filter_extrinsics(cfg)
    mi = list(cfg.marker_id[:cfg.n_markers]).index(marker_id)
    P_M = np.array(cfg.marker_pos[mi * 3:mi * 3 + 3])
    Q_M = quat_from_rotmat(np.array(cfg.marker_rot[mi * 9:mi * 9 + 9]).reshape(3, 3))
    pt = pos(t_frames)
    pht = rotvec(t_frames)
    truth_p = np.zeros((n_frames, 3))
    truth_q = np.zeros((n_frames, 4))
    base_pose = np.zeros((n_frames, 7))
    for w in range(n_frames):
        q = _qmul(q0, _exp_q(pht[w]))
        R = _q2R(q)
        truth_p[w], truth_q[w] = pt[w], q
        base_pose[w, 0:3] = R_IL @ R.T @ (P_M - pt[w] - R @ P_IL)
        base_pose[w, 3:7] = _qmul(_qmul(Q_IL, _qconj(q)), Q_M)
    win_off = (per * np.arange(n_frames + 1)).astype(np.uint32)
    return {"t_imu": t_imu, "t_frames": t_frames, "base_imu": np.ascontiguousarray(base_imu),
            "base_pose": np.ascontiguousarray(base_pose), "truth_p": truth_p, "truth_q": truth_q, "win_off": win_off,
            "marker_id": marker_id, "per": per}


# noise levels measured on the static phases of the reference's logs (SURVEY 8d, config 3)
DEFAULT_NOISE = dict(sigma_acc=0.015, sigma_gyro=1e-3, sigma_ba=0.05, sigma_bg=2e-3, sigma_pos=2.5e-4, sigma_quat=1.5e-3)


def make_synth_spec(traj: dict, seed: int, filter_offset: int = 0, **noise) -> capi.SynthSpec:
    nz = dict(DEFAULT_NOISE)
    nz.update(noise)
    sp = capi.SynthSpec()
    sp.n_samples = traj["base_imu"].shape[0]
    sp.n_frames = traj["base_pose"].shape[0]
    sp.base_imu = capi.dptr(traj["base_imu"])
    sp.base_pose = capi.dptr(traj["base_pose"])
    sp.marker_id = traj["marker_id"]
    for k_, v in nz.items():
        setattr(sp, k_, v)
    sp.seed = seed
    sp.filter_offset = filter_offset
    sp._keep = traj
    return sp


# ---------------------------------------------------------------------------------------------- refraction workload


def forward_project(cfg: capi.FbusConfig, X: np.ndarray) -> np.ndarray:
    """Flat-port forward projection of points X [n,3] given in a camera's own frame (interfaces at z = d_air and
    z = d_air + d_glass, normal (0,0,1)) -> normalised image coordinates [n,2].  Solves the monotone 1-D equation of
    SURVEY A.1-4 for s0 = sin(theta_air) by safeguarded Newton iterations."""
    X = np.asarray(X, dtype=np.float64)
    d0, d1 = cfg.d_air, cfg.d_glass
    k1, k2 = cfg.n_air / cfg.n_glass, cfg.n_air / cfg.n_water
    rho = np.hypot(X[:, 0], X[:, 1])
    Zw = X[:, 2] - d0 - d1

    def tfun(s):
        return s / np.sqrt(1 - s * s)

    def dtfun(s):
        return (1 - s * s) ** -1.5

    s = rho / np.sqrt(rho * rho + X[:, 2] ** 2)
    lo, hi = np.zeros_like(s), np.full_like(s, 1 - 1e-12)
    for _ in range(60):
        f = d0 * tfun(s) + d1 * tfun(k1 * s) + Zw * tfun(k2 * s) - rho
        lo = np.where(f < 0, s, lo)
        hi = np.where(f > 0, s, hi)
        df = d0 * dtfun(s) + d1 * k1 * dtfun(k1 * s) + Zw * k2 * dtfun(k2 * s)
        sn = s - f / df
        bad = ~((sn > lo) & (sn < hi))
        s = np.where(bad, 0.5 * (lo + hi), sn)
    tan0 = tfun(s)
    with np.errstate(invalid="ignore", divide="ignore"):
        scale = np.where(rho > 0, tan0 / rho, 1.0 / (d0 + k1 * d1 + k2 * Zw))
    return X[:, :2] * scale[:, None]


def random_marker_poses(n: int, rng, far_fraction: float = 0.0, max_tilt: float = 0.6):
    """marker poses (R_M [n,3,3], p [n,3]) in the FLIPPED left-camera frame; marker Z axis towards the camera."""
    dist = rng.uniform(0.5, 1.5, size=n)
    far = rng.random(n) < far_fraction
    dist = np.where(far, rng.uniform(2.3, 3.0, size=n), dist)
    p = np.stack([rng.uniform(-0.25, 0.25, n) * dist, rng.uniform(-0.2, 0.2, n) * dist, dist], axis=1)
    Rb = np.diag([1.0, -1.0, -1.0])
    Rm = np.zeros((n, 3, 3))
    for i in range(n):
        phi = rng.uniform(-max_tilt, max_tilt, size=3) * np.array([1.0, 1.0, 3.0])
        Rm[i] = Rb @ _q2R(_exp_q(phi))
    return Rm, p


def marker_corners_from_pose(cfg: capi.FbusConfig, Rm: np.ndarray, p: np.ndarray, size: float = 0.28, noise: float = 0.0, rng=None):
    """stereo corner observations float32 [16][n] of square markers (corner order of SURVEY A.6:
    (0,0,0),(s,0,0),(s,s,0),(0,s,0); the pose is that of corner 0)."""
    n = p.shape[0]
    R_RL, P_LR = stereo_extrinsics(cfg)
    R_RL_inv = np.linalg.inv(R_RL)  # true inverse: the calibration is ~2.5e-6 non-orthonormal (SURVEY A.3-5)
    cm = np.array([[0, 0, 0], [size, 0, 0], [size, size, 0], [0, size, 0]], dtype=np.float64)
    out = np.zeros((16, n))
    flip = np.array([-1.0, -1.0, 1.0])
    for i in range(4):
        XL = (p + np.einsum("nij,j->ni", Rm, cm[i])) * flip  # un-flip into the left camera frame
        XR = (XL - P_LR) @ R_RL_inv.T
        uvL = forward_project(cfg, XL)
        uvR = forward_project(cfg, XR)
        out[2 * i], out[2 * i + 1] = uvL[:, 0], uvL[:, 1]
        out[8 + 2 * i], out[8 + 2 * i + 1] = uvR[:, 0], uvR[:, 1]
    if noise > 0:
        out = out + (rng or np.random.default_rng(0)).normal(size=out.shape) * noise
    return np.ascontiguousarray(out.astype(np.float32))


def random_marker_corners(cfg: capi.FbusConfig, n: int, rng, far_fraction: float = 0.0, noise: float = 2e-4):
    Rm, p = random_marker_poses(n, rng, far_fraction)
    return marker_corners_from_pose(cfg, Rm, p, noise=noise, rng=rng)


def marker_corners_inair(cfg: capi.FbusConfig, Rm: np.ndarray, p: np.ndarray, size: float = 0.28, noise: float = 0.0, rng=None):
    """in-air (pinhole) stereo corner observations float32 [16][n] consistent with VISION::NormalTriangulation's geometry:
    x_R ~ T_L_R [X_L; 1] with T_L_R = [R_IR R_IL^T | P_LI - R P_RI] (vision.cpp:402-408)."""
    n = p.shape[0]
    TL = np.array(cfg.tsc_left, dtype=np.float64).reshape(4, 4)
    TR = np.array(cfg.tsc_right, dtype=np.float64).reshape(4, 4)
    R = TR[:3, :3] @ TL[:3, :3].T
    t = TL[:3, 3] - R @ TR[:3, 3]
    cm = np.array([[0, 0, 0], [size, 0, 0], [size, size, 0], [0, size, 0]], dtype=np.float64)
    out = np.zeros((16, n))
    flip = np.array([-1.0, -1.0, 1.0])
    for i in range(4):
        XL = (p + np.einsum("nij,j->ni", Rm, cm[i])) * flip
        XR = XL @ R.T + t
        out[2 * i], out[2 * i + 1] = XL[:, 0] / XL[:, 2], XL[:, 1] / XL[:, 2]
        out[8 + 2 * i], out[8 + 2 * i + 1] = XR[:, 0] / XR[:, 2], XR[:, 1] / XR[:, 2]
    if noise > 0:
        out = out + (rng or np.random.default_rng(0)).normal(size=out.shape) * noise
    return np.ascontiguousarray(out.astype(np.float32))


# ---------------------------------------------------------------------------------------------- config 4: marker board
def board_config(cfg: capi.FbusConfig, pitch: float = 0.35) -> capi.FbusConfig:
    """BASELINE configs[3]: markers 0-7 re-posed as a 4 x 2 planar grid (pitch 0.35 m, side 0.28 m) in the plane of marker 0"""
    import copy
    c = copy.copy(cfg)
    c.n_markers = 8
    eye = [1, 0, 0, 0, 1, 0, 0, 0, 1]
    for m in range(8):
        i, j = m % 4, m // 4
        c.marker_id[m] = m
        c.marker_pos[3 * m + 0] = (i - 1.5) * pitch
        c.marker_pos[3 * m + 1] = (j - 0.5) * pitch
        c.marker_pos[3 * m + 2] = 0.0
        for e in range(9):
            c.marker_rot[9 * m + e] = eye[e]
    return c


def board_base_corners(cfg: capi.FbusConfig, traj: dict):
    """noise-free stereo corner observations of every board marker for every frame of the truth trajectory, consistent with
    the filter's own measurement model (P_ML = R_IL R^T (P_M - p - R P_IL), Q_ML = Q_IL * conj(q) * Q_M).
    -> (corners float64 [16][W*m] with item index frame*m + slot, ids int32 [W][m])"""
    R_IL, Q_IL, P_IL = filter_extrinsics(cfg)
    m, W = cfg.n_markers, traj["truth_p"].shape[0]
    p_all, R_all = np.zeros((W * m, 3)), np.zeros((W * m, 3, 3))
    for w in range(W):
        q = traj["truth_q"][w]
        R = _q2R(q)
        for s in range(m):
            P_M = np.array(cfg.marker_pos[3 * s:3 * s + 3])
            Q_M = quat_from_rotmat(np.array(cfg.marker_rot[9 * s:9 * s + 9]).reshape(3, 3))
            p_all[w * m + s] = R_IL @ R.T @ (P_M - traj["truth_p"][w] - R @ P_IL)
            qml = _qmul(_qmul(Q_IL, _qconj(q)), Q_M)
            R_all[w * m + s] = _q2R(qml / np.linalg.norm(qml))
    n = W * m
    R_RL, P_LR = stereo_extrinsics(cfg)
    Ri = np.linalg.inv(R_RL)
    size = cfg.marker_size
    cm = np.array([[0, 0, 0], [size, 0, 0], [size, size, 0], [0, size, 0]], dtype=np.float64)
    out = np.zeros((16, n))
    flip = np.array([-1.0, -1.0, 1.0])
    for i in range(4):
        XL = (p_all + np.einsum("nij,j->ni", R_all, cm[i])) * flip
        XR = (XL - P_LR) @ Ri.T
        uvL, uvR = forward_project(cfg, XL), forward_project(cfg, XR)
        out[2 * i], out[2 * i + 1] = uvL[:, 0], uvL[:, 1]
        out[8 + 2 * i], out[9 + 2 * i] = uvR[:, 0], uvR[:, 1]
    ids = np.tile(np.arange(m, dtype=np.int32)[None, :], (W, 1))
    return np.ascontiguousarray(out), np.ascontiguousarray(ids), p_all


# white noise on the normalised corner coordinates of the logs (2e-4, the level of BASELINE configs[3] and random_marker_corners)
DEFAULT_CORNER_NOISE = 2e-4


def base_marker_poses(cfg: capi.FbusConfig, traj: dict):
    """noise-free pose of every map marker for every frame of the truth trajectory, as the filter's own measurement model
    predicts it (the first half of board_base_corners): p = R_IL R^T (P_M - p_true - R P_IL), q = Q_IL * conj(q_true) * Q_M (not
    normalised; the projection normalises it).  -> (pose float64 [W][m][7], ids int32 [W][m] = the map's marker ids)"""
    R_IL, Q_IL, P_IL = filter_extrinsics(cfg)
    m, W = cfg.n_markers, traj["truth_p"].shape[0]
    pose = np.zeros((W, m, 7))
    for w in range(W):
        q = traj["truth_q"][w]
        R = _q2R(q)
        for s in range(m):
            P_M = np.array(cfg.marker_pos[3 * s:3 * s + 3])
            Q_M = quat_from_rotmat(np.array(cfg.marker_rot[9 * s:9 * s + 9]).reshape(3, 3))
            pose[w, s, 0:3] = R_IL @ R.T @ (P_M - traj["truth_p"][w] - R @ P_IL)
            pose[w, s, 3:7] = _qmul(_qmul(Q_IL, _qconj(q)), Q_M)
    ids = np.tile(np.array(cfg.marker_id[:m], dtype=np.int32)[None, :], (W, 1))
    return np.ascontiguousarray(pose), np.ascontiguousarray(ids)


def make_corner_spec(pose: np.ndarray, ids: np.ndarray, seed: int, filter_offset: int = 0, underwater: bool = True,
                     sigma_corner: float = DEFAULT_CORNER_NOISE, p_drop: float = 0.0, p_outlier: float = 0.0,
                     sigma_outlier: float = 0.0) -> capi.CornerSpec:
    """fbus_corner_spec over base poses [W][m][7] and ids [W][m] (base_marker_poses); the arrays are kept alive by the spec"""
    pose = np.ascontiguousarray(pose, dtype=np.float64)
    ids = np.ascontiguousarray(ids, dtype=np.int32)
    assert pose.ndim == 3 and pose.shape[2] == 7 and ids.shape == pose.shape[:2], (pose.shape, ids.shape)
    sp = capi.CornerSpec()
    sp.n_frames, sp.max_markers = pose.shape[0], pose.shape[1]
    sp.base_pose = capi.dptr(pose)
    sp.base_id = capi.dptr(ids, capi.c_int32_p)
    sp.underwater = int(underwater)
    sp.sigma_corner, sp.p_drop, sp.p_outlier, sp.sigma_outlier = sigma_corner, p_drop, p_outlier, sigma_outlier
    sp.seed, sp.filter_offset = seed, filter_offset
    sp._keep = (pose, ids)
    return sp
