"""50-digit reference of one filter (TEST INFRASTRUCTURE, not a test module).

Restates fbus_oracle_np.Filter line for line in mpmath at DPS decimal digits, so that the covariance the kernels (and the
double oracles) compute can be compared with what exact arithmetic gives on the same inputs:

- the inputs are the doubles a kernel saw (a state from GetState, stream values copied back from the device) and the
  constants of fbus_oracle_np.Consts, each converted to mpmath exactly;
- update_covariance / update_nominal follow filter.cpp:533-616, including the `wn > 10e-5` branch and the carried rotation
  that the measurement update does not refresh (SURVEY A.3-2);
- observation_update solves S exactly.  The standard (I-KH)P and the Joseph form are equal in exact arithmetic, so one
  reference serves both;
- windows_job drives fused frames [w0, w1) of a stream in which the filter gets one known-marker detection every frame and
  no reset gap (the caller checks the kernel's status for that).

F P F^T uses F's block sparsity.  `reference_many` evaluates many independent jobs in a process pool and caches results per
job key at module scope, so test modules that share inputs pay for them once.
"""
from __future__ import annotations

import concurrent.futures as cf
import multiprocessing
import os

import mpmath as mp
import numpy as np

import fbus_oracle_np as onp

DPS = 50
IX6 = (0, 1, 2, 6, 7, 8)  # (position, attitude) rows / columns of P
NOISE_FIELDS = ("accel_n_cov", "gyro_n_cov", "accel_b_cov", "gyro_b_cov", "pos_n_cov", "quat_n_cov")
mp.mp.dps = DPS


# ----------------------------------------------------------------------------- conversions
def mpa(a):
    """float64 array -> object array of mpf (exact: every double is an mpf)"""
    a = np.asarray(a)
    if a.dtype == object:
        return a
    out = np.empty(a.shape, dtype=object)
    for i, x in np.ndenumerate(a.astype(np.float64)):
        out[i] = mp.mpf(float(x))
    return out


def to_np(a):
    """object array of mpf -> float64 (round to nearest)"""
    a = np.asarray(a, dtype=object)
    out = np.empty(a.shape)
    for i, x in np.ndenumerate(a):
        out[i] = float(x)
    return out


def _eye(n):
    out = np.empty((n, n), dtype=object)
    for i in range(n):
        for j in range(n):
            out[i, j] = mp.mpf(1 if i == j else 0)
    return out


def _zeros(*shape):
    out = np.empty(shape, dtype=object)
    out.fill(mp.mpf(0))
    return out


def _norm(v):
    return mp.sqrt(sum(x * x for x in v))


def _inv(M):
    """exact-ish (DPS digits) inverse of a small square object matrix"""
    n = M.shape[0]
    Mi = mp.inverse(mp.matrix([[M[i, j] for j in range(n)] for i in range(n)]))
    return np.array([[Mi[i, j] for j in range(n)] for i in range(n)], dtype=object)


def _chol(M):
    n = M.shape[0]
    L = mp.cholesky(mp.matrix([[M[i, j] for j in range(n)] for i in range(n)]))
    return np.array([[L[i, j] for j in range(n)] for i in range(n)], dtype=object)


# ----------------------------------------------------------------------------- quaternion / rotation helpers (fbus_oracle_np)
def skew(v):
    z = mp.mpf(0)
    return np.array([[z, -v[2], v[1]], [v[2], z, -v[0]], [-v[1], v[0], z]], dtype=object)


def quat_left(q):
    w, x, y, z = q
    return np.array([[w, -x, -y, -z], [x, w, -z, y], [y, z, w, -x], [z, -y, x, w]], dtype=object)


def quat_right(q):
    w, x, y, z = q
    return np.array([[w, -x, -y, -z], [x, w, z, -y], [y, -z, w, x], [z, y, -x, w]], dtype=object)


def qmul(a, b):
    return quat_left(a) @ np.asarray(b, dtype=object)


def qconj(a):
    return np.array([a[0], -a[1], -a[2], -a[3]], dtype=object)


def q2R(q):
    w, x, y, z = q
    tx, ty, tz = 2 * x, 2 * y, 2 * z
    twx, twy, twz = tx * w, ty * w, tz * w
    txx, txy, txz = tx * x, ty * x, tz * x
    tyy, tyz, tzz = ty * y, tz * y, tz * z
    return np.array([[1 - (tyy + tzz), txy - twz, txz + twy],
                     [txy + twz, 1 - (txx + tzz), tyz - twx],
                     [txz - twy, tyz + twx, 1 - (txx + tyy)]], dtype=object)


# ----------------------------------------------------------------------------- constants
class Consts:
    """fbus_oracle_np.Consts of the default configuration with the six noise values of one filter, converted exactly"""

    def __init__(self, noise=None):
        cfg = onp.default_config()
        if noise is not None:
            for n, v in zip(NOISE_FIELDS, noise):
                setattr(cfg, n, float(v))
        k = onp.Consts(cfg)
        self.R_IL, self.Q_IL, self.P_IL = mpa(k.R_IL), mpa(k.Q_IL), mpa(k.P_IL)
        self.markers = {mid: (mpa(p), mpa(q)) for mid, (p, q) in k.markers.items()}
        self.Qbar = mpa(k.Qbar)
        self.Rn = mpa(np.diag(k.Rn))
        self.reset_gap = mp.mpf(cfg.reset_gap)
        self.marker_max_dist = mp.mpf(cfg.marker_max_dist)


# ----------------------------------------------------------------------------- one filter
class Filter:
    """fbus_oracle_np.Filter in mpmath, built from one column of a fbus_state_soa dict (capi.alloc_state layout)"""

    def __init__(self, k: Consts, st: dict, b: int = 0):
        self.k = k
        col = lambda f: mpa(np.asarray(st[f])[..., b])  # noqa: E731
        self.t = col("t")[()]
        self.q, self.R = col("q"), col("R").reshape(3, 3)
        self.p, self.v, self.ba, self.bg, self.g = col("p"), col("v"), col("ba"), col("bg"), col("g")
        self.P = col("P").reshape(18, 18)
        self.prev_marker_id = int(np.asarray(st["prev_marker_id"])[b])

    def state(self) -> dict:
        """the nominal state and P as float64 columns ([n][1], capi.alloc_state layout)"""
        out = {f: to_np(getattr(self, f)).reshape(-1, 1) for f in ("q", "p", "v", "ba", "bg", "g")}
        out["t"] = np.array([float(self.t)])
        out["R"] = to_np(self.R).reshape(9, 1)
        out["P"] = to_np(self.P).reshape(324, 1)
        return out

    # filter.cpp:588-616: P <- F P F^T + diag(Qbar), F = I except the blocks below (3x3 blocks, block row/col 0..5)
    #   F01 = dt I, F12 = -R [a]x dt, F13 = -R dt, F15 = dt I, F22 = I - [w]x dt, F24 = -dt I
    def update_covariance(self, dt, accel, gyro):
        w = gyro - self.bg
        a = accel - self.ba
        F12 = -(self.R @ skew(a)) * dt
        F13 = -self.R * dt
        F22 = _eye(3) - skew(w) * dt
        P = self.P
        B = [P[3 * i:3 * i + 3, :] for i in range(6)]  # block rows of P
        FP = P.copy()
        FP[0:3, :] = B[0] + B[1] * dt
        FP[3:6, :] = B[1] + F12 @ B[2] + F13 @ B[3] + B[5] * dt
        FP[6:9, :] = F22 @ B[2] - B[4] * dt
        C = [FP[:, 3 * i:3 * i + 3] for i in range(6)]  # block columns of F P
        Pn = FP.copy()
        Pn[:, 0:3] = C[0] + C[1] * dt
        Pn[:, 3:6] = C[1] + C[2] @ F12.T + C[3] @ F13.T + C[5] * dt
        Pn[:, 6:9] = C[2] @ F22.T - C[4] * dt
        for i in range(18):
            Pn[i, i] = Pn[i, i] + self.k.Qbar[i]
        self.P = (Pn + Pn.T) / 2

    # filter.cpp:533-582
    def update_nominal(self, dt, accel, gyro):
        w = gyro - self.bg
        wn = _norm(w)
        R0 = q2R(self.q)
        one = mp.mpf(1)
        if wn > mp.mpf(10e-5):
            ax = w / wn
            ah = wn * dt / 2
            qh = qmul(self.q, np.concatenate([[mp.cos(ah / 2)], mp.sin(ah / 2) * ax]))
            af = wn * dt
            qn = qmul(self.q, np.concatenate([[mp.cos(af / 2)], mp.sin(af / 2) * ax]))
        else:
            qh = qmul(self.q, np.concatenate([[one], mp.mpf("0.5") * dt * w / 2]))
            qn = qmul(self.q, np.concatenate([[one], mp.mpf("0.5") * dt * w]))
        qh = qh / _norm(qh)
        self.q = qn / _norm(qn)
        Rh = q2R(qh)
        self.R = q2R(self.q)
        a = accel - self.ba
        k1 = R0 @ a + self.g
        k2 = Rh @ a + self.g
        k3 = k2
        k4 = self.R @ a + self.g
        v0 = self.v.copy()
        self.v = v0 + dt / 6 * (k1 + 2 * k2 + 2 * k3 + k4)
        self.p = self.p + dt / 6 * (v0 + 2 * (v0 + k1 * dt / 2) + 2 * (v0 + k2 * dt / 2) + (v0 + k3 * dt / 2))

    # filter.cpp:483-531
    def batch_imu(self, t_rows, imu_rows, t_end):
        start = self.t
        for t, row in zip(t_rows, imu_rows):
            if t < start:
                continue
            if t > t_end:
                break
            dt = t - self.t
            self.update_covariance(dt, row[0:3], row[3:6])
            self.update_nominal(dt, row[0:3], row[3:6])
            self.t = t

    def measurement_model(self, d):
        """(hP, hQ, H) for detection d = (id, p(3), q(4)) before the sign choice (filter.cpp:677-694)"""
        k = self.k
        P_M, Q_M = k.markers[int(d[0])]
        hP = k.R_IL @ self.R.T @ (P_M - self.p - self.R @ k.P_IL)
        hQ = qmul(qmul(k.Q_IL, qconj(self.q)), Q_M)
        H = _zeros(7, 18)
        H[0:3, 0:3] = -(k.R_IL @ self.R.T)
        H[0:3, 6:9] = k.R_IL @ skew(self.R.T @ (P_M - self.p))
        L1 = _zeros(4, 3)
        L1[1:4, :] = _eye(3) / 2
        L2 = _eye(4)
        for i in range(1, 4):
            L2[i, i] = -L2[i, i]
        H[3:7, 6:9] = quat_right(Q_M) @ quat_left(k.Q_IL) @ L2 @ quat_left(self.q) @ L1
        return hP, hQ, H

    # filter.cpp:622-739 for a frame with one detection (the marker-switch rule then always picks it)
    def observation_update(self, d):
        d = mpa(np.asarray(d, dtype=np.float64))
        k = self.k
        assert int(d[0]) in k.markers
        self.prev_marker_id = int(d[0])
        hP, hQ, H = self.measurement_model(d)
        yP, yQ = d[1:4], d[4:8]
        if sum((yQ - hQ) ** 2) > sum((yQ + hQ) ** 2):
            hQ = -hQ
            H[3:7, 6:9] = -H[3:7, 6:9]
        # H only has columns {0,1,2,6,7,8}: S = Hs P6 Hs^T + R, K^T = S^-1 Hs G with G = P[IX6, :]
        ix = list(IX6)
        Hs = H[:, ix]
        G = self.P[ix, :]
        HP = Hs @ G
        S = Hs @ G[:, ix].T @ Hs.T
        for i in range(7):
            S[i, i] = S[i, i] + k.Rn[i]
        KT = _inv(S) @ HP
        r = np.concatenate([yP - hP, yQ - hQ])
        dx = KT.T @ r
        self.p = self.p + dx[0:3]
        self.v = self.v + dx[3:6]
        th = dx[6:9]
        vn = _norm(th)
        dq = np.concatenate([[mp.cos(vn / 2)], th / vn * mp.sin(vn / 2)])
        q = qmul(self.q, dq)
        self.q = q / _norm(q)  # R not refreshed (SURVEY A.3-2)
        self.ba = self.ba + dx[9:12]
        self.bg = self.bg + dx[12:15]
        self.g = self.g + dx[15:18]
        P = self.P - KT.T @ HP
        self.P = (P + P.T) / 2

    # one fused frame (FilterThreadFunction, SURVEY A.2) of an initialised filter: reset check, IMU batch, update
    def window(self, t_det, t_rows, imu_rows, det):
        t_det = mp.mpf(float(t_det))
        # reset_state: with one detection in range and no gap it only refreshes pv/qv, which nothing here reads
        assert np.linalg.norm(np.asarray(det[1:4], dtype=np.float64)) <= float(self.k.marker_max_dist)
        assert not (t_det - self.t > self.k.reset_gap), "reset gap: the reference would overwrite the state"
        self.batch_imu(mpa(t_rows), mpa(imu_rows), t_det)
        self.observation_update(det)


def nees(st: dict, b: int, truth_p, truth_q):
    """6-dof NEES of column b of a state against a truth, exact: e = [p - p_true, 2 sign(w) vec(conj(q) q_true)],
    e^T P6^-1 e (the terms of fbus_filter_errors)"""
    p, q = mpa(np.asarray(st["p"])[:, b]), mpa(np.asarray(st["q"])[:, b])
    tp, tq = mpa(np.asarray(truth_p, dtype=np.float64)), mpa(np.asarray(truth_q, dtype=np.float64))
    d = qmul(qconj(q), tq)
    e = np.concatenate([p - tp, 2 * (-1 if d[0] < 0 else 1) * d[1:4]])
    P6 = mpa(np.asarray(st["P"])[:, b].reshape(18, 18)[np.ix_(IX6, IX6)])
    return e @ _inv(P6) @ e


# ----------------------------------------------------------------------------- jobs
def update_job(noise, st: dict, det):
    """one measurement update of a single-column state -> the exact updated Filter"""
    f = Filter(Consts(noise), st, 0)
    f.observation_update(det)
    return f


def propagate_job(noise, st: dict, t_rows, imu_rows):
    """IMU samples (t [n], rows [n][6]) -> the exact propagated Filter (no start / end filtering)"""
    f = Filter(Consts(noise), st, 0)
    for t, row in zip(mpa(t_rows), mpa(imu_rows)):
        dt = t - f.t
        f.update_covariance(dt, row[0:3], row[3:6])
        f.update_nominal(dt, row[0:3], row[3:6])
        f.t = t
    return f


def windows_job(noise, st: dict, t_imu, imu, t_frames, dets, win_off, w0, w1):
    """fused frames [w0, w1) of one filter's stream: imu [N][6], dets [W][8] (id, p, q), win_off [W+1]"""
    f = Filter(Consts(noise), st, 0)
    for w in range(w0, w1):
        s0, s1 = int(win_off[w]), int(win_off[w + 1])
        f.window(t_frames[w], t_imu[s0:s1], imu[s0:s1], dets[w])
    return f


def _run(job):
    kind, args = job
    f = {"update": update_job, "propagate": propagate_job, "windows": windows_job}[kind](*args)
    return f.state(), f.P


def _key(job):
    import hashlib
    import pickle
    return hashlib.sha1(pickle.dumps(job, protocol=4)).hexdigest()


_CACHE: dict = {}


def reference_many(jobs, workers: int | None = None):
    """[(kind, args), ...] -> [(state dict of float64 columns, exact P as an 18x18 object array), ...]; cached per job"""
    keys = [_key(j) for j in jobs]
    todo = {k: j for k, j in zip(keys, jobs) if k not in _CACHE}
    if todo:
        n = min(len(todo), workers or min(8, os.cpu_count() or 1))
        if n <= 1:
            for k, j in todo.items():
                _CACHE[k] = _run(j)
        else:
            # spawn: the caller may hold a CUDA context and threads, which a forked child must not inherit
            with cf.ProcessPoolExecutor(n, mp_context=multiprocessing.get_context("spawn")) as ex:
                for k, r in zip(todo, ex.map(_run, todo.values())):
                    _CACHE[k] = r
    return [_CACHE[k] for k in keys]


def column(st: dict, b: int) -> dict:
    """column b of a state dict as a one-filter state dict"""
    return {f: np.ascontiguousarray(np.asarray(v)[..., b:b + 1]) for f, v in st.items()}
