"""Precision of the structured device math (fbus_math.cuh compiled for the host by tests/host_math_harness.cpp) against a
50-digit reference (mp_reference), across the measurement-noise range of the noise sweep and below it.

cov_close scales every covariance error by max|P|, which is the gravity block; it cannot see the (position, attitude) block
that the NEES inverts once that block is small.  These tests measure the error of that block whitened by its exact value
(cov_whitened_err) and every entry's error on its correlation scale (cov_corr_err), and hold the device algorithm to a small
multiple of what the dense double oracle (LAPACK-style solve of S) loses on the same inputs.  The kernels themselves are held
to the same envelope on the GPU by test_gpu_precision.py."""
import copy
import ctypes as C
import os

import numpy as np
import pytest

import mp_reference as mpr
from helpers import cov_corr_err, cov_whitened_err, state_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (pos_n_cov, quat_n_cov): the default, the sweep's corner (1e-8, 1e-7) and beyond
R_GRID = [(1e-3, 1e-3), (1e-5, 1e-5), (1e-8, 1e-7), (1e-10, 1e-10), (1e-12, 1e-12)]
SWEEP_MIN_R = 1e-8  # the committed sweep (profiles/sweep_pos_quat.jsonl) has no R below this
RATIO = 8.0  # allowed multiple of the double oracle's own error against the 50-digit reference
FLOOR = 1e-15
ABS_MAX = 1e-9  # on the sweep's range
TRIALS = 4
STATE = ("q", "p", "v", "ba", "bg", "g")


@pytest.fixture(scope="module")
def hm(built):
    from fbus_ekf_b200 import capi
    lib = C.CDLL(os.path.join(ROOT, "tests", "_build_host_math.so"))
    P = C.POINTER(capi.FbusConfig)
    lib.hm_propagate.argtypes = [P, capi.c_double_p, capi.c_double_p, capi.c_double_p, capi.c_double_p, C.c_double]
    for n in ("hm_update", "hm_update_coop", "hm_update_joseph"):
        getattr(lib, n).argtypes = [P, capi.c_double_p, capi.c_double_p, C.c_int, capi.c_double_p, capi.c_double_p]
    return lib


def _pack(P):
    return np.array([P[i, j] for i in range(18) for j in range(i, 18)])


def _unpack(p):
    P = np.zeros((18, 18))
    iu = np.triu_indices(18)
    P[iu] = p
    P.T[iu] = p
    return P


_NOM = (("t", 1), ("q", 4), ("R", 9), ("p", 3), ("v", 3), ("ba", 3), ("bg", 3), ("g", 3))


def _nom(st):
    return np.concatenate([np.atleast_1d(st[f][..., 0]) for f, _ in _NOM]).copy()


def _from_nom(nom, P171):
    out, k = {}, 0
    for f, n in _NOM:
        out[f] = nom[k:k + n].reshape(-1, 1) if n > 1 else nom[k:k + 1].copy()
        k += n
    out["P"] = _unpack(P171).reshape(324, 1)
    return out


def pose_state(rng, t0=1.0):
    """one filter, P shaped like the suite's: pose block 1e-4 to 1e-2, gravity block 100, random correlations"""
    from fbus_ekf_b200 import capi
    import fbus_oracle_np as onp
    st = capi.alloc_state(1, True)
    A = rng.normal(size=(18, 18))
    P = A @ A.T * 1e-6 + np.diag(np.repeat([1e-4, 1e-2, 1e-4, 1e-2, 1e-2, 100.0], 3))
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    q2 = q + 1e-3 * rng.normal(size=4)  # carried rotation slightly stale (SURVEY A.3-2)
    st["q"][:, 0] = q
    st["R"][:, 0] = onp.q2R(q2 / np.linalg.norm(q2)).ravel()
    st["p"][:, 0] = rng.normal(size=3) * 0.3
    st["v"][:, 0] = rng.normal(size=3) * 0.2
    st["ba"][:, 0] = rng.normal(size=3) * 0.05
    st["bg"][:, 0] = rng.normal(size=3) * 2e-3
    st["g"][:, 0] = [9.8, 0, 0]
    st["P"][:, 0] = ((P + P.T) / 2).ravel()
    st["t"][:] = t0
    st["initialised"][:] = 1
    return st


def detection(rng):
    yP = rng.normal(size=3) * 0.2 + np.array([0, 0, 0.5])
    yQ = rng.normal(size=4)
    return np.concatenate([[0.0], yP, yQ / np.linalg.norm(yQ)])


def noise_of(cfg, Rp, Rq):
    from fbus_ekf_b200 import capi
    return tuple(float(getattr(cfg, n)) for n in capi.NOISE_FIELDS[:4]) + (Rp, Rq)


def cfg_with(cfg, noise, joseph=False):
    from fbus_ekf_b200 import capi
    c = copy.copy(cfg)
    for n, v in zip(capi.NOISE_FIELDS, noise):
        setattr(c, n, float(v))
    if joseph:
        c.flags |= capi.FBUS_FLAG_JOSEPH
    return c


def oracle_update(cfg, st, det):
    import orc
    from fbus_ekf_b200 import capi
    o = orc.Oracle(cfg, 1)
    o.set_state(st)
    pose = np.ascontiguousarray(det[1:8].reshape(1, 1, 7, 1))
    o.update(capi.make_det_frames(np.array([float(st["t"][0])]), np.zeros((1, 1, 1), dtype=np.int32), pose, 1, 1), 0)
    return o.get_state()


def check_envelope(tag, got, ref_err, in_sweep_range):
    """got / ref_err: (whitened P6, correlation-scaled P, nominal state) maxima of the tested code / of the double oracle
    against the 50-digit reference.  Prints the ratio row, then applies the gates: at most RATIO x the oracle's error
    everywhere, and at most ABS_MAX (covariance) / 1e-9 (state_close) on the sweep's range.  Below that range the state
    itself is only as good as the oracle's: at R = 1e-12 both lose ~1e-9 of dx to the conditioning of S."""
    ratio = [g / max(r, 1e-300) for g, r in zip(got, ref_err)]
    print(f"{tag}: whitened {got[0]:.2e} (oracle {ref_err[0]:.2e}, x{ratio[0]:.2f})  corr {got[1]:.2e} "
          f"(oracle {ref_err[1]:.2e}, x{ratio[1]:.2f})  state {got[2]:.1e} (oracle {ref_err[2]:.1e})")
    for g, r, name in zip(got[:2], ref_err[:2], ("whitened P6", "correlation-scaled P")):
        assert g <= RATIO * r + FLOOR, f"{tag}: {name} error {g:.3e} > {RATIO} x oracle {r:.3e}"
        if in_sweep_range:
            assert g <= ABS_MAX, f"{tag}: {name} error {g:.3e} > {ABS_MAX} on the sweep's range"
    assert got[2] <= (1e-9 if in_sweep_range else max(1e-9, RATIO * ref_err[2])), \
        f"{tag}: nominal state differs from the 50-digit reference by {got[2]:.3e} (oracle {ref_err[2]:.3e})"


def accumulate(acc, st, ref_state, ref_P):
    """running maxima of (whitened P6, correlation-scaled P, state_close) errors of `st` against the 50-digit result"""
    P = np.asarray(st["P"])[:, 0]
    e = (cov_whitened_err(P, ref_P), cov_corr_err(P, ref_P), state_close(st, ref_state, 1.0, fields=STATE)[1])
    return [max(a, b) for a, b in zip(acc, e)]


def _cases(cfg, Rp, Rq, seed):
    rng = np.random.default_rng(seed)
    noise = noise_of(cfg, Rp, Rq)
    cases = [(pose_state(rng), detection(rng)) for _ in range(TRIALS)]
    refs = mpr.reference_many([("update", (noise, st, det)) for st, det in cases])
    return noise, cases, refs


@pytest.mark.parametrize("entry", ["hm_update", "hm_update_coop", "hm_update_joseph"])
@pytest.mark.parametrize("Rp,Rq", R_GRID)
def test_update_vs_50_digits(cfg, hm, entry, Rp, Rq):
    from fbus_ekf_b200 import capi
    noise, cases, refs = _cases(cfg, Rp, Rq, seed=100 + R_GRID.index((Rp, Rq)))
    ck = cfg_with(cfg, noise, joseph=entry == "hm_update_joseph")
    # The yardstick is the oracle's standard form (I-KH)P for the Joseph entry too.  The device evaluates Joseph in the
    # reduced form P - G^T C_J G, which subtracts from P like the standard form and so cannot reach the accuracy of the
    # oracle's dense (I-KH) P (I-KH)^T + K R K^T (see DESIGN.md, "Numerical envelope of the update").
    c_std = cfg_with(cfg, noise)
    got, ref_err = [0.0] * 3, [0.0] * 3
    for (st, det), (mst, mP) in zip(cases, refs):
        so = oracle_update(c_std, st, det)
        P171 = _pack(st["P"][:, 0].reshape(18, 18))
        nom = _nom(st)
        yP, yQ = np.ascontiguousarray(det[1:4]), np.ascontiguousarray(det[4:8])
        assert getattr(hm, entry)(C.byref(ck), capi.dptr(P171), capi.dptr(nom), 0, capi.dptr(yP), capi.dptr(yQ)) == 0
        got = accumulate(got, _from_nom(nom, P171), mst, mP)
        ref_err = accumulate(ref_err, so, mst, mP)
    check_envelope(f"{entry} R=({Rp:g},{Rq:g})", got, ref_err, min(Rp, Rq) >= SWEEP_MIN_R)


@pytest.mark.parametrize("small_gyro", [False, True])
def test_propagate_from_converged_pose_vs_50_digits(cfg, hm, small_gyro):
    """one window of IMU samples (8 x 5 ms) from a pose block that one update at R = 1e-10 shrank to ~1e-10"""
    import orc
    from fbus_ekf_b200 import capi
    rng = np.random.default_rng(31 + small_gyro)
    noise = noise_of(cfg, 1e-10, 1e-10)
    ck = cfg_with(cfg, noise)
    n, dt = 8, 0.005
    got, ref_err = [0.0] * 3, [0.0] * 3
    jobs, cases = [], []
    for _ in range(TRIALS):
        st = oracle_update(ck, pose_state(rng), detection(rng))
        assert np.asarray(st["P"])[:, 0].reshape(18, 18)[0, 0] < 1e-9
        t = float(st["t"][0]) + dt * (1 + np.arange(n))
        imu = np.zeros((n, 6))
        imu[:, 0:3] = rng.normal(size=(n, 3)) * 0.3 + np.array([0, 9.8, -0.1])
        imu[:, 3:6] = rng.normal(size=(n, 3)) * (1e-6 if small_gyro else 0.05)
        cases.append((st, t, imu))
        jobs.append(("propagate", (noise, st, t, imu)))
    for (st, t, imu), (mst, mP) in zip(cases, mpr.reference_many(jobs)):
        o = orc.Oracle(ck, 1)
        o.set_state(st)
        o.propagate(capi.make_imu_stream(t, np.ascontiguousarray(imu.reshape(n, 6, 1)), 1), 0, n, t[-1])
        so = o.get_state()
        P171, nom = _pack(st["P"][:, 0].reshape(18, 18)), _nom(st)
        for i in range(n):
            h = float(t[i] - (t[i - 1] if i else float(st["t"][0])))
            a, g = np.ascontiguousarray(imu[i, 0:3]), np.ascontiguousarray(imu[i, 3:6])
            assert hm.hm_propagate(C.byref(ck), capi.dptr(P171), capi.dptr(nom), capi.dptr(a), capi.dptr(g), h) == 0
        got = accumulate(got, _from_nom(nom, P171), mst, mP)
        ref_err = accumulate(ref_err, so, mst, mP)
    check_envelope(f"hm_propagate x{n} small_gyro={small_gyro}", got, ref_err, True)
