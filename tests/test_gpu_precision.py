"""Precision of every form of the window kernel against a 50-digit reference (mp_reference) across the measurement-noise range
of the noise sweep, measured where the NEES looks: the (position, attitude) block of P whitened by its exact value, every entry
of P on its correlation scale, and the NEES of fbus_filter_errors itself.

The yardstick is the double oracle (orc.Oracle, dense (I-KH)P with a solve of S) on the same inputs: a kernel may lose at most
RATIO times what the oracle loses against the 50-digit result, and on the committed sweep's range (R >= 1e-8) at most 1e-9.
Run with -s to print the measured ratios."""
import numpy as np
import pytest

import mp_reference as mpr
from test_gpu_noise import _errors_np, _streams
from test_precision_host import (R_GRID, RATIO, SWEEP_MIN_R, accumulate, cfg_with, check_envelope, detection, noise_of,
                                 pose_state)

pytestmark = pytest.mark.gpu

FORMS = ["lane", "lane32", "lane1", "smem", "tmem"]
BAD_STATUS = 0x2 | 0x4 | 0x8 | 0x10 | 0x20 | 0x40  # reset skipped / done, update skipped, non-finite, no detection, rejected
# the default setting and the corners of profiles/sweep_pos_quat.jsonl's (pos_n_cov, quat_n_cov) grid, and its middle
SWEEP_SETTINGS = [(1e-3, 1e-3), (1e-8, 1e-7), (1e-8, 1e-3), (1e-3, 1e-7), (1e-5, 1e-5)]
K0 = 3  # frames run before the comparison starts (past the initialisation at frame 0)


def _merge(cols):
    """one-filter state dicts -> one batch state dict"""
    return {f: np.ascontiguousarray(np.concatenate([c[f] for c in cols], axis=-1)) for f in cols[0]}


def _oracle_windows(c, traj, imu_h, id_h, pose_h, st0, cols, w0, w1):
    import orc
    from fbus_ekf_b200 import capi
    n = len(cols)
    s = capi.make_imu_stream(traj["t_imu"], np.ascontiguousarray(imu_h[:, :, cols]), n)
    d = capi.make_det_frames(traj["t_frames"], np.ascontiguousarray(id_h[:, :, cols]), np.ascontiguousarray(pose_h[:, :, :, cols]), n, 1)
    o = orc.Oracle(c, n)
    o.set_state({k: np.ascontiguousarray(v[..., cols]) for k, v in st0.items()})
    o.step_windows(s, d, traj["win_off"], w0, w1)
    return o.get_state()


@pytest.mark.parametrize("cov_store", FORMS, indirect=True)
@pytest.mark.parametrize("joseph", [False, True], ids=["standard", "joseph"])
def test_one_update_vs_50_digits(cfg, cov_store, joseph):
    """one MeasureUpdate of a batch whose filters carry R from R_GRID (fbus_set_noise), from P shaped like the suite's"""
    from fbus_ekf_b200 import BatchFilter, capi
    from test_precision_host import oracle_update
    per = 6
    rng = np.random.default_rng(41)
    settings = [noise_of(cfg, Rp, Rq) for Rp, Rq in R_GRID]
    B = per * len(settings)
    cols = [pose_state(rng) for _ in range(B)]
    dets = [detection(rng) for _ in range(B)]
    st = _merge(cols)
    noise = np.ascontiguousarray(np.repeat(np.array(settings).T, per, axis=1))
    pose = np.ascontiguousarray(np.array(dets)[:, 1:8].T.reshape(1, 1, 7, B))
    det = capi.make_det_frames(np.array([1.0]), np.zeros((1, 1, B), dtype=np.int32), pose, B, 1)
    f = BatchFilter(cfg_with(cfg, settings[0], joseph), batch=B)
    f.SetNoise(noise)
    f.SetState(st)
    f.MeasureUpdate(det, 0)
    sg = f.GetState()
    f.close()
    assert not np.any(sg["status"] & BAD_STATUS)
    refs = mpr.reference_many([("update", (settings[b // per], cols[b], dets[b])) for b in range(B)])
    for k, (Rp, Rq) in enumerate(R_GRID):
        got, ref_err = [0.0] * 3, [0.0] * 3
        c_std = cfg_with(cfg, settings[k])  # the Joseph form is held to the standard form's oracle (test_precision_host)
        for b in range(k * per, (k + 1) * per):
            mst, mP = refs[b]
            got = accumulate(got, mpr.column(sg, b), mst, mP)
            ref_err = accumulate(ref_err, oracle_update(c_std, cols[b], dets[b]), mst, mP)
        check_envelope(f"{cov_store} {'joseph' if joseph else 'standard'} update R=({Rp:g},{Rq:g})", got, ref_err,
                       min(Rp, Rq) >= SWEEP_MIN_R)


@pytest.mark.parametrize("cov_store", FORMS, indirect=True)
def test_sweep_workload_vs_50_digits(cfg, cov_store):
    """The sweep's workload (its trajectory, seed 1, a setting-major fbus_set_noise batch over the default setting and the
    corners of the committed grid), 1 s: the kernel runs to frame K0, its state is read, then the kernel and the 50-digit
    reference both continue over [K0, W).  Then fbus_filter_errors' NEES of the kernel's final state against the 50-digit
    NEES of that same state, which tests the kernel's 6x6 solve at an ill-conditioned P6 without trajectory differences."""
    from fbus_ekf_b200 import BatchFilter, capi, sweep
    runs, ncmp = 8, 3
    base = {n: getattr(cfg, n) for n in capi.NOISE_FIELDS}
    grid = [dict(base, pos_n_cov=Rp, quat_n_cov=Rq) for Rp, Rq in SWEEP_SETTINGS]
    B = runs * len(grid)
    traj, imu_d, id_d, pose_d = _streams(cfg, B, 1.0, seed=1)
    W = len(traj["t_frames"])
    f = BatchFilter(cfg, batch=B)
    f.SetNoise(sweep.noise_array(grid, runs))
    imu = capi.make_imu_stream(traj["t_imu"], imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE)
    det = capi.make_det_frames(traj["t_frames"], id_d.data_ptr(), pose_d.data_ptr(), B, 1, capi.FBUS_MEM_DEVICE)
    f.StepWindows(imu, det, traj["win_off"], 0, K0)
    st0 = f.GetState()
    f.StepWindows(imu, det, traj["win_off"], K0, W)
    sg = f.GetState()
    tp = np.ascontiguousarray(np.repeat(traj["truth_p"][-1][:, None], B, axis=1))
    tq = np.ascontiguousarray(np.repeat(traj["truth_q"][-1][:, None], B, axis=1))
    err = f.FilterErrors(tp, tq)
    f.close()
    assert st0["initialised"].all() and np.all(err[3] == 1.0)
    imu_h, id_h, pose_h = imu_d.cpu().numpy(), id_d.cpu().numpy(), pose_d.cpu().numpy()
    dets = np.concatenate([id_h[:, 0:1, :].astype(np.float64), pose_h[:, 0, :, :]], axis=1)  # [W][8][B]: id, p, q
    cmp = [s * runs + r for s in range(len(grid)) for r in range(ncmp)]
    assert not np.any(sg["status"][cmp] & BAD_STATUS), sg["status"][cmp]
    noises = [tuple(grid[b // runs][n] for n in capi.NOISE_FIELDS) for b in cmp]
    refs = dict(zip(cmp, mpr.reference_many([
        ("windows", (noises[i], mpr.column(st0, b), traj["t_imu"], imu_h[:, :, b], traj["t_frames"], dets[:, :, b],
                     traj["win_off"], K0, W)) for i, b in enumerate(cmp)])))
    for s, (Rp, Rq) in enumerate(SWEEP_SETTINGS):
        cols = cmp[s * ncmp:(s + 1) * ncmp]
        so = _oracle_windows(cfg_with(cfg, noises[s * ncmp]), traj, imu_h, id_h, pose_h, st0, cols, K0, W)
        got, ref_err = [0.0] * 3, [0.0] * 3
        for i, b in enumerate(cols):
            mst, mP = refs[b]
            got = accumulate(got, mpr.column(sg, b), mst, mP)
            ref_err = accumulate(ref_err, mpr.column(so, i), mst, mP)
        check_envelope(f"{cov_store} sweep frames [{K0},{W}) R=({Rp:g},{Rq:g})", got, ref_err, True)
    # NEES of the kernel's own final state, every filter
    ref = _errors_np(sg, tp, tq)
    for s, (Rp, Rq) in enumerate(SWEEP_SETTINGS):
        e_gpu = e_ref = 0.0
        for b in range(s * runs, (s + 1) * runs):
            exact = mpr.nees(sg, b, tp[:, b], tq[:, b])
            e_gpu = max(e_gpu, float(abs((err[2, b] - exact) / exact)))
            e_ref = max(e_ref, float(abs((ref[2, b] - exact) / exact)))
        print(f"{cov_store} NEES R=({Rp:g},{Rq:g}): relative {e_gpu:.2e} (double reference {e_ref:.2e}, x{e_gpu / max(e_ref, 1e-300):.2f})")
        assert e_gpu <= RATIO * e_ref + 1e-12, (Rp, Rq, e_gpu, e_ref)
