"""fbus_marker_project and fbus_synth_corners on the device: the forward model against its float64 NumPy restatement and
through the solves, the generated corner streams against the NumPy restatement of the generator (tests/corner_synth_ref.py),
their chunk and shard invariance, their statistics at 65,536 filters, the pipeline into the filter, the sweep's corner mode and
the argument errors."""
import copy
import ctypes as C
import json

import numpy as np
import pytest

import corner_synth_ref as ref

pytestmark = pytest.mark.gpu


def _poses(rng, n, far_fraction=0.3, max_tilt=0.6):
    """[7][n] marker poses (p, q of corner 0, flipped left-camera frame) of synth.random_marker_poses"""
    from fbus_ekf_b200 import synth
    Rm, p = synth.random_marker_poses(n, rng, far_fraction, max_tilt)
    q = np.stack([synth.quat_from_rotmat(R) for R in Rm], axis=1)
    return np.ascontiguousarray(np.concatenate([p.T, q], axis=0))


def _special_poses(cfg):
    """a paraxial corner 0 (on the left camera's axis), an unnormalised quaternion, a marker inside the port (in front of the
    camera: valid in air only), a NaN pose"""
    pose = np.zeros((7, 4))
    pose[3] = 1.0
    pose[2] = [0.8, 0.7, cfg.d_air + cfg.d_glass - 0.005, 1.0]
    pose[0:2, 1] = [0.1, -0.05]
    pose[3:7, 1] = np.array([0.9, 0.1, -0.2, 0.3]) * 1.7
    pose[0, 3] = np.nan
    return pose


def _f32_ulp_close(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.abs(a.astype(np.float64) - b.astype(np.float64)) <= np.spacing(np.maximum(np.abs(a), np.abs(b))).astype(np.float64)


@pytest.mark.parametrize("underwater", [True, False])
def test_marker_project_matches_restatement(cfg, underwater):
    import torch
    from fbus_ekf_b200 import BatchFilter, capi
    rng = np.random.default_rng(5)
    pose = np.ascontiguousarray(np.concatenate([_poses(rng, 2000), _poses(rng, 500, 0.0, 1.2), _special_poses(cfg)], axis=1))
    f = BatchFilter(cfg, batch=1)
    c, v = f.MarkerProject(pose, underwater=underwater)
    rc, rv = ref.project_poses(cfg, pose, underwater)
    assert np.array_equal(v, rv)
    assert v[-4:].tolist() == ([1, 1, 0, 0] if underwater else [1, 1, 1, 0])
    assert np.isnan(c[:, v == 0]).all() and np.isfinite(c[:, v == 1]).all()
    # 1e-12 in normalised units inside a camera's field (|u|, |v| <= 2).  The tilted near markers also put corners on rays that
    # leave the port almost grazing (|u| up to 93): there one ulp of the air angle moves u by ~1e-12 of its value, and
    # synth.forward_project itself is only that good (its bracket falls back to bisection when an iterate hits the root), so
    # those are compared relatively.
    fov = (v == 1) & (np.abs(rc).max(axis=0) <= 2.0)
    wide = (v == 1) & ~fov
    err = float(np.abs(c[:, fov] - rc[:, fov]).max())
    rel = float((np.abs(c[:, wide] - rc[:, wide]) / np.abs(rc[:, wide]).max(axis=0)).max()) if wide.any() else 0.0
    print(f"marker_project underwater={underwater}: max |device - restatement| = {err:.2e} over {int(fov.sum())} markers; "
          f"{int(wide.sum())} with grazing rays: relative {rel:.2e}")
    assert err <= 1e-12 and rel <= 1e-9
    assert c[0, -4] == 0.0 and c[1, -4] == 0.0  # paraxial corner 0 of the left camera
    # device memory: the same numbers; valid may be omitted
    pd = torch.from_numpy(pose).cuda()
    torch.cuda.synchronize()
    cd = torch.empty((16, pose.shape[1]), dtype=torch.float64, device="cuda")
    vd = torch.empty(pose.shape[1], dtype=torch.int32, device="cuda")
    f.MarkerProject(pd.data_ptr(), underwater, n=pose.shape[1], corners=cd.data_ptr(), valid=vd.data_ptr(), mem=capi.FBUS_MEM_DEVICE)
    f.Synchronize()
    assert np.array_equal(cd.cpu().numpy(), c, equal_nan=True) and np.array_equal(vd.cpu().numpy(), v)
    f.MarkerProject(pd.data_ptr(), underwater, n=pose.shape[1], corners=cd.data_ptr(), valid=None, mem=capi.FBUS_MEM_DEVICE)
    f.Synchronize()
    assert np.array_equal(cd.cpu().numpy(), c, equal_nan=True)
    f.close()


def _q_err(q, qt):
    """sign-aligned max |q - q_true| per column"""
    s = np.where(np.sum(q * qt, axis=0) < 0, -1.0, 1.0)
    return np.abs(q * s - qt).max(axis=0)


def test_round_trip_through_the_solves(cfg):
    """underwater projections through fbus_refract_solve_gn (double corners): 0 iterations give p to 1e-9; q differs from the
    truth by the closed form's rotation of (pi - 3.1415926) / 4 about the marker normal (the reference's truncated M_PI), which
    one Gauss-Newton iteration removes.  In-air projections, rounded to float32, through fbus_inair_solve."""
    from fbus_ekf_b200 import BatchFilter, capi
    rng = np.random.default_rng(6)
    pose = _poses(rng, 4000, 0.0)
    pose[3:7] /= np.linalg.norm(pose[3:7], axis=0)
    f = BatchFilter(cfg, batch=1)
    c, v = f.MarkerProject(pose, underwater=True)
    assert v.all()
    p0, _, ok0 = f.RefractSolveGN(np.ascontiguousarray(c), iters=0)
    assert ok0.all()
    ep = float(np.abs(p0[:3] - pose[:3]).max())
    # the closed-form rotation error: an angle of (pi - REF_M_PI) / 4 = 1.34e-8 rad, i.e. |dq| = 6.7e-9
    eq0 = _q_err(p0[3:7], pose[3:7])
    p1, _, _ = f.RefractSolveGN(np.ascontiguousarray(c), iters=1)
    eq1 = float(_q_err(p1[3:7], pose[3:7]).max())
    ep1 = float(np.abs(p1[:3] - pose[:3]).max())
    half = (np.pi - capi.REF_M_PI) / 8
    print(f"round trip underwater: p err {ep:.2e} (0 it), q err {eq0.min():.2e}..{eq0.max():.2e} (0 it, expected {half:.2e}), "
          f"q err {eq1:.2e} p err {ep1:.2e} (1 it)")
    assert ep <= 1e-9
    assert eq0.max() <= half + 1e-9
    assert eq1 <= 1e-9 and ep1 <= 1e-9
    # in air: float32 corners through the DLT triangulation
    ca, va = f.MarkerProject(pose, underwater=False)
    assert va.all()
    pa, _, oka = f.InAirSolve(np.ascontiguousarray(ca.astype(np.float32)))
    assert oka.all()
    epa = float(np.abs(pa[:3] - pose[:3]).max())
    eqa = float(_q_err(pa[3:7], pose[3:7]).max())
    print(f"round trip in air (float32 corners): p err {epa:.2e} m, q err {eqa:.2e}")
    # measured on a B200: 3.3e-7 m and 1.0e-6, from the float32 rounding of the corners (~3e-8) through a 0.12 m baseline
    assert epa <= 2e-6 and eqa <= 5e-6
    f.close()


def _board(cfg, duration, extra_slots=False):
    """board trajectory of BASELINE configs[3] and its base poses / ids; extra_slots adds an empty slot and a slot whose
    pose lies behind the port"""
    from fbus_ekf_b200 import synth
    bcfg = synth.board_config(cfg)
    traj = synth.truth_trajectory(bcfg, duration, standoff=1.0)
    pose, ids = synth.base_marker_poses(bcfg, traj)
    if extra_slots:
        W = pose.shape[0]
        extra = np.zeros((W, 2, 7))
        extra[:, :, 3] = 1.0
        extra[:, 0, 2] = 1.0
        extra[:, 1, 2] = 0.01  # inside the port
        pose = np.concatenate([pose, extra], axis=1)
        ids = np.concatenate([ids, np.array([[-1, 9]] * W, dtype=np.int32)], axis=1)
    return bcfg, traj, np.ascontiguousarray(pose), np.ascontiguousarray(ids)


def _synth(f, spec, w0, w1, B):
    import torch
    m = spec.max_markers
    c = torch.full((16, (w1 - w0) * m * B), 7.0, dtype=torch.float32, device="cuda")
    i = torch.full((w1 - w0, m, B), 7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()  # the fills run on torch's stream, the handle has its own
    f.SynthCorners(spec, w0, w1, c.data_ptr(), i.data_ptr())
    return c.cpu().numpy(), i.cpu().numpy()


def _base_of(f, pose, ids, underwater=True):
    """device projection of the base poses and the ids the generator starts from"""
    c, v = f.MarkerProject(np.ascontiguousarray(pose.reshape(-1, 7).T), underwater)
    bid = np.where((v == 1) & (ids.reshape(-1) >= 0), ids.reshape(-1), -1).astype(np.int32)
    return c, bid


def test_synth_noise_free_is_the_projection(cfg):
    from fbus_ekf_b200 import BatchFilter, synth
    bcfg, traj, pose, ids = _board(cfg, 0.2, extra_slots=True)
    B = 37
    f = BatchFilter(bcfg, batch=B)
    base, bid = _base_of(f, pose, ids)
    assert bid[-1] == -1 and bid[-2] == -1 and (bid[:-2] >= 0).any()
    for uw in (True, False):
        base, bid = _base_of(f, pose, ids, uw)
        c, i = _synth(f, synth.make_corner_spec(pose, ids, seed=3, underwater=uw, sigma_corner=0.0), 0, pose.shape[0], B)
        want = np.repeat(base, B, axis=1)
        live = np.repeat(bid, B) >= 0
        assert np.array_equal(i.reshape(-1), np.repeat(bid, B))
        assert np.array_equal(c[:, live], want[:, live].astype(np.float32))
        assert np.all(c[:, ~live] == 0.0)
    f.close()


@pytest.mark.parametrize("B", [1, 33, 4096])
def test_synth_matches_restatement(cfg, B):
    from fbus_ekf_b200 import BatchFilter, synth
    bcfg, traj, pose, ids = _board(cfg, 0.2 if B < 4096 else 0.08, extra_slots=True)
    W, m = pose.shape[:2]
    f = BatchFilter(bcfg, batch=B)
    base, bid = _base_of(f, pose, ids)
    kw = dict(sigma_corner=2e-4, p_drop=0.15, p_outlier=0.1, sigma_outlier=5e-3)
    seed, off = 0xDEADBEEF12345, (1 << 32) + 5
    c, i = _synth(f, synth.make_corner_spec(pose, ids, seed=seed, filter_offset=off, **kw), 1, W, B)
    rc, ri, drop, out = ref.synth_corners(base[:, m:], bid[m:], B, m, 1, seed, off, **kw)
    assert np.array_equal(i, ri)
    close = _f32_ulp_close(c, rc)
    print(f"B={B}: {int((c != rc).sum())} of {c.size} coordinates differ from the restatement by one float32 ulp; "
          f"{int(drop.sum())} dropped, {int(out.sum())} outliers")
    assert close.all()
    assert drop.any() and out.any()
    f.close()


def test_device_normals_match_restatement(cfg):
    """the Philox / Box-Muller normals of fbus_synth_streams' bias_out are the restatement's, to rounding"""
    import torch
    from fbus_ekf_b200 import BatchFilter, synth
    B, seed, off = 4096, 0x1234567890AB, 3 << 31
    traj = synth.truth_trajectory(cfg, 0.2)
    f = BatchFilter(cfg, batch=B)
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    imu = torch.empty((N, 6, B), dtype=torch.float64, device="cuda")
    did = torch.empty((W, 1, B), dtype=torch.int32, device="cuda")
    dp = torch.empty((W, 1, 7, B), dtype=torch.float64, device="cuda")
    bias = torch.empty((6, B), dtype=torch.float64, device="cuda")
    f.SynthStreams(synth.make_synth_spec(traj, seed=seed, filter_offset=off, sigma_ba=1.0, sigma_bg=1.0), imu.data_ptr(),
                   did.data_ptr(), dp.data_ptr(), bias.data_ptr())
    z = bias.cpu().numpy()
    gf = np.uint64(off) + np.arange(B, dtype=np.uint64)
    want = np.concatenate([np.stack(ref.normal2(seed, gf, 0, s)) for s in range(3)])
    err = float(np.abs(z - want).max())
    print(f"device normals vs restatement: max abs diff {err:.2e}")
    assert err <= 1e-13
    f.close()


def test_chunks_and_shards_are_bitwise_invariant(cfg):
    from fbus_ekf_b200 import BatchFilter, synth
    bcfg, traj, pose, ids = _board(cfg, 0.4, extra_slots=True)
    W, B, k = pose.shape[0], 300, 4
    kw = dict(seed=99, sigma_corner=2e-4, p_drop=0.1, p_outlier=0.1, sigma_outlier=1e-2)
    f = BatchFilter(bcfg, batch=B)
    c, i = _synth(f, synth.make_corner_spec(pose, ids, **kw), 0, W, B)
    ca, ia = _synth(f, synth.make_corner_spec(pose, ids, **kw), 0, k, B)
    cb, ib = _synth(f, synth.make_corner_spec(pose, ids, **kw), k, W, B)
    m = pose.shape[1]
    assert np.array_equal(np.concatenate([ca, cb], axis=1), c) and np.array_equal(np.concatenate([ia, ib]), i)
    f.close()
    parts = []
    for off, nb in ((0, 100), (100, 200)):
        g = BatchFilter(bcfg, batch=nb)
        parts.append(_synth(g, synth.make_corner_spec(pose, ids, filter_offset=off, **kw), 0, W, nb))
        g.close()
    cs = np.concatenate([parts[0][0].reshape(16, W, m, 100), parts[1][0].reshape(16, W, m, 200)], axis=3)
    assert np.array_equal(cs.reshape(16, -1), c)
    assert np.array_equal(np.concatenate([parts[0][1], parts[1][1]], axis=2), i)


def test_statistics_at_65536_filters(cfg):
    import torch
    from fbus_ekf_b200 import BatchFilter, synth
    bcfg, traj, pose, ids = _board(cfg, 0.08)
    W, m = pose.shape[:2]
    B, s, pd, po, so = 65536, 2e-4, 0.1, 0.05, 1e-2
    seed = 2718
    f = BatchFilter(bcfg, batch=B)
    base, bid = _base_of(f, pose, ids)
    assert (bid >= 0).all()
    c, i = _synth(f, synth.make_corner_spec(pose, ids, seed=seed, sigma_corner=s, p_drop=pd, p_outlier=po, sigma_outlier=so), 0, W, B)
    ii = i.reshape(-1)
    r = (c.astype(np.float64) - np.repeat(base, B, axis=1)) / s
    n_items = ii.size
    dropped = ii < 0
    share = dropped.mean()
    assert abs(share - pd) <= 5 * np.sqrt(pd * (1 - pd) / n_items), share
    kept = ~dropped
    outl = kept & (np.abs(r).max(axis=0) > 10.0)
    oshare = outl.sum() / kept.sum()
    assert abs(oshare - po) <= 5 * np.sqrt(po * (1 - po) / kept.sum()), oshare
    clean = r[:, kept & ~outl]
    nz = clean.size
    mean, var = clean.mean(), clean.var()
    print(f"statistics: drop share {share:.5f}, outlier share {oshare:.5f}, residual mean {mean:.2e} var {var:.5f} over {nz} values")
    assert abs(mean) <= 5 / np.sqrt(nz)
    assert abs(var - 1.0) <= 5 * np.sqrt(2.0 / nz)
    ro = r[:, outl]
    assert abs(ro.var() / (1 + (so / s) ** 2) - 1.0) <= 5 * np.sqrt(2.0 / ro.size)
    # no correlation with fbus_synth_streams' draws under the same seed (bias, IMU sample w and pose noise of frame w)
    N = traj["base_imu"].shape[0]
    imu = torch.empty((N, 6, B), dtype=torch.float64, device="cuda")
    did = torch.empty((W, 1, B), dtype=torch.int32, device="cuda")
    dp = torch.empty((W, 1, 7, B), dtype=torch.float64, device="cuda")
    bias = torch.empty((6, B), dtype=torch.float64, device="cuda")
    f.SynthStreams(synth.make_synth_spec(traj, seed=seed, sigma_ba=1.0, sigma_bg=1.0, sigma_acc=1.0, sigma_gyro=1.0, sigma_pos=1.0),
                   imu.data_ptr(), did.data_ptr(), dp.data_ptr(), bias.data_ptr())
    other = [bias.cpu().numpy()]
    for w in range(W):
        other.append(imu[w].cpu().numpy() - traj["base_imu"][w][:, None] - bias.cpu().numpy())
        other.append(dp[w, 0, :3].cpu().numpy() - traj["base_pose"][w, :3][:, None])
    other = np.concatenate(other)  # [K][B], all N(0,1)
    rr = r.reshape(16, W * m, B)
    ok = kept.reshape(W * m, B) & ~outl.reshape(W * m, B)
    worst = 0.0
    for ws in (0, m - 1, W * m - 1):
        sel = ok[ws]
        a = rr[:, ws, sel]
        b = other[:, sel]
        a = (a - a.mean(1, keepdims=True)) / a.std(1, keepdims=True)
        b = (b - b.mean(1, keepdims=True)) / b.std(1, keepdims=True)
        corr = a @ b.T / sel.sum()
        worst = max(worst, float(np.abs(corr).max()) * np.sqrt(sel.sum()))
    print(f"max |correlation| with fbus_synth_streams: {worst:.2f} sigma")
    assert worst <= 5.0
    f.close()


def test_pipeline_into_the_filter(cfg):
    """sigma = 0: fbus_solve_to_detections gives back the base poses within the float32 corner rounding; a noisy board run of
    the filter stays finite with the nearest marker and with every marker"""
    import torch
    from fbus_ekf_b200 import BatchFilter, capi, synth
    bcfg, traj, pose, ids = _board(cfg, 2.0)
    W, m = pose.shape[:2]
    B = 512
    f = BatchFilter(bcfg, batch=B)
    c = torch.empty((16, W * m * B), dtype=torch.float32, device="cuda")
    i = torch.empty((W, m, B), dtype=torch.int32, device="cuda")
    did = torch.empty((W, m, B), dtype=torch.int32, device="cuda")
    dp = torch.empty((W, m, 7, B), dtype=torch.float64, device="cuda")
    f.SynthCorners(synth.make_corner_spec(pose, ids, seed=1, sigma_corner=0.0), 0, W, c.data_ptr(), i.data_ptr())
    f.SolveToDetections(c.data_ptr(), i.data_ptr(), W, m, True, 5, did.data_ptr(), dp.data_ptr(), capi.FBUS_MEM_DEVICE)
    f.Synchronize()
    got = dp.cpu().numpy()
    assert (did.cpu().numpy() == np.repeat(ids[:, :, None], B, axis=2)).all()
    want = pose[:, :, :, None]
    ep = float(np.abs(got[:, :, :3] - want[:, :, :3]).max())
    qw = want[:, :, 3:] / np.linalg.norm(want[:, :, 3:], axis=2, keepdims=True)
    sg = np.where(np.sum(got[:, :, 3:] * qw, axis=2, keepdims=True) < 0, -1.0, 1.0)
    eq = float(np.abs(got[:, :, 3:] * sg - qw).max())
    print(f"pipeline sigma=0: p err {ep:.2e} m, q err {eq:.2e}")
    assert ep <= 1e-5 and eq <= 1e-5
    N = traj["base_imu"].shape[0]
    imu = torch.empty((N, 6, B), dtype=torch.float64, device="cuda")
    tid = torch.empty((W, 1, B), dtype=torch.int32, device="cuda")
    tpose = torch.empty((W, 1, 7, B), dtype=torch.float64, device="cuda")
    f.SynthStreams(synth.make_synth_spec(traj, seed=4), imu.data_ptr(), tid.data_ptr(), tpose.data_ptr())
    f.SynthCorners(synth.make_corner_spec(pose, ids, seed=4, p_drop=0.1, p_outlier=0.01, sigma_outlier=2e-3), 0, W, c.data_ptr(), i.data_ptr())
    f.SolveToDetections(c.data_ptr(), i.data_ptr(), W, m, True, 5, did.data_ptr(), dp.data_ptr(), capi.FBUS_MEM_DEVICE)
    f.Synchronize()
    tp = np.ascontiguousarray(np.repeat(traj["truth_p"][-1][:, None], B, axis=1))
    tq = np.ascontiguousarray(np.repeat(traj["truth_q"][-1][:, None], B, axis=1))
    for flags in (0, capi.FBUS_FLAG_ALL_MARKERS):
        fc = copy.copy(bcfg)
        fc.flags = flags
        g = BatchFilter(fc, batch=B)
        g.StepWindows(capi.make_imu_stream(traj["t_imu"], imu.data_ptr(), B, capi.FBUS_MEM_DEVICE),
                      capi.make_det_frames(traj["t_frames"], did.data_ptr(), dp.data_ptr(), B, m, capi.FBUS_MEM_DEVICE), traj["win_off"], 0, W)
        e = g.FilterErrors(tp, tq)
        print(f"pipeline flags={flags}: position RMSE {np.sqrt(e[0].mean()):.2e} m")
        assert (e[3] == 1.0).all()
        g.close()
    f.close()


def test_sweep_corner_mode(tmp_path):
    from fbus_ekf_b200 import sweep
    args = ["--set", "pos_n_cov=1e-6,1e-4", "--runs", "256", "--duration", "2"]
    outs = []
    for extra in (["--detections", "corners", "--board"], ["--detections", "corners", "--board"],
                  ["--detections", "corners", "--board", "--all-markers", "--p-drop", "0.1"], [], ["--detections", "poses"]):
        p = tmp_path / f"rows{len(outs)}.jsonl"
        assert sweep.main(args + extra + ["--out", str(p)]) == 0
        outs.append(p.read_text())
    rows = [json.loads(x) for x in outs[0].splitlines()]
    assert len(rows) == 2 and [r["pos_n_cov"] for r in rows] == [1e-6, 1e-4]
    for r in rows + [json.loads(x) for x in outs[2].splitlines()]:
        assert r["detections"] == "corners" and r["n_markers"] == 8 and r["gn_iters"] == 5 and r["n_nonfinite"] == 0
        assert np.isfinite(r["nees6_mean"]).all() and np.isfinite([r["rmse_pos_m"], r["rmse_att_rad"]]).all()
    assert json.loads(outs[2].splitlines()[0])["all_markers"] is True
    assert outs[0] == outs[1]  # deterministic
    assert outs[3] == outs[4]  # --detections poses is the default
    assert "detections" not in outs[3]


def test_argument_errors(cfg):
    import torch
    from fbus_ekf_b200 import BatchFilter, FbusError, capi, synth
    f = BatchFilter(cfg, batch=4)
    L, h = f._lib, f._h
    pose = np.zeros((7, 2))
    pose[2], pose[3] = 1.0, 1.0
    out = np.zeros((16, 2))
    assert L.fbus_marker_project(h, None, 2, 1, out.ctypes.data, None, capi.FBUS_MEM_HOST) == capi.FBUS_E_BADARG
    assert L.fbus_marker_project(h, pose.ctypes.data, 2, 1, None, None, capi.FBUS_MEM_HOST) == capi.FBUS_E_BADARG
    assert L.fbus_marker_project(h, pose.ctypes.data, 2, 2, out.ctypes.data, None, capi.FBUS_MEM_HOST) == capi.FBUS_E_BADARG
    assert L.fbus_marker_project(h, pose.ctypes.data, 2, 1, out.ctypes.data, None, 5) == capi.FBUS_E_BADARG
    assert L.fbus_marker_project(h, pose.ctypes.data, 0, 1, out.ctypes.data, None, capi.FBUS_MEM_HOST) == capi.FBUS_OK
    bpose, bids = np.zeros((3, 2, 7)), np.zeros((3, 2), dtype=np.int32)
    bpose[:, :, 2], bpose[:, :, 3] = 1.0, 1.0
    c = torch.empty((16, 3 * 2 * 4), dtype=torch.float32, device="cuda")
    i = torch.empty((3, 2, 4), dtype=torch.int32, device="cuda")

    def call(spec, w0=0, w1=3, cp=c.data_ptr(), ip=i.data_ptr()):
        return L.fbus_synth_corners(h, C.byref(spec), w0, w1, cp, ip)
    good = synth.make_corner_spec(bpose, bids, seed=1)
    assert call(good) == capi.FBUS_OK
    assert call(good, 2, 2) == capi.FBUS_OK
    assert call(good, cp=None) == capi.FBUS_E_BADARG
    assert call(good, ip=None) == capi.FBUS_E_BADARG
    assert call(good, 2, 1) == capi.FBUS_E_BADARG
    assert call(good, 0, 4) == capi.FBUS_E_BADARG
    for field, val in (("sigma_corner", -1e-4), ("sigma_outlier", -1.0), ("p_drop", -0.1), ("p_drop", 1.5), ("p_outlier", 1.01),
                       ("p_outlier", float("nan")), ("underwater", 2), ("max_markers", 0)):
        bad = synth.make_corner_spec(bpose, bids, seed=1)
        setattr(bad, field, val)
        assert call(bad) == capi.FBUS_E_BADARG, field
    for field in ("base_pose", "base_id"):
        bad = synth.make_corner_spec(bpose, bids, seed=1)
        setattr(bad, field, None)
        assert call(bad) == capi.FBUS_E_BADARG, field
    assert L.fbus_synth_corners(h, None, 0, 3, c.data_ptr(), i.data_ptr()) == capi.FBUS_E_BADARG
    with pytest.raises(FbusError):
        f.SynthCorners(synth.make_corner_spec(bpose, bids, seed=1, p_drop=2.0), 0, 3, c.data_ptr(), i.data_ptr())
    edge = synth.make_corner_spec(bpose, bids, seed=1, p_drop=1.0, p_outlier=1.0, sigma_corner=0.0)
    assert call(edge) == capi.FBUS_OK
    f.Synchronize()
    assert (i.cpu().numpy() == -1).all()  # p_drop = 1 drops every detection
    f.close()
