"""Per-filter noise covariances in one batch (fbus_set_noise), per-filter error terms (fbus_filter_errors) and the sweep built on
them, on every form of the window kernel.  Streams come from fbus_synth_streams; batches are ragged."""
import numpy as np
import pytest

from helpers import cov_close, random_states, state_close

pytestmark = pytest.mark.gpu

FORMS = ["lane", "lane32", "lane1", "smem", "tmem"]
RTOL = 1e-9


def _streams(cfg, B, duration, seed=7, offset=0):
    import torch
    from fbus_ekf_b200 import BatchFilter, synth
    traj = synth.truth_trajectory(cfg, duration)
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    g = BatchFilter(cfg, batch=B)
    imu_d = torch.empty((N, 6, B), dtype=torch.float64, device="cuda")
    id_d = torch.empty((W, 1, B), dtype=torch.int32, device="cuda")
    pose_d = torch.empty((W, 1, 7, B), dtype=torch.float64, device="cuda")
    g.SynthStreams(synth.make_synth_spec(traj, seed=seed, filter_offset=offset), imu_d.data_ptr(), id_d.data_ptr(), pose_d.data_ptr())
    g.close()
    return traj, imu_d, id_d, pose_d


def _run(cfg, B, traj, imu_d, id_d, pose_d, noise=None, f32=False, noise_mem=None):
    """one handle over the whole stream -> (trace, state)"""
    import torch
    from fbus_ekf_b200 import BatchFilter, capi
    W = len(traj["t_frames"])
    f = BatchFilter(cfg, batch=B)
    if noise is not None:
        if noise_mem == "device":
            nd = torch.from_numpy(noise).cuda()
            torch.cuda.synchronize()
            f.SetNoise(nd.data_ptr(), capi.FBUS_MEM_DEVICE)
            f.Synchronize()
        else:
            f.SetNoise(noise)
    keep = None
    if f32:
        keep = torch.from_numpy(capi.si_to_sensor(imu_d.cpu().numpy(), cfg.imu_g)).cuda()
        torch.cuda.synchronize()
        imu = capi.make_imu_stream(traj["t_imu"], keep.data_ptr(), B, capi.FBUS_MEM_DEVICE, fmt=capi.FBUS_IMU_F32_SENSOR)
    else:
        imu = capi.make_imu_stream(traj["t_imu"], imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE)
    det = capi.make_det_frames(traj["t_frames"], id_d.data_ptr(), pose_d.data_ptr(), B, 1, capi.FBUS_MEM_DEVICE)
    tr = f.StepWindows(imu, det, traj["win_off"], 0, W, trace=True)
    st = f.GetState()
    f.close()
    return tr, st


def _same(a, b):
    tra, sa = a
    trb, sb = b
    assert np.array_equal(tra, trb, equal_nan=True)
    for k in sa:
        assert np.array_equal(sa[k], sb[k], equal_nan=True), k


def _cfg_with(cfg, values):
    import copy
    from fbus_ekf_b200 import capi
    c = copy.copy(cfg)
    for n, v in zip(capi.NOISE_FIELDS, values):
        setattr(c, n, float(v))
    return c


def _settings(cfg, n, seed):
    """n settings, every value log-uniform over two decades around the config's"""
    from fbus_ekf_b200 import capi
    rng = np.random.default_rng(seed)
    base = np.array([getattr(cfg, n_) for n_ in capi.NOISE_FIELDS])
    return base[None, :] * 10.0 ** rng.uniform(-1.0, 1.0, size=(n, len(base)))


def _grouped(vals, runs):
    return np.ascontiguousarray(np.repeat(vals.T, runs, axis=1))


def _oracle_cols(cfg, traj, imu_d, id_d, pose_d, cols):
    import orc
    from fbus_ekf_b200 import capi
    n, W = len(cols), len(traj["t_frames"])
    s = capi.make_imu_stream(traj["t_imu"], np.ascontiguousarray(imu_d.cpu().numpy()[:, :, cols]), n)
    d = capi.make_det_frames(traj["t_frames"], np.ascontiguousarray(id_d.cpu().numpy()[:, :, cols]),
                             np.ascontiguousarray(pose_d.cpu().numpy()[:, :, :, cols]), n, 1)
    o = orc.Oracle(cfg, n)
    tr = np.zeros((W, 17, n))
    o.step_windows(s, d, traj["win_off"], 0, W, tr, 8)
    return tr, o.get_state()


def _sub(st, cols):
    return {k: v[..., cols] for k, v in st.items()}


def _oracle_close(run, ref):
    (tr, st), (tro, so) = run, ref
    assert np.array_equal(st["status"], so["status"])
    ok, w = state_close(st, so, RTOL)
    assert ok, w
    ok, w = cov_close(st["P"], so["P"], RTOL)
    assert ok, w
    assert np.abs(tr - tro).max() <= RTOL


@pytest.mark.parametrize("cov_store,f32", [(f, False) for f in FORMS] + [("tmem", True)], indirect=["cov_store"])
def test_config_values_change_nothing(cfg, cov_store, f32):
    from fbus_ekf_b200 import capi
    B = 207
    traj, imu_d, id_d, pose_d = _streams(cfg, B, 1.0)
    plain = _run(cfg, B, traj, imu_d, id_d, pose_d, f32=f32)
    _same(_run(cfg, B, traj, imu_d, id_d, pose_d, noise=capi.noise_from_config(cfg, B), f32=f32), plain)


@pytest.mark.parametrize("cov_store", FORMS, indirect=True)
def test_groups_of_settings(cfg, cov_store):
    runs, K = 41, 5
    B = runs * K
    vals = _settings(cfg, K, 1)
    traj, imu_d, id_d, pose_d = _streams(cfg, B, 1.0, seed=8)
    tr, st = _run(cfg, B, traj, imu_d, id_d, pose_d, noise=_grouped(vals, runs))
    assert st["initialised"].all()
    for k in range(K):
        cols = np.arange(k * runs, (k + 1) * runs)
        ck = _cfg_with(cfg, vals[k])
        trk, stk = _run(ck, B, traj, imu_d, id_d, pose_d)
        assert np.array_equal(tr[..., cols], trk[..., cols])
        for f in st:
            assert np.array_equal(st[f][..., cols], stk[f][..., cols]), (k, f)
        _oracle_close((tr[..., cols], _sub(st, cols)), _oracle_cols(ck, traj, imu_d, id_d, pose_d, cols))
    # the settings really differ
    assert not np.array_equal(st["P"][:, :runs], stk["P"][:, :runs])


@pytest.mark.parametrize("cov_store", FORMS, indirect=True)
def test_every_filter_different(cfg, cov_store):
    B = 90
    vals = _settings(cfg, B, 2)
    traj, imu_d, id_d, pose_d = _streams(cfg, B, 0.6, seed=9)
    tr, st = _run(cfg, B, traj, imu_d, id_d, pose_d, noise=np.ascontiguousarray(vals.T))
    for b in range(B):
        _oracle_close((tr[..., [b]], _sub(st, [b])), _oracle_cols(_cfg_with(cfg, vals[b]), traj, imu_d, id_d, pose_d, [b]))


@pytest.mark.parametrize("cov_store", FORMS, indirect=True)
@pytest.mark.parametrize("mode", ["joseph", "matlab"])
def test_joseph_and_matlab_modes(cfg, cov_store, mode):
    from fbus_ekf_b200 import capi
    if mode == "matlab":
        c = capi.config_matlab()
    else:
        import copy
        c = copy.copy(cfg)
        c.flags |= capi.FBUS_FLAG_JOSEPH
    runs, K = 37, 3
    B = runs * K
    vals = _settings(c, K, 3)
    traj, imu_d, id_d, pose_d = _streams(c, B, 1.0, seed=10)
    tr, st = _run(c, B, traj, imu_d, id_d, pose_d, noise=_grouped(vals, runs))
    for k in range(K):
        cols = np.arange(k * runs, (k + 1) * runs)
        trk, stk = _run(_cfg_with(c, vals[k]), B, traj, imu_d, id_d, pose_d)
        assert np.array_equal(tr[..., cols], trk[..., cols])
        for f in st:
            assert np.array_equal(st[f][..., cols], stk[f][..., cols]), (k, f)


@pytest.mark.parametrize("cov_store", FORMS, indirect=True)
def test_unfused_calls(cfg, cov_store):
    """ImuUpdate, ResetState and MeasureUpdate take every filter's own values"""
    from fbus_ekf_b200 import BatchFilter, capi
    rng = np.random.default_rng(5)
    runs, K, m, W = 23, 3, 2, 4
    B = runs * K
    vals = _settings(cfg, K, 4)
    st0 = random_states(B, rng)
    st0["prev_marker_id"][:] = rng.choice([0, 1, 5], size=B)
    n = 12
    t = 1.0 + 0.005 * (1 + np.arange(n))
    data = np.zeros((n, 6, B))
    data[:, 0:3] = rng.normal(size=(n, 3, B)) * 0.3 + np.array([0, 9.8, -0.1])[None, :, None]
    data[:, 3:6] = rng.normal(size=(n, 3, B)) * 0.05
    imu = capi.make_imu_stream(t, np.ascontiguousarray(data), B)
    ids = rng.choice([0, 1, 5], size=(W, m, B)).astype(np.int32)
    pose = np.zeros((W, m, 7, B))
    pose[:, :, 0:3] = rng.normal(size=(W, m, 3, B)) * 0.4 + np.array([0, 0, 0.8])[None, None, :, None]
    q = rng.normal(size=(W, m, 4, B))
    pose[:, :, 3:7] = q / np.linalg.norm(q, axis=2, keepdims=True)
    det = capi.make_det_frames(1.07 + 0.04 * np.arange(W), ids, np.ascontiguousarray(pose), B, m)

    def drive(c, noise=None):
        f = BatchFilter(c, batch=B)
        if noise is not None:
            f.SetNoise(noise)
        f.SetState(st0)
        out = []
        for w in range(W):
            f.ImuUpdate(imu, 3 * w, 3, 1.0 + 0.015 * (w + 1))
            f.ResetState(det, w)
            f.MeasureUpdate(det, w)
            out.append(f.GetState())
        f.close()
        return out

    got = drive(cfg, _grouped(vals, runs))
    for k in range(K):
        cols = slice(k * runs, (k + 1) * runs)
        ref = drive(_cfg_with(cfg, vals[k]))
        for w in range(W):
            for f in got[w]:
                assert np.array_equal(got[w][f][..., cols], ref[w][f][..., cols]), (k, w, f)


@pytest.mark.parametrize("cov_store", FORMS, indirect=True)
def test_set_clear_and_device_source(cfg, cov_store):
    from fbus_ekf_b200 import BatchFilter
    runs, K = 30, 3
    B = runs * K
    noise = _grouped(_settings(cfg, K, 6), runs)
    traj, imu_d, id_d, pose_d = _streams(cfg, B, 0.6, seed=12)
    plain = _run(cfg, B, traj, imu_d, id_d, pose_d)
    # set, then cleared before any stepping
    import torch
    from fbus_ekf_b200 import capi
    W = len(traj["t_frames"])
    f = BatchFilter(cfg, batch=B)
    f.SetNoise(noise)
    f.SetNoise(None)
    imu = capi.make_imu_stream(traj["t_imu"], imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE)
    det = capi.make_det_frames(traj["t_frames"], id_d.data_ptr(), pose_d.data_ptr(), B, 1, capi.FBUS_MEM_DEVICE)
    tr = f.StepWindows(imu, det, traj["win_off"], 0, W, trace=True)
    _same((tr, f.GetState()), plain)
    # host and device sources
    _same(_run(cfg, B, traj, imu_d, id_d, pose_d, noise=noise, noise_mem="device"), _run(cfg, B, traj, imu_d, id_d, pose_d, noise=noise))
    assert torch.cuda.is_available()


def _errors_np(st, tp, tq):
    B = tp.shape[1]
    ix = [0, 1, 2, 6, 7, 8]
    out = np.zeros((4, B))
    for b in range(B):
        e = np.zeros(6)
        e[:3] = st["p"][:, b] - tp[:, b]
        q = st["q"][:, b]
        qt = tq[:, b]
        cq = np.array([q[0], -q[1], -q[2], -q[3]])
        w = cq[0] * qt[0] - cq[1] * qt[1] - cq[2] * qt[2] - cq[3] * qt[3]
        v = cq[0] * qt[1:] + qt[0] * cq[1:] + np.cross(cq[1:], qt[1:])
        e[3:] = 2.0 * (-1.0 if w < 0 else 1.0) * v
        P = st["P"][:, b].reshape(18, 18)[np.ix_(ix, ix)]
        L = np.linalg.cholesky(P)
        y = np.linalg.solve(L, e)
        out[:, b] = [e[:3] @ e[:3], e[3:] @ e[3:], y @ y, 1.0]
    return out


@pytest.mark.parametrize("cov_store", FORMS, indirect=True)
def test_filter_errors(cfg, cov_store):
    from fbus_ekf_b200 import BatchFilter, capi
    runs, K = 31, 3
    B = runs * K
    traj, imu_d, id_d, pose_d = _streams(cfg, B, 1.0, seed=13)
    W = len(traj["t_frames"])
    f = BatchFilter(cfg, batch=B)
    f.SetNoise(_grouped(_settings(cfg, K, 7), runs))
    f.StepWindows(capi.make_imu_stream(traj["t_imu"], imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE),
                  capi.make_det_frames(traj["t_frames"], id_d.data_ptr(), pose_d.data_ptr(), B, 1, capi.FBUS_MEM_DEVICE), traj["win_off"], 0, W)
    tp = np.ascontiguousarray(np.repeat(traj["truth_p"][-1][:, None], B, axis=1))
    tq = np.ascontiguousarray(np.repeat(traj["truth_q"][-1][:, None], B, axis=1))
    err = f.FilterErrors(tp, tq)
    ref = _errors_np(f.GetState(), tp, tq)
    assert np.array_equal(err[3], ref[3])
    assert np.all(np.abs(err[:3] - ref[:3]) <= 1e-12 * np.abs(ref[:3]))
    st = f.Stats(tp, tq)
    ok = err[3] == 1.0
    assert np.all(np.abs(err[:3, ok].sum(1) - st[:3]) <= 1e-12 * np.abs(st[:3]))
    assert st[3] == ok.sum() and st[4] == (~ok).sum()
    assert np.sqrt(err[0, ok]).max() == st[5]
    # a non-finite filter: flag 0, counted as non-finite by fbus_stats
    s = f.GetState()
    s["p"][1, 4] = np.nan
    f.SetState(s)
    err2 = f.FilterErrors(tp, tq)
    assert err2[3, 4] == 0.0 and np.all(np.delete(err2[3], 4) == 1.0)
    assert f.Stats(tp, tq)[4] == 1
    f.close()


def test_bad_arguments(cfg):
    from fbus_ekf_b200 import BatchFilter, FbusError
    from fbus_ekf_b200 import capi
    f = BatchFilter(cfg, batch=33)
    L = capi.lib()
    assert L.fbus_set_noise(None, None, 0) == capi.FBUS_E_BADARG
    n = capi.noise_from_config(cfg, 33)
    assert L.fbus_set_noise(f._h, n.ctypes.data, 7) == capi.FBUS_E_BADARG
    assert L.fbus_filter_errors(None, None, None, 0, None, 0) == capi.FBUS_E_BADARG
    with pytest.raises(AssertionError):
        f.SetNoise(np.zeros((6, 32)))
    with pytest.raises(FbusError):
        f._ck(L.fbus_filter_errors(f._h, n.ctypes.data, n.ctypes.data, 0, n.ctypes.data, 3))
    f.close()


def test_sweep_end_to_end(cfg):
    """3 settings x 64 runs x 1 s: the row of the default-valued setting equals what a plain default handle gives on the same 64
    streams (same seed, same filter offsets), evaluated at the same times"""
    from fbus_ekf_b200 import BatchFilter, capi, sweep
    runs, seed = 64, 17
    sets = [("pos_n_cov", [cfg.pos_n_cov * 0.1, cfg.pos_n_cov, cfg.pos_n_cov * 10.0])]
    rows = sweep.run_sweep(sets, runs, 1.0, eval_every=0.2, seed=seed)
    assert len(rows) == 3 and [r["pos_n_cov"] for r in rows] == sets[0][1]
    row = rows[1]
    for n in capi.NOISE_FIELDS:
        assert row[n] == getattr(cfg, n)
    traj, imu_d, id_d, pose_d = _streams(cfg, runs, 1.0, seed=seed, offset=runs)
    W = len(traj["t_frames"])
    f = BatchFilter(cfg, batch=runs)
    imu = capi.make_imu_stream(traj["t_imu"], imu_d.data_ptr(), runs, capi.FBUS_MEM_DEVICE)
    det = capi.make_det_frames(traj["t_frames"], id_d.data_ptr(), pose_d.data_ptr(), runs, 1, capi.FBUS_MEM_DEVICE)
    w0, nees = 0, []
    ends = [5, 10, 15, 20, W]
    assert row["t_eval"] == [float(traj["t_frames"][w - 1]) for w in ends]
    for w1 in ends:
        f.StepWindows(imu, det, traj["win_off"], w0, w1)
        tp = np.ascontiguousarray(np.repeat(traj["truth_p"][w1 - 1][:, None], runs, axis=1))
        tq = np.ascontiguousarray(np.repeat(traj["truth_q"][w1 - 1][:, None], runs, axis=1))
        e = f.FilterErrors(tp, tq)
        ok = e[3] == 1.0
        nees.append(e[2, ok].mean())
        w0 = w1
    assert np.allclose(row["nees6_mean"], nees, rtol=1e-9, atol=0)
    assert np.isclose(row["rmse_pos_m"], np.sqrt(e[0, ok].mean()), rtol=1e-9, atol=0)
    assert np.isclose(row["rmse_att_rad"], np.sqrt(e[1, ok].mean()), rtol=1e-9, atol=0)
    assert row["n_nonfinite"] == int((~ok).sum())
    assert abs(row[sweep.FRAC_KEY] - (ok & (e[2] <= sweep.CHI2_6_95)).sum() / runs) <= 1.0 / runs  # a NEES at the threshold may flip
    # the settings differ in their rows
    assert rows[0]["nees6_mean"][-1] != rows[2]["nees6_mean"][-1]
