"""Host-side parts of the corner-level Monte-Carlo workload: the NumPy restatement of the device generator (Philox4x32-10,
Box-Muller, the rules of fbus_synth_corners), the base marker poses, the ctypes mirror of fbus_corner_spec and the corner
mode of the noise-tuning sweep.  No GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import corner_synth_ref as ref
from fbus_ekf_b200 import capi, sweep, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_philox_known_answer():
    """Philox4x32-10 of counter 0, key 0 (the published known-answer vector of the Random123 family)"""
    r = ref.philox4x32_10(0, 0, 0, 0, 0, 0)
    assert [int(v) for v in r] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]


def test_normal2_is_box_muller_of_two_53_bit_uniforms():
    seed, filt, idx, st = 0x123456789ABCDEF, np.arange(5, dtype=np.uint64) + (1 << 33), 7, 64
    z0, z1 = ref.normal2(seed, filt, idx, st)
    r = ref.philox4x32_10(filt & ref.MASK, filt >> np.uint64(32), idx, st, seed & 0xFFFFFFFF, seed >> 32)
    a = [(int(r[0][k]) << 32 | int(r[1][k])) >> 11 for k in range(5)]
    bb = [(int(r[2][k]) << 32 | int(r[3][k])) >> 11 for k in range(5)]
    for k in range(5):
        rad = np.sqrt(-2.0 * np.log((a[k] + 1) / 2.0 ** 53))
        ang = 2.0 * np.pi * bb[k] / 2.0 ** 53
        assert z0[k] == pytest.approx(rad * np.cos(ang), abs=1e-14)
        assert z1[k] == pytest.approx(rad * np.sin(ang), abs=1e-14)
    # the high word of the filter index and the stream enter the counter
    assert not np.array_equal(ref.normal2(seed, filt & ref.MASK, idx, st)[0], z0)
    assert not np.array_equal(ref.normal2(seed, filt, idx, st + 1)[0], z0)


def test_base_marker_poses_reproduce_board_corners(cfg):
    """base_marker_poses + the forward model on synth.forward_project == synth.board_base_corners, bit for bit"""
    bcfg = synth.board_config(cfg)
    traj = synth.truth_trajectory(bcfg, 1.0, standoff=1.0)
    pose, ids = synth.base_marker_poses(bcfg, traj)
    W, m = traj["truth_p"].shape[0], bcfg.n_markers
    assert pose.shape == (W, m, 7) and ids.shape == (W, m) and ids.dtype == np.int32
    base, bids, p_all = synth.board_base_corners(bcfg, traj)
    assert np.array_equal(ids, bids)
    assert np.array_equal(pose.reshape(-1, 7)[:, :3], p_all)
    corners, valid = ref.project_poses(bcfg, pose.reshape(-1, 7).T, underwater=True)
    assert valid.all()
    assert np.array_equal(corners, base)


def test_base_marker_poses_default_map(cfg):
    """every marker of the default map, with the map's own ids; marker 0's pose is the trajectory's single-marker pose"""
    traj = synth.truth_trajectory(cfg, 0.4)
    pose, ids = synth.base_marker_poses(cfg, traj)
    assert pose.shape == (10, cfg.n_markers, 7)
    assert np.array_equal(ids[0], np.array(cfg.marker_id[:cfg.n_markers], dtype=np.int32))
    s0 = list(cfg.marker_id[:cfg.n_markers]).index(0)
    assert np.allclose(pose[:, s0], traj["base_pose"], rtol=0, atol=1e-15)


def test_forward_model_validity_rule(cfg):
    """a corner at or behind the port (in air: behind the camera) makes the item invalid and NaN"""
    n = 3
    pose = np.zeros((7, n))
    pose[3] = 1.0
    pose[2] = [1.0, cfg.d_air + cfg.d_glass - 0.01, -0.5]
    pose[0], pose[1] = -0.14, -0.14
    c, v = ref.project_poses(cfg, pose, underwater=True)
    assert list(v) == [1, 0, 0]
    assert np.isfinite(c[:, 0]).all() and np.isnan(c[:, 1:]).all()
    c, v = ref.project_poses(cfg, pose, underwater=False)
    assert list(v) == [1, 1, 0]


def _rules_base(nws, rng):
    base = rng.uniform(-0.3, 0.3, size=(16, nws))
    bid = rng.integers(-1, 5, size=nws).astype(np.int32)
    return base, bid


def test_restated_rules_drop_outlier_and_empty_slots():
    rng = np.random.default_rng(3)
    m, nw, B = 3, 4, 50
    base, bid = _rules_base(nw * m, rng)
    c, ids, drop, out = ref.synth_corners(base, bid, B, m, w0=2, seed=9, sigma_corner=1e-3, p_drop=0.3, p_outlier=0.4,
                                          sigma_outlier=0.05)
    assert c.dtype == np.float32 and c.shape == (16, nw * m * B) and ids.shape == (nw, m, B)
    flat = ids.reshape(-1)
    empty = np.repeat(bid < 0, B)
    assert np.all(flat[empty] == -1) and not drop[empty].any() and not out[empty].any()
    assert np.all(flat[drop] == -1) and not (drop & out).any()
    assert np.all(c[:, flat < 0] == 0.0)
    live = flat >= 0
    resid = c[:, live].astype(np.float64) - base[:, np.repeat(np.arange(nw * m), B)[live]]
    assert np.abs(resid[:, ~out[live]]).max() < 1e-2  # white noise only
    assert np.abs(resid[:, out[live]]).max() > 5e-2   # outliers carry the extra std
    # sigma = 0 and no drop: float32 of the base, for every filter
    c0, ids0, _, _ = ref.synth_corners(base, bid, B, m, w0=0, seed=9)
    keep = np.repeat(bid >= 0, B)
    assert np.array_equal(c0[:, keep], base[:, np.repeat(np.arange(nw * m), B)[keep]].astype(np.float32))


def test_restated_streams_are_chunk_and_shard_invariant():
    rng = np.random.default_rng(4)
    m, nw, B = 2, 6, 40
    base, bid = _rules_base(nw * m, rng)
    kw = dict(seed=77, sigma_corner=1e-3, p_drop=0.2, p_outlier=0.2, sigma_outlier=0.01)
    full, ids, _, _ = ref.synth_corners(base, bid, B, m, 0, **kw)
    full = full.reshape(16, nw, m, B)
    a, ia, _, _ = ref.synth_corners(base[:, :2 * m], bid[:2 * m], B, m, 0, **kw)
    b, ib, _, _ = ref.synth_corners(base[:, 2 * m:], bid[2 * m:], B, m, 2, **kw)
    assert np.array_equal(np.concatenate([a.reshape(16, 2, m, B), b.reshape(16, nw - 2, m, B)], axis=1), full)
    assert np.array_equal(np.concatenate([ia, ib]), ids)
    s0, j0, _, _ = ref.synth_corners(base, bid, 15, m, 0, filter_offset=0, **kw)
    s1, j1, _, _ = ref.synth_corners(base, bid, B - 15, m, 0, filter_offset=15, **kw)
    assert np.array_equal(np.concatenate([s0.reshape(16, nw, m, 15), s1.reshape(16, nw, m, B - 15)], axis=3), full)
    assert np.array_equal(np.concatenate([j0, j1], axis=2), ids)


def test_corner_spec_mirror_matches_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu %%zu %%zu\\n", '
                   'sizeof(fbus_corner_spec), offsetof(fbus_corner_spec, sigma_corner), offsetof(fbus_corner_spec, seed));'
                   'return 0;}\n' % os.path.join(ROOT, "include", "fbus_ekf.h"))
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert sizes == [C.sizeof(capi.CornerSpec), capi.CornerSpec.sigma_corner.offset, capi.CornerSpec.seed.offset]


def test_make_corner_spec_fields():
    pose = np.zeros((3, 2, 7))
    ids = np.array([[0, -1]] * 3, dtype=np.int32)
    sp = synth.make_corner_spec(pose, ids, seed=5, filter_offset=7, underwater=False, p_drop=0.1)
    assert (sp.n_frames, sp.max_markers, sp.underwater, sp.seed, sp.filter_offset) == (3, 2, 0, 5, 7)
    assert sp.sigma_corner == synth.DEFAULT_CORNER_NOISE == 2e-4 and sp.p_drop == 0.1 and sp.p_outlier == 0.0
    assert sp.base_id[1] == -1


def _args(argv):
    """sweep.main's parsed corner options, with run_sweep replaced by a recorder"""
    captured = {}

    def fake_run(sets, runs, duration, eval_every, seed, device, log=None, corners=None):
        captured.update(sets=sets, runs=runs, corners=corners)
        return []
    orig = sweep.run_sweep
    sweep.run_sweep = fake_run
    try:
        sweep.main(argv)
    finally:
        sweep.run_sweep = orig
    return captured


def test_sweep_corner_arguments():
    c = _args(["--detections", "corners", "--board", "--p-drop", "0.1", "--all-markers", "--set", "pos_n_cov=1e-6"])["corners"]
    assert c == dict(board=True, corner_noise=2e-4, p_drop=0.1, p_outlier=0.0, sigma_outlier=0.0, gn_iters=5, all_markers=True)
    c = _args(["--detections", "corners", "--corner-noise", "5e-4", "--gn-iters", "0", "--p-outlier", "0.01",
               "--sigma-outlier", "0.02"])["corners"]
    assert c == dict(board=False, corner_noise=5e-4, p_drop=0.0, p_outlier=0.01, sigma_outlier=0.02, gn_iters=0, all_markers=False)
    assert _args([])["corners"] is None
    assert _args(["--detections", "poses"])["corners"] is None


@pytest.mark.parametrize("bad", [["--board"], ["--all-markers"], ["--corner-noise", "1e-4"], ["--detections", "poses", "--gn-iters", "3"],
                                 ["--detections", "corners", "--p-drop", "1.5"], ["--detections", "corners", "--p-outlier", "-0.1"],
                                 ["--detections", "corners", "--corner-noise", "-1"], ["--detections", "corners", "--gn-iters", "51"],
                                 ["--detections", "edges"]])
def test_sweep_corner_argument_errors(bad):
    with pytest.raises(SystemExit):
        _args(bad)


def test_sweep_corner_memory_and_chunks():
    base = sweep.bytes_per_filter(1000, 125)
    assert sweep.bytes_per_filter(1000, 125, 1, 0) == base
    per = sweep.bytes_per_filter(1000, 125, 8, 25)
    assert per == base + 125 * 7 * 60 + 25 * 8 * 68
    assert sweep.plan_batches(30, 4096, per, 30 * 4096 * per * 2) == [(0, 30)]
    plan = sweep.plan_batches(30, 4096, per, int(10.5 * 4096 * per / 0.8))
    assert plan == [(0, 10), (10, 10), (20, 10)]
    assert sweep.corner_chunks(125, 5.0, 1.0) == [(0, 25), (25, 50), (50, 75), (75, 100), (100, 125)]
    assert sweep.corner_chunks(50, 2.0, 5.0) == [(0, 50)]
    assert sweep.corner_chunks(10, 1.0, 0.3) == [(0, 3), (3, 6), (6, 9), (9, 10)]

