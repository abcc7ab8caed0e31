"""Noise-tuning sweep: many settings of the six noise covariances in ONE batch, scored by their NEES consistency.

    python -m fbus_ekf_b200.sweep --set pos_n_cov=1e-7,1e-6,1e-5 --set quat_n_cov=1e-6,1e-5,1e-4 \\
           --runs 4096 --duration 5 --eval-every 1 [--seed S] [--device D] [--out rows.jsonl]

The grid is the Cartesian product of the --set lists (the last list varies fastest); parameters not named keep
fbus_config_default's value.  Every setting gets --runs Monte-Carlo runs of the synthetic workload (synth.truth_trajectory,
per-filter noisy streams from fbus_synth_streams with synth.DEFAULT_NOISE).  The batch is setting-major: filter b belongs to
setting b // runs and runs with that setting's values (fbus_set_noise).  A batch holds at most 1,048,576 filters and no more than
the device-resident streams leave room for; larger grids run as several batches, one after another.  The streams are stepped in
chunks of --eval-every seconds; after each chunk fbus_filter_errors scores every filter against the truth of the chunk's last
frame and torch reduces the rows per setting on the device.

One JSON row per setting: the six values, rmse_pos_m / rmse_att_rad at the last evaluation, t_eval and nees6_mean (mean NEES over
(p, theta), 6 dof, at each evaluation; about 6 for a consistent filter), frac_nees6_le_12.59 (share of the runs whose last NEES is
within the chi-square(6) 95 % quantile: about 0.95 when consistent; non-finite runs count as outside) and n_nonfinite.

Corner-level detections (--detections corners): the marker detections are no longer the iid-Gaussian poses of
fbus_synth_streams but what the front end makes of noisy corners.  Every map marker is projected from the truth trajectory
(synth.base_marker_poses, fbus_synth_corners: white noise --corner-noise on every normalised coordinate, a detection missing
with probability --p-drop, an outlier with probability --p-outlier and extra std --sigma-outlier), solved back to poses by
fbus_solve_to_detections (refractive solve plus --gn-iters Gauss-Newton iterations, default 5) and fused by the filter: the
nearest marker, or with --all-markers every known one (FBUS_FLAG_ALL_MARKERS).  --board uses the 4 x 2 marker board of
BASELINE configs[3] (synth.board_config) seen from 1 m.  The IMU streams still come from fbus_synth_streams.  The corners are
generated one evaluation chunk at a time, so only the chunk's corners are resident.  These rows also carry detections,
corner_noise, p_drop, p_outlier, sigma_outlier, gn_iters, all_markers, board and n_markers.

Innovation gate (--set gate_chi2=v1,v2,...): one more grid dimension, the NIS threshold of fbus_set_gate (<= 0: no gate).  Every
filter gets its setting's threshold (same setting-major layout as the noise values), in both detection modes.  Only with
gate_chi2 in --set do the rows carry gate_chi2 and rejected_per_run (mean count of rejected updates per run at the end).

Validated range: pos_n_cov and quat_n_cov >= 1e-8.  There every kernel form's (position, attitude) covariance block, and so the
NEES, is within 1e-9 relative of a 50-digit evaluation (DESIGN.md, "Numerical envelope of the update").  Smaller measurement noise
runs, but the double-precision update loses digits to cancellation: at 1e-12 the NEES is good to about 1e-7.
"""
from __future__ import annotations

import argparse
import itertools
import json
import math
import sys

import numpy as np

from . import capi

CHI2_6_95 = 12.591587243743977  # 95 % quantile of the chi-square distribution with 6 degrees of freedom
MAX_BATCH = 1 << 20
FRAC_KEY = "frac_nees6_le_12.59"
GATE_KEY = "gate_chi2"  # the innovation gate's threshold, a grid dimension beside the noise values
SET_NAMES = capi.NOISE_FIELDS + (GATE_KEY,)


def parse_sets(items) -> list[tuple[str, list[float]]]:
    """["name=v1,v2", ...] -> [(name, [v1, v2]), ...] in the given order; unknown or repeated names are errors"""
    out, seen = [], set()
    for it in items or ():
        name, sep, vals = it.partition("=")
        name = name.strip()
        if not sep or not vals.strip():
            raise ValueError(f"--set {it!r}: expected name=v1,v2,...")
        if name not in SET_NAMES:
            raise ValueError(f"--set {it!r}: unknown parameter {name!r} (one of {', '.join(SET_NAMES)})")
        if name in seen:
            raise ValueError(f"--set {it!r}: {name} given twice")
        seen.add(name)
        out.append((name, [float(v) for v in vals.split(",")]))
    return out


def expand_grid(sets, base: dict) -> list[dict]:
    """Cartesian product of the --set lists over the base values (dict of all six NOISE_FIELDS); the last list varies fastest.
    A setting has gate_chi2 only when it is in `sets`."""
    names = [n for n, _ in sets]
    grid = []
    for combo in itertools.product(*[v for _, v in sets]):
        s = {n: float(base[n]) for n in capi.NOISE_FIELDS}
        s.update(zip(names, combo))
        grid.append(s)
    return grid


def setting_of(b, runs: int):
    """setting of filter b (setting-major layout): b // runs"""
    return b // runs


def noise_array(settings: list[dict], runs: int) -> np.ndarray:
    """[6][len(settings) * runs] fbus_set_noise array, setting-major"""
    col = np.array([[s[n] for n in capi.NOISE_FIELDS] for s in settings], dtype=np.float64).T  # [6][S]
    return np.ascontiguousarray(np.repeat(col, runs, axis=1))


def gate_array(settings: list[dict], runs: int) -> np.ndarray | None:
    """[len(settings) * runs] fbus_set_gate array, setting-major; None when the settings have no gate_chi2"""
    if GATE_KEY not in settings[0]:
        return None
    return np.ascontiguousarray(np.repeat(np.array([s[GATE_KEY] for s in settings], dtype=np.float64), runs))


def _rejected_per_run(f, n_set: int, runs: int) -> np.ndarray:
    """mean count of rejected updates per run, per setting"""
    return f.RejectedUpdates().reshape(n_set, runs).mean(axis=1)


def bytes_per_filter(n_samples: int, n_frames: int, n_markers: int = 1, chunk_frames: int = 0) -> int:
    """device bytes one filter of the sweep needs: its streams (IMU [N][6], marker id and pose per frame and slot), the
    corner-mode chunk buffer (16 float32 coordinates and an id per slot of chunk_frames frames), the handle's state (nominal 37 +
    packed covariance 171 doubles, 5 ints), the noise column, the error rows and the truth columns of one evaluation (run_sweep
    builds them per evaluation)"""
    return (n_samples * 6 * 8 + n_frames * n_markers * (4 + 7 * 8) + chunk_frames * n_markers * (16 * 4 + 4) + (37 + 171) * 8 +
            5 * 4 + 6 * 8 + 4 * 8 + 7 * 8)


def plan_batches(n_settings: int, runs: int, per_filter: int, free_bytes: int, max_filters: int = MAX_BATCH,
                 headroom: float = 0.8) -> list[tuple[int, int]]:
    """[(first setting, number of settings), ...]: whole settings per batch, at most max_filters filters and at most `headroom`
    of the free device memory each"""
    if runs <= 0 or n_settings <= 0:
        raise ValueError("need at least one setting and one run")
    fit = min(max_filters, int(free_bytes * headroom) // max(per_filter, 1))
    per_batch = fit // runs
    if per_batch < 1:
        raise ValueError(f"{runs} runs of one setting do not fit one batch (at most {fit} filters)")
    return [(s, min(per_batch, n_settings - s)) for s in range(0, n_settings, per_batch)]


def _reduce(err, n_set: int, runs: int):
    """per-setting reductions of one fbus_filter_errors result (torch [4][B] on the device)"""
    import torch
    e = err.view(4, n_set, runs)
    ok = e[3] == 1.0
    n_ok = ok.sum(1)
    zero = torch.zeros((), dtype=e.dtype, device=e.device)
    sums = torch.stack([torch.where(ok, e[i], zero).sum(1) for i in range(3)])  # [3][S]
    den = n_ok.clamp(min=1).to(e.dtype)
    nan = torch.full_like(den, float("nan"))
    mean = torch.where(n_ok > 0, sums / den, nan)
    inside = (ok & (e[2] <= CHI2_6_95)).sum(1).to(e.dtype) / runs
    return torch.stack([mean[0], mean[1], mean[2], inside, (runs - n_ok).to(e.dtype)])  # [5][S]


def run_sweep(sets, runs: int, duration: float, eval_every: float = 1.0, seed: int = 1, device: int = 0, data_noise: dict | None = None,
              cfg: capi.FbusConfig | None = None, max_filters: int = MAX_BATCH, log=None, corners: dict | None = None) -> list[dict]:
    """Runs the grid of `sets` ([(name, values), ...], see parse_sets) and returns one row per setting (see the module text).
    data_noise overrides synth.DEFAULT_NOISE for the generated streams (make_synth_spec keywords).  corners (a dict of
    corner_options) switches to corner-level detections."""
    if corners is not None:
        return _run_sweep_corners(sets, runs, duration, eval_every, seed, device, data_noise, cfg, max_filters, log, **corners)
    import torch
    from . import synth
    from .filter import BatchFilter
    cfg = cfg if cfg is not None else capi.config_default()
    base = {n: getattr(cfg, n) for n in capi.NOISE_FIELDS}
    grid = expand_grid(sets, base)
    traj = synth.truth_trajectory(cfg, duration)
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    chunk = max(1, int(round(eval_every * W / duration)))  # frames per evaluation
    ends = list(range(chunk, W, chunk)) + [W]
    dev = torch.device("cuda", device)
    free, _ = torch.cuda.mem_get_info(dev)
    rows = []
    for s0, ns in plan_batches(len(grid), runs, bytes_per_filter(N, W), free, max_filters):
        B = ns * runs
        if log:
            log(f"settings {s0}..{s0 + ns - 1} of {len(grid)}: {B} filters")
        f = BatchFilter(cfg, batch=B, device=device)
        imu_d = torch.empty((N, 6, B), dtype=torch.float64, device=dev)
        id_d = torch.empty((W, 1, B), dtype=torch.int32, device=dev)
        pose_d = torch.empty((W, 1, 7, B), dtype=torch.float64, device=dev)
        f.SynthStreams(synth.make_synth_spec(traj, seed=seed, filter_offset=s0 * runs, **(data_noise or {})), imu_d.data_ptr(),
                       id_d.data_ptr(), pose_d.data_ptr())
        f.SetNoise(noise_array(grid[s0:s0 + ns], runs))
        gate = gate_array(grid[s0:s0 + ns], runs)
        if gate is not None:
            f.SetGate(gate)
        imu = capi.make_imu_stream(traj["t_imu"], imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE)
        det = capi.make_det_frames(traj["t_frames"], id_d.data_ptr(), pose_d.data_ptr(), B, 1, capi.FBUS_MEM_DEVICE)
        err = torch.empty((4, B), dtype=torch.float64, device=dev)
        reds = []
        w0 = 0
        with torch.cuda.device(dev):
            torch_stream = torch.cuda.current_stream(dev)
            for w1 in ends:
                f.StepWindows(imu, det, traj["win_off"], w0, w1)  # device streams: the next chunk continues this one exactly
                tp = torch.from_numpy(traj["truth_p"][w1 - 1]).to(dev)[:, None].expand(3, B).contiguous()
                tq = torch.from_numpy(traj["truth_q"][w1 - 1]).to(dev)[:, None].expand(4, B).contiguous()
                # the handle's stream is not ordered with torch's: the truth columns must be written, and the previous
                # evaluation's reduction must have read `err`, before fbus_filter_errors writes it again
                torch_stream.synchronize()
                f.FilterErrors(tp.data_ptr(), tq.data_ptr(), capi.FBUS_MEM_DEVICE, err.data_ptr(), capi.FBUS_MEM_DEVICE)
                f.Synchronize()  # the rows are complete before torch's stream reduces them
                reds.append(_reduce(err, ns, runs))
                w0 = w1
            red = torch.stack(reds).cpu().numpy()  # [eval][5][S]
        rej = _rejected_per_run(f, ns, runs) if gate is not None else None
        f.close()
        del imu_d, id_d, pose_d, err
        rows += _rows(grid[s0:s0 + ns], runs, red, [float(traj["t_frames"][w - 1]) for w in ends], rej)
    return rows


def _rows(settings, runs: int, red, t_eval, rejected=None) -> list[dict]:
    """one JSON row per setting from the per-evaluation reductions red [eval][5][S] of _reduce (and, with a gate, the mean
    rejection counts per run [S])"""
    rows = []
    for j, setting in enumerate(settings):
        row = dict(setting)
        row["runs"] = runs
        row["rmse_pos_m"] = math.sqrt(red[-1, 0, j])
        row["rmse_att_rad"] = math.sqrt(red[-1, 1, j])
        row["t_eval"] = t_eval
        row["nees6_mean"] = [float(v) for v in red[:, 2, j]]
        row[FRAC_KEY] = float(red[-1, 3, j])
        row["n_nonfinite"] = int(red[-1, 4, j])
        if rejected is not None:
            row["rejected_per_run"] = float(rejected[j])
        rows.append(row)
    return rows


def corner_options(board: bool = False, corner_noise: float | None = None, p_drop: float = 0.0, p_outlier: float = 0.0,
                   sigma_outlier: float = 0.0, gn_iters: int = 5, all_markers: bool = False) -> dict:
    """validated options of the corner-level detections (the `corners` argument of run_sweep)"""
    from . import synth
    corner_noise = synth.DEFAULT_CORNER_NOISE if corner_noise is None else float(corner_noise)
    if corner_noise < 0 or sigma_outlier < 0:
        raise ValueError("--corner-noise and --sigma-outlier must be >= 0")
    for name, p in (("--p-drop", p_drop), ("--p-outlier", p_outlier)):
        if not 0.0 <= p <= 1.0:
            raise ValueError(f"{name} must be within [0, 1]")
    if not 0 <= gn_iters <= 50:
        raise ValueError("--gn-iters must be within [0, 50]")
    return dict(board=bool(board), corner_noise=corner_noise, p_drop=float(p_drop), p_outlier=float(p_outlier),
                sigma_outlier=float(sigma_outlier), gn_iters=int(gn_iters), all_markers=bool(all_markers))


def corner_chunks(n_frames: int, duration: float, eval_every: float) -> list[tuple[int, int]]:
    """the evaluation chunks [w0, w1) of the sweep (the same frames run_sweep evaluates after in both modes)"""
    chunk = max(1, int(round(eval_every * n_frames / duration)))
    ends = list(range(chunk, n_frames, chunk)) + [n_frames]
    return list(zip([0] + ends[:-1], ends))


def _run_sweep_corners(sets, runs, duration, eval_every, seed, device, data_noise, cfg, max_filters, log, board, corner_noise, p_drop,
                       p_outlier, sigma_outlier, gn_iters, all_markers) -> list[dict]:
    import copy
    import torch
    from . import synth
    from .filter import BatchFilter
    cfg = cfg if cfg is not None else capi.config_default()
    base = {n: getattr(cfg, n) for n in capi.NOISE_FIELDS}
    grid = expand_grid(sets, base)
    if board:
        cfg = synth.board_config(cfg)
    if all_markers:
        cfg = copy.copy(cfg)
        cfg.flags |= capi.FBUS_FLAG_ALL_MARKERS
    traj = synth.truth_trajectory(cfg, duration, standoff=1.0) if board else synth.truth_trajectory(cfg, duration)
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    mpose, mids = synth.base_marker_poses(cfg, traj)
    m = mpose.shape[1]
    chunks = corner_chunks(W, duration, eval_every)
    cmax = max(b - a for a, b in chunks)
    dev = torch.device("cuda", device)
    free, _ = torch.cuda.mem_get_info(dev)
    rows = []
    for s0, ns in plan_batches(len(grid), runs, bytes_per_filter(N, W, m, cmax), free, max_filters):
        B = ns * runs
        if log:
            log(f"settings {s0}..{s0 + ns - 1} of {len(grid)}: {B} filters, {m} markers")
        f = BatchFilter(cfg, batch=B, device=device)
        imu_d = torch.empty((N, 6, B), dtype=torch.float64, device=dev)
        tmp_id = torch.empty((W, 1, B), dtype=torch.int32, device=dev)  # the single-marker poses of fbus_synth_streams: unused
        tmp_pose = torch.empty((W, 1, 7, B), dtype=torch.float64, device=dev)
        f.SynthStreams(synth.make_synth_spec(traj, seed=seed, filter_offset=s0 * runs, **(data_noise or {})), imu_d.data_ptr(),
                       tmp_id.data_ptr(), tmp_pose.data_ptr())
        f.Synchronize()
        del tmp_id, tmp_pose
        torch.cuda.empty_cache()
        spec = synth.make_corner_spec(mpose, mids, seed=seed, filter_offset=s0 * runs, underwater=True, sigma_corner=corner_noise,
                                      p_drop=p_drop, p_outlier=p_outlier, sigma_outlier=sigma_outlier)
        id_d = torch.empty((W, m, B), dtype=torch.int32, device=dev)
        pose_d = torch.empty((W, m, 7, B), dtype=torch.float64, device=dev)
        c_d = torch.empty((16, cmax * m * B), dtype=torch.float32, device=dev)
        cid_d = torch.empty((cmax, m, B), dtype=torch.int32, device=dev)
        f.SetNoise(noise_array(grid[s0:s0 + ns], runs))
        gate = gate_array(grid[s0:s0 + ns], runs)
        if gate is not None:
            f.SetGate(gate)
        imu = capi.make_imu_stream(traj["t_imu"], imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE)
        det = capi.make_det_frames(traj["t_frames"], id_d.data_ptr(), pose_d.data_ptr(), B, m, capi.FBUS_MEM_DEVICE)
        err = torch.empty((4, B), dtype=torch.float64, device=dev)
        reds = []
        with torch.cuda.device(dev):
            torch_stream = torch.cuda.current_stream(dev)
            for w0, w1 in chunks:
                # this chunk's corners -> its frames of the full-length detection buffers (frame-major: a pointer offset)
                f.SynthCorners(spec, w0, w1, c_d.data_ptr(), cid_d.data_ptr())
                f.SolveToDetections(c_d.data_ptr(), cid_d.data_ptr(), w1 - w0, m, True, gn_iters,
                                    id_d.data_ptr() + w0 * m * B * 4, pose_d.data_ptr() + w0 * m * 7 * B * 8, capi.FBUS_MEM_DEVICE)
                f.StepWindows(imu, det, traj["win_off"], w0, w1)  # device streams: the next chunk continues this one exactly
                tp = torch.from_numpy(traj["truth_p"][w1 - 1]).to(dev)[:, None].expand(3, B).contiguous()
                tq = torch.from_numpy(traj["truth_q"][w1 - 1]).to(dev)[:, None].expand(4, B).contiguous()
                torch_stream.synchronize()  # as in run_sweep: truth written, previous reduction done with `err`
                f.FilterErrors(tp.data_ptr(), tq.data_ptr(), capi.FBUS_MEM_DEVICE, err.data_ptr(), capi.FBUS_MEM_DEVICE)
                f.Synchronize()
                reds.append(_reduce(err, ns, runs))
            red = torch.stack(reds).cpu().numpy()  # [eval][5][S]
        rej = _rejected_per_run(f, ns, runs) if gate is not None else None
        f.close()
        del imu_d, id_d, pose_d, c_d, cid_d, err
        for row in _rows(grid[s0:s0 + ns], runs, red, [float(traj["t_frames"][w1 - 1]) for _, w1 in chunks], rej):
            row.update(detections="corners", corner_noise=corner_noise, p_drop=p_drop, p_outlier=p_outlier, sigma_outlier=sigma_outlier,
                       gn_iters=gn_iters, all_markers=all_markers, board=board, n_markers=m)
            rows.append(row)
    return rows


def parse_corner_args(a) -> dict | None:
    """the corner options of parsed arguments (None in pose mode, where giving one is an error)"""
    given = {k: getattr(a, k) for k in ("corner_noise", "p_drop", "p_outlier", "sigma_outlier", "gn_iters")
             if getattr(a, k) is not None}
    if a.detections != "corners":
        if given or a.board or a.all_markers:
            raise ValueError("--board, --corner-noise, --p-drop, --p-outlier, --sigma-outlier, --gn-iters and --all-markers "
                             "need --detections corners")
        return None
    return corner_options(board=a.board, all_markers=a.all_markers, **given)


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="python -m fbus_ekf_b200.sweep", description=__doc__.split("\n\n")[0],
                                 formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--set", action="append", default=[], metavar="NAME=V1,V2,...",
                    help=f"values of one noise parameter ({', '.join(capi.NOISE_FIELDS)}) or of the innovation gate's NIS threshold "
                         f"({GATE_KEY}, <= 0: no gate); repeat for a grid")
    ap.add_argument("--runs", type=int, default=4096, help="Monte-Carlo runs per setting (default 4096)")
    ap.add_argument("--duration", type=float, default=5.0, help="seconds of synthetic stream (default 5)")
    ap.add_argument("--eval-every", type=float, default=1.0, help="seconds between evaluations (default 1)")
    ap.add_argument("--seed", type=int, default=1, help="seed of the Monte-Carlo streams (default 1)")
    ap.add_argument("--device", type=int, default=0, help="CUDA device (default 0)")
    ap.add_argument("--out", default=None, help="write the JSON rows here instead of stdout")
    ap.add_argument("--detections", choices=("poses", "corners"), default="poses",
                    help="poses: iid-Gaussian marker poses of fbus_synth_streams (default); corners: noisy stereo corners of every "
                         "map marker solved to poses on the device")
    cg = ap.add_argument_group("corner-level detections (--detections corners only)")
    cg.add_argument("--board", action="store_true", help="the 4 x 2 marker board of BASELINE configs[3], seen from 1 m")
    cg.add_argument("--corner-noise", type=float, default=None, help="std of the white noise on every normalised corner coordinate "
                                                                     "(default synth.DEFAULT_CORNER_NOISE = 2e-4)")
    cg.add_argument("--p-drop", type=float, default=None, help="probability that a detection is missing (default 0)")
    cg.add_argument("--p-outlier", type=float, default=None, help="probability of a gross error on a detection (default 0)")
    cg.add_argument("--sigma-outlier", type=float, default=None, help="extra std of an outlier's coordinates (default 0)")
    cg.add_argument("--gn-iters", type=int, default=None, help="Gauss-Newton iterations of the marker solve (default 5)")
    cg.add_argument("--all-markers", action="store_true", help="fuse every known marker of a frame (FBUS_FLAG_ALL_MARKERS)")
    a = ap.parse_args(argv)
    try:
        sets = parse_sets(a.set)
        corners = parse_corner_args(a)
    except ValueError as e:
        ap.error(str(e))
    rows = run_sweep(sets, a.runs, a.duration, a.eval_every, a.seed, a.device, log=lambda m: print(m, file=sys.stderr),
                     corners=corners)
    text = "".join(json.dumps(r) + "\n" for r in rows)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text)
    else:
        sys.stdout.write(text)
    return 0


if __name__ == "__main__":
    sys.exit(main())
