"""Cost of FBUS_FLAG_ALL_MARKERS on BASELINE configs[3]'s shape: 65,536 filters, the 8-marker board, 1 s of 200 Hz IMU + 25 Hz
frames, device-resident detections (refractive solve + Gauss-Newton of 256 distinct runs, tiled over the batch).  The same frames
are stepped three ways, each on its own handle and timed with CUDA events on that handle's stream:

  (a) default  -- the nearest marker only, on the kernel the library picks for this batch
  (b) lane1    -- the nearest marker only, forced onto the first-generation lanes-per-filter kernel (FBUS_LANE=1 FBUS_LANE_GEN=1)
  (c) all      -- FBUS_FLAG_ALL_MARKERS (always that kernel)

Reported: ms per second of stream, and filter-steps/s with every applied marker update counted as one step (SURVEY 8d: IMU samples
+ updates per filter).  The three are timed alternately after a warm-up; the median of --reps is printed.  One JSON line with the
GPU's name and power limit.

    python profiles/probes/all_markers_rate.py [--batch 65536] [--reps 5] [--warmup 2]
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    sys.stdout.flush()
    out_fd = os.dup(1)
    os.dup2(2, 1)  # the build's own output goes to stderr: stdout carries the JSON line only
    try:
        ge.build()
    finally:
        sys.stdout.flush()
        os.dup2(out_fd, 1)
    from fbus_ekf_b200 import BatchFilter, capi, synth
    assert torch.cuda.is_available(), "this probe measures the GPU; there is no CPU fallback"
    B, m, R = a.batch, 8, min(a.batch, 256)
    cfg = capi.config_default()
    bcfg = synth.board_config(cfg)
    traj = synth.truth_trajectory(bcfg, 1.0, standoff=1.0)
    W, N = len(traj["t_frames"]), len(traj["t_imu"])
    base, ids, _ = synth.board_base_corners(bcfg, traj)
    rng = np.random.default_rng(31)
    corners = np.ascontiguousarray((np.repeat(base, R, axis=1) + rng.normal(size=(16, W * m * R)) * 2e-4).astype(np.float32))
    mids = np.ascontiguousarray(np.repeat(ids[:, :, None], R, axis=2))
    det_id, det_pose = BatchFilter(bcfg, batch=R).SolveToDetections(corners, mids, W, m, underwater=True, gn_iters=4)
    imu = traj["base_imu"][:, :, None] + rng.normal(size=(N, 6, R)) * np.array([0.015] * 3 + [1e-3] * 3)[None, :, None]
    reps = (B + R - 1) // R
    dev = torch.device("cuda:0")
    til = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev).repeat(*([1] * (x.ndim - 1) + [reps]))[..., :B].contiguous()
    imu_d, id_d, pose_d = til(imu), til(det_id), til(det_pose)
    s = capi.make_imu_stream(traj["t_imu"], imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE)
    d = capi.make_det_frames(traj["t_frames"], id_d.data_ptr(), pose_d.data_ptr(), B, m, capi.FBUS_MEM_DEVICE)
    # applied updates per filter: frames after the initialising one, times the known markers of each frame
    known = (id_d >= 0).sum(dim=1).double()              # [W][B]
    n_upd_all = float(known[1:].sum() / B)
    n_upd_one = float((known[1:] > 0).sum() / B)
    n_imu = float(N)

    def make(flags, env):
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            c = copy.copy(bcfg)
            c.flags = flags
            return BatchFilter(c, batch=B)
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v

    modes = {"default": make(0, {}), "lane1": make(0, {"FBUS_LANE": "1", "FBUS_LANE_GEN": "1"}),
             "all": make(capi.FBUS_FLAG_ALL_MARKERS, {})}
    init = BatchFilter(bcfg, batch=B)  # every timed pass starts from the same state (after the initialising frame)
    init.StepWindows(s, d, traj["win_off"], 0, 1)
    st0 = init.GetState()

    def timed(f):
        f.SetState(st0)
        f.ClearStatus()
        st = torch.cuda.ExternalStream(f.stream, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        f.StepWindows(s, d, traj["win_off"], 1, W)
        e1.record(st)
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e-3

    for _ in range(a.warmup):
        for f in modes.values():
            timed(f)
    times = {k: [] for k in modes}
    for _ in range(a.reps):
        for k, f in modes.items():
            times[k].append(timed(f))
    secs = (traj["t_frames"][-1] - traj["t_frames"][0])
    out = {"probe": "all_markers_rate", "gpu": gpu_info(), "batch": B, "markers": m, "frames": W - 1, "imu_samples": N,
           "stream_seconds": float(secs), "updates_per_filter": {"nearest": n_upd_one, "all": n_upd_all}}
    for k, ts in times.items():
        t = float(np.median(ts))
        n_steps = n_imu + (n_upd_all if k == "all" else n_upd_one)
        out[k] = {"ms_per_stream_second": t / secs * 1e3, "filter_steps_per_s": B * n_steps / t, "seconds": ts}
    # the nearest-marker result is the same on both kernels (a sanity check of the comparison, not of the flag)
    a_st, b_st = modes["default"].GetState(), modes["lane1"].GetState()
    out["default_vs_lane1_max_p_diff"] = float(np.abs(a_st["p"] - b_st["p"]).max())
    out["all_slower_than_default"] = out["all"]["ms_per_stream_second"] / out["default"]["ms_per_stream_second"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
