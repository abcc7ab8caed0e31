"""Cost of the innovation gate (fbus_set_gate) on BASELINE configs[3]'s shape: 65,536 filters, the 8-marker board, 1 s of 200 Hz
IMU + 25 Hz frames (24 frames after the initialising one), device-resident detections (refractive solve + Gauss-Newton of 256
distinct runs, tiled over the batch).  The same frames are stepped four ways, each on its own handle and timed with CUDA events on
that handle's stream:

  (a) default     -- no gate, the kernel the library picks for this batch
  (b) lane1       -- no gate, forced onto the first-generation lanes-per-filter kernel (FBUS_LANE=1 FBUS_LANE_GEN=1)
  (c) gated       -- the gate with a threshold no update fails (every filter's NIS is formed and tested, nothing is rejected)
  (d) gated_all   -- the same under FBUS_FLAG_ALL_MARKERS

(c) and (d) run on the first-generation lanes-per-filter kernel, where the gate lives.  Reported: ms per second of stream and
filter-steps/s (IMU samples + applied updates per filter, as all_markers_rate.py counts them), the median of --reps passes timed
alternately after a warm-up.  One JSON line with the GPU's name and power limit.

    python profiles/probes/gate_rate.py [--batch 65536] [--reps 7] [--warmup 2]
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from all_markers_rate import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=7)
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
    known = (id_d >= 0).sum(dim=1).double()              # [W][B]
    n_upd_all = float(known[1:].sum() / B)
    n_upd_one = float((known[1:] > 0).sum() / B)

    def make(flags, env, gate=None):
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            c = copy.copy(bcfg)
            c.flags = flags
            f = BatchFilter(c, batch=B)
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        if gate is not None:
            f.SetGate(np.full(B, gate))
        return f

    modes = {"default": make(0, {}), "lane1": make(0, {"FBUS_LANE": "1", "FBUS_LANE_GEN": "1"}), "gated": make(0, {}, 1e12),
             "gated_all": make(capi.FBUS_FLAG_ALL_MARKERS, {}, 1e12)}
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
    out = {"probe": "gate_rate", "gpu": gpu_info(), "batch": B, "markers": m, "frames": W - 1, "imu_samples": N,
           "stream_seconds": float(secs), "updates_per_filter": {"nearest": n_upd_one, "all": n_upd_all}, "reps": a.reps}
    for k, ts in times.items():
        t = float(np.median(ts))
        n_steps = N + (n_upd_all if k == "gated_all" else n_upd_one)
        out[k] = {"ms_per_stream_second": t / secs * 1e3, "filter_steps_per_s": B * n_steps / t, "seconds": ts}
    # nothing was rejected, so the gated pass computes what the ungated lane-1 pass computes, bit for bit
    a_st, g_st = modes["lane1"].GetState(), modes["gated"].GetState()
    out["gated_rejected"] = int(modes["gated"].RejectedUpdates().sum() + modes["gated_all"].RejectedUpdates().sum())
    out["gated_equals_lane1"] = bool(all(np.array_equal(a_st[k], g_st[k]) for k in ("p", "q", "v", "P")))
    out["gated_vs_lane1"] = out["gated"]["ms_per_stream_second"] / out["lane1"]["ms_per_stream_second"]
    out["gated_vs_default"] = out["gated"]["ms_per_stream_second"] / out["default"]["ms_per_stream_second"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
