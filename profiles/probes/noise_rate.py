"""Cost of per-filter noise values (fbus_set_noise) on the bench's workload shape: 1 s of 200 Hz IMU + 25 Hz marker poses per
launch, device-resident streams, periodic trajectory replayed with shifted time stamps (as bench.py does).

  (a) 1,048,576 filters on the default path
  (b) the same batch with fbus_set_noise set to the config's values: must give the same state, bit for bit (checked here)
  (c) a 256-setting x 4,096-run grid as ONE handle (per-filter values), against 256 handles of 4,096 filters (one setting each)
      run one after another.  Both sides are timed with CUDA events on the handles' streams: c_many_handles is the sum over the
      256 handles of the event time of each handle's launches (the device time of the 256 handles); c_many_handles_wall is the
      host clock around the whole sequence, which adds what the host spends between the handles (launch calls, synchronising)

(a) and (b) are two handles in this process, timed alternately with CUDA events after a warm-up.  Rates are filter-steps/s
(IMU samples + frames per filter per second).  Prints one JSON line with the GPU's name and power limit.

    python profiles/probes/noise_rate.py [--batch 1048576] [--steps 5] [--reps 3] [--warmup 3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

PERIOD, IMU_RATE, FRAME_RATE = 1.0, 200.0, 25.0


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--settings", type=int, default=256)
    ap.add_argument("--runs", type=int, default=4096)
    a = ap.parse_args()

    import torch
    import __graft_entry__ as ge
    sys.stdout.flush()
    out_fd = os.dup(1)
    os.dup2(2, 1)  # the build's own output (nvcc, make) goes to stderr: stdout carries the JSON line only
    try:
        ge.build()
    finally:
        sys.stdout.flush()
        os.dup2(out_fd, 1)
        os.close(out_fd)
    from fbus_ekf_b200 import BatchFilter, capi, synth

    assert torch.cuda.is_available(), "noise_rate.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    cfg = capi.config_default()
    traj = synth.truth_trajectory(cfg, PERIOD, IMU_RATE, FRAME_RATE, periodic=True)
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    spf = N + W  # filter-steps per filter per launch

    def streams(B, seed=20260117 + 5):
        g = BatchFilter(cfg, batch=B)
        imu_d = torch.empty((N, 6, B), dtype=torch.float64, device=dev)
        id_d = torch.empty((W, 1, B), dtype=torch.int32, device=dev)
        pose_d = torch.empty((W, 1, 7, B), dtype=torch.float64, device=dev)
        g.SynthStreams(synth.make_synth_spec(traj, seed=seed), imu_d.data_ptr(), id_d.data_ptr(), pose_d.data_ptr())
        g.close()
        return imu_d, id_d, pose_d

    def stepper(f, B, s):
        imu_d, id_d, pose_d = s

        def step(k):
            ti, tf = traj["t_imu"] + k * PERIOD, traj["t_frames"] + k * PERIOD
            f.StepWindows(capi.make_imu_stream(ti, imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE),
                          capi.make_det_frames(tf, id_d.data_ptr(), pose_d.data_ptr(), B, 1, capi.FBUS_MEM_DEVICE), traj["win_off"], 0, W)
        return step

    def timed(f, step, k0, K):
        st = torch.cuda.ExternalStream(f.stream, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f.Synchronize()
        e0.record(st)
        for k in range(K):
            step(k0 + k)
        e1.record(st)
        f.Synchronize()
        return e0.elapsed_time(e1) * 1e-3

    B = a.batch
    s = streams(B)
    fa = BatchFilter(cfg, batch=B)
    fb = BatchFilter(cfg, batch=B)
    fb.SetNoise(capi.noise_from_config(cfg, B))
    sa, sb = stepper(fa, B, s), stepper(fb, B, s)
    for k in range(a.warmup):
        sa(k)
        sb(k)
    ta, tb = [], []
    k0 = a.warmup
    for r in range(a.reps):  # alternate the two arms
        ta.append(timed(fa, sa, k0, a.steps))
        tb.append(timed(fb, sb, k0, a.steps))
        k0 += a.steps
    rate_a = [B * spf * a.steps / t for t in ta]
    rate_b = [B * spf * a.steps / t for t in tb]
    ga, gb = fa.GetState(), fb.GetState()
    identical = all(np.array_equal(ga[k], gb[k], equal_nan=True) for k in ga)
    fa.close()
    fb.close()
    del ga, gb

    # (c) the grid as one handle vs one handle per setting
    S, R = a.settings, a.runs
    side = int(round(np.sqrt(S)))
    pos = cfg.pos_n_cov * np.logspace(-2, 1, side)
    quat = cfg.quat_n_cov * np.logspace(-2, 1, S // side)
    grid = [(p, q) for p in pos for q in quat][:S]
    Bg = S * R
    noise = capi.noise_from_config(cfg, Bg)
    noise[capi.NOISE_FIELDS.index("pos_n_cov")] = np.repeat([g[0] for g in grid], R)
    noise[capi.NOISE_FIELDS.index("quat_n_cov")] = np.repeat([g[1] for g in grid], R)
    sg = s if Bg == B else streams(Bg)
    fg = BatchFilter(cfg, batch=Bg)
    fg.SetNoise(np.ascontiguousarray(noise))
    stg = stepper(fg, Bg, sg)
    for k in range(a.warmup):
        stg(k)
    tg = timed(fg, stg, a.warmup, a.steps)
    fg.close()
    del sg, s
    torch.cuda.empty_cache()
    ss = streams(R)
    import copy
    handles = []
    for p, q in grid:
        c = copy.copy(cfg)
        c.pos_n_cov, c.quat_n_cov = float(p), float(q)
        handles.append(BatchFilter(c, batch=R))
    steps = [stepper(h, R, ss) for h in handles]
    for h, st in zip(handles, steps):  # warm-up
        for k in range(a.warmup):
            st(k)
        h.Synchronize()
    torch.cuda.synchronize(dev)
    tm = 0.0
    t0 = time.perf_counter()
    for h, st in zip(handles, steps):  # one after another
        tm += timed(h, st, a.warmup, a.steps)
    tm_wall = time.perf_counter() - t0
    for h in handles:
        h.close()
    one = Bg * spf * a.steps / tg
    many = Bg * spf * a.steps / tm
    many_wall = Bg * spf * a.steps / tm_wall
    line = {
        "gpu": gpu_info(), "batch": B, "steps_per_timing": a.steps, "reps": a.reps, "unit": "filter-steps/s",
        "a_default": float(np.median(rate_a)), "a_all": rate_a,
        "b_noise_config_values": float(np.median(rate_b)), "b_all": rate_b,
        "b_over_a": float(np.median(rate_b) / np.median(rate_a)), "b_state_identical_to_a": bool(identical),
        "c_settings": S, "c_runs": R, "c_one_handle": one, "c_many_handles": many, "c_one_over_many": one / many,
        "c_many_handles_wall": many_wall, "c_one_over_many_wall": one / many_wall,
    }
    print(json.dumps(line))
    if not identical:
        raise SystemExit("noise_rate.py: (b) differs from (a)")


if __name__ == "__main__":
    main()
