"""Cost of the corner-level Monte-Carlo workload at BASELINE configs[3]'s shape: 65,536 filters x the 8-marker board x 25
frames (1 s of stream).  Timed with CUDA events on the handle's stream, median of --reps after --warmup passes:

  synth_corners      fbus_synth_corners for all 25 frames (the call: staging of the 200 base poses, their projection, and the
                     per-filter kernel writing 16 float32 corners + 1 id = 68 B per item)
  solve_gn0 / gn5    fbus_solve_to_detections of those corners with 0 and 5 Gauss-Newton iterations
  marker_project     fbus_marker_project of 524,288 random marker poses (device memory), underwater

One JSON object with the GPU's name and power limit, written to --out (and printed).

    python profiles/probes/corner_synth_rate.py [--batch 65536] [--reps 7] [--warmup 2] [--out profiles/corner_synth_rate.json]
"""
from __future__ import annotations

import argparse
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
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--n-project", type=int, default=524288)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "corner_synth_rate.json"))
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
    B = a.batch
    bcfg = synth.board_config(capi.config_default())
    traj = synth.truth_trajectory(bcfg, 1.0, standoff=1.0)
    pose, ids = synth.base_marker_poses(bcfg, traj)
    W, m = pose.shape[:2]
    n = W * m * B
    spec = synth.make_corner_spec(pose, ids, seed=11, sigma_corner=synth.DEFAULT_CORNER_NOISE)
    f = BatchFilter(bcfg, batch=B)
    dev = torch.device("cuda:0")
    st = torch.cuda.ExternalStream(f.stream, device=dev)
    corners = torch.empty((16, n), dtype=torch.float32, device=dev)
    cid = torch.empty((W, m, B), dtype=torch.int32, device=dev)
    det_id = torch.empty((W, m, B), dtype=torch.int32, device=dev)
    det_pose = torch.empty((W, m, 7, B), dtype=torch.float64, device=dev)
    rng = np.random.default_rng(3)
    Rm, p = synth.random_marker_poses(a.n_project, rng, 0.3)
    qs = np.stack([synth.quat_from_rotmat(R) for R in Rm], axis=1)
    pp = torch.from_numpy(np.ascontiguousarray(np.concatenate([p.T, qs]))).to(dev)
    pc = torch.empty((16, a.n_project), dtype=torch.float64, device=dev)
    pv = torch.empty(a.n_project, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        fn()
        e1.record(st)
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e-3

    work = {
        "synth_corners": lambda: f.SynthCorners(spec, 0, W, corners.data_ptr(), cid.data_ptr()),
        "solve_gn0": lambda: f.SolveToDetections(corners.data_ptr(), cid.data_ptr(), W, m, True, 0, det_id.data_ptr(),
                                                 det_pose.data_ptr(), capi.FBUS_MEM_DEVICE),
        "solve_gn5": lambda: f.SolveToDetections(corners.data_ptr(), cid.data_ptr(), W, m, True, 5, det_id.data_ptr(),
                                                 det_pose.data_ptr(), capi.FBUS_MEM_DEVICE),
        "marker_project": lambda: f.MarkerProject(pp.data_ptr(), True, n=a.n_project, corners=pc.data_ptr(), valid=pv.data_ptr(),
                                                  mem=capi.FBUS_MEM_DEVICE),
    }
    for _ in range(a.warmup):
        for fn in work.values():
            timed(fn)
    times = {k: [] for k in work}
    for _ in range(a.reps):  # alternated, so that a slow moment of the shared host touches every entry alike
        for k, fn in work.items():
            times[k].append(timed(fn))
    med = {k: float(np.median(v)) for k, v in times.items()}
    f.Synchronize()
    dropped = int((cid < 0).sum())
    out = {"probe": "corner_synth_rate", "gpu": gpu_info(), "batch": B, "markers": m, "frames": W, "items": n,
           "synth_corners": {"ms": med["synth_corners"] * 1e3, "items_per_s": n / med["synth_corners"],
                             "written_bytes_per_item": 16 * 4 + 4, "write_GB_per_s": n * 68 / med["synth_corners"] / 1e9,
                             "seconds": times["synth_corners"]},
           "solve_gn0": {"ms": med["solve_gn0"] * 1e3, "solves_per_s": n / med["solve_gn0"], "seconds": times["solve_gn0"]},
           "solve_gn5": {"ms": med["solve_gn5"] * 1e3, "solves_per_s": n / med["solve_gn5"], "seconds": times["solve_gn5"]},
           "marker_project": {"markers": a.n_project, "ms": med["marker_project"] * 1e3,
                              "projections_per_s": a.n_project / med["marker_project"], "seconds": times["marker_project"]},
           "synth_over_solve_gn5": med["synth_corners"] / med["solve_gn5"],
           "synth_over_solve_gn0": med["synth_corners"] / med["solve_gn0"],
           "empty_slots": dropped}
    text = json.dumps(out)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")
    print(text)
    f.close()


if __name__ == "__main__":
    main()
