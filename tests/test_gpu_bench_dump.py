"""bench.py --dump-outputs: the files hold the state that the timed steps left in the sampled filters -- the same batch
stepped directly through BatchFilter over the same seeded streams gives the same columns bit for bit -- and --steps is the
number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_state_after_the_timed_steps(cfg, tmp_path):
    import torch
    from fbus_ekf_b200 import BatchFilter, capi, synth
    B, n_dump, K, Wm = 96, 40, 2, 3
    out_dir = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(K), "--warmup", str(Wm),
                          "--no-solves", "--no-e2e", "--no-cpu", "--dump-outputs", str(out_dir)],
                         env=dict(os.environ, FBUS_BENCH_BATCH=str(B), FBUS_BENCH_DUMP_FILTERS=str(n_dump)),
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == K and line["gpu_launches"] == K and line["warmup"] == Wm

    dumped = {p[:-4]: np.load(out_dir / p) for p in os.listdir(out_dir)}
    assert all(a.dtype == np.float64 for a in dumped.values())
    idx = dumped.pop("filter_index")
    assert idx.shape == (n_dump,) and np.array_equal(idx, np.unique(idx)) and idx[0] >= 0 and idx[-1] < B
    idx = idx.astype(np.int64)
    stats = dumped.pop("stats")
    assert stats.shape == (capi.FBUS_NSTATS,) and stats[3] == B

    # bench.py's workload: periodic 1 s trajectory, streams from seed 20260117 + 5, step k shifted by k seconds
    traj = synth.truth_trajectory(cfg, 1.0, 200.0, 25.0, periodic=True)
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    f = BatchFilter(cfg, batch=B, device=0)
    imu_d = torch.empty((N, 6, B), dtype=torch.float64, device="cuda:0")
    id_d = torch.empty((W, 1, B), dtype=torch.int32, device="cuda:0")
    pose_d = torch.empty((W, 1, 7, B), dtype=torch.float64, device="cuda:0")
    f.SynthStreams(synth.make_synth_spec(traj, seed=20260117 + 5), imu_d.data_ptr(), id_d.data_ptr(), pose_d.data_ptr())
    for k in range(Wm + K):
        f.StepWindows(capi.make_imu_stream(traj["t_imu"] + k, imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE),
                      capi.make_det_frames(traj["t_frames"] + k, id_d.data_ptr(), pose_d.data_ptr(), B, 1, capi.FBUS_MEM_DEVICE),
                      traj["win_off"], 0, W)
    st = f.GetState()
    f.close()
    assert sorted(dumped) == sorted(st)
    for name, a in st.items():
        assert np.array_equal(dumped[name], a[..., idx].astype(np.float64)), name
