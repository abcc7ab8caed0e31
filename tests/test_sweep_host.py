"""Host-side parts of the noise-tuning sweep (fbus_ekf_b200.sweep): grid, batch layout and split, command line.  No GPU."""
import os
import subprocess
import sys

import numpy as np
import pytest

from fbus_ekf_b200 import capi, sweep

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = dict(zip(capi.NOISE_FIELDS, (1e-3, 1e-4, 1e-3, 1e-4, 1e-3, 1e-3)))


def test_grid_is_the_product_in_order():
    sets = sweep.parse_sets(["pos_n_cov=1e-7,1e-6,1e-5", "quat_n_cov=1e-6,1e-4"])
    assert sets == [("pos_n_cov", [1e-7, 1e-6, 1e-5]), ("quat_n_cov", [1e-6, 1e-4])]
    grid = sweep.expand_grid(sets, BASE)
    assert len(grid) == 6
    assert [(g["pos_n_cov"], g["quat_n_cov"]) for g in grid] == [(1e-7, 1e-6), (1e-7, 1e-4), (1e-6, 1e-6), (1e-6, 1e-4),
                                                                  (1e-5, 1e-6), (1e-5, 1e-4)]
    for g in grid:  # parameters not named keep the base value
        assert list(g) == list(capi.NOISE_FIELDS)
        for n in ("accel_n_cov", "gyro_n_cov", "accel_b_cov", "gyro_b_cov"):
            assert g[n] == BASE[n]
    assert sweep.expand_grid([], BASE) == [BASE]


@pytest.mark.parametrize("bad", ["pos_cov=1e-3", "accel_n_cov", "accel_n_cov=", "Rp=1"])
def test_unknown_or_malformed_names_are_rejected(bad):
    with pytest.raises(ValueError):
        sweep.parse_sets([bad])


def test_repeated_name_is_rejected():
    with pytest.raises(ValueError):
        sweep.parse_sets(["pos_n_cov=1", "pos_n_cov=2"])


def test_setting_major_layout():
    runs = 5
    settings = sweep.expand_grid(sweep.parse_sets(["gyro_b_cov=1,2,3"]), BASE)
    nz = sweep.noise_array(settings, runs)
    assert nz.shape == (6, 15) and nz.dtype == np.float64 and nz.flags["C_CONTIGUOUS"]
    b = np.arange(15)
    assert np.array_equal(sweep.setting_of(b, runs), np.repeat(np.arange(3), runs))
    row = capi.NOISE_FIELDS.index("gyro_b_cov")
    assert np.array_equal(nz[row], np.array([1.0, 2.0, 3.0])[sweep.setting_of(b, runs)])
    assert np.all(nz[capi.NOISE_FIELDS.index("pos_n_cov")] == BASE["pos_n_cov"])


def test_batch_split_by_memory():
    per = sweep.bytes_per_filter(1000, 125)
    assert per == 1000 * 48 + 125 * 60 + 208 * 8 + 20 + 48 + 32 + 56
    # everything fits: one batch
    assert sweep.plan_batches(9, 4096, per, 10 * 9 * 4096 * per) == [(0, 9)]
    # the 1 Mi filter cap: 256 settings x 4096 runs in one batch, 257 in two
    assert sweep.plan_batches(256, 4096, 1, 1 << 40) == [(0, 256)]
    assert sweep.plan_batches(257, 4096, 1, 1 << 40) == [(0, 256), (256, 1)]
    # memory for 2.5 settings (after the 0.8 headroom): whole settings, two per batch
    free = int(2.5 * 100 * per / 0.8) + 1
    assert sweep.plan_batches(5, 100, per, free) == [(0, 2), (2, 2), (4, 1)]
    with pytest.raises(ValueError):
        sweep.plan_batches(1, 100, per, 10 * per)  # not even one setting fits
    with pytest.raises(ValueError):
        sweep.plan_batches(1, 0, per, 1 << 40)


def test_help_runs_without_a_device():
    r = subprocess.run([sys.executable, "-m", "fbus_ekf_b200.sweep", "--help"], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    for flag in ("--set", "--runs", "--duration", "--eval-every", "--seed", "--device", "--out"):
        assert flag in r.stdout


def test_unknown_name_on_the_command_line_fails_before_any_device_work():
    r = subprocess.run([sys.executable, "-m", "fbus_ekf_b200.sweep", "--set", "pos_cov=1"], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 2 and "unknown parameter" in r.stderr
