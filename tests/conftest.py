import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device visible")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    """the reference's bundled logs, {"land_imu": rows, ...}, from tests/golden/*.txt.xz (see make_golden.py)"""
    return {f"{log}_{kind}": np.loadtxt(os.path.join(ROOT, "tests", "golden", f"{log}_{kind}.txt.xz"), ndmin=2)
            for log in ("land", "water") for kind in ("corners", "image", "imu", "fusion")}


@pytest.fixture(scope="session")
def built():
    """in-tree builds: CUDA library (nvcc cross-compiles without a GPU) and the oracle"""
    import __graft_entry__ as ge
    ge.build()
    return True


@pytest.fixture(scope="session")
def cfg(built):
    from fbus_ekf_b200 import capi
    return capi.config_default()


# The window kernel exists in three forms: nine lanes per filter with the covariance in registers (small batches,
# fbus_kernel_lane.cuh; two generations, "lane" = the current one with the batch spread thin over the SMs as fbus_create does, "lane32" = the same with full 32-filter CTAs, "lane1" = the first, which the MATLAB-semantics mode still uses), one thread per filter with the covariance in shared memory (32-filter CTAs) and one thread per filter
# with the covariance in tensor memory (128-filter CTAs, batches that fill the GPU).  The parity tests work on small batches,
# so the modules listed here run once per form, forcing each kernel in turn.
_ALL_PATHS = ("test_gpu_step_parity", "test_gpu_replay_parity", "test_gpu_synth_batch", "test_gpu_init_overshoot")
_PATH_ENV = {"auto": {}, "lane": {"FBUS_LANE": "1"}, "lane32": {"FBUS_LANE": "1", "FBUS_LANE_FPC": "32"},
             "lane1": {"FBUS_LANE": "1", "FBUS_LANE_GEN": "1"},
             "smem": {"FBUS_LANE": "0", "FBUS_SMALL_BATCH": "1"}, "tmem": {"FBUS_LANE": "0", "FBUS_SMALL_BATCH": "0"}}


def pytest_generate_tests(metafunc):
    if metafunc.module.__name__.split(".")[-1] in _ALL_PATHS and "cov_store" in metafunc.fixturenames:
        metafunc.parametrize("cov_store", ["lane", "lane32", "lane1", "smem", "tmem"], indirect=True)


@pytest.fixture(autouse=True)
def cov_store(request):
    mode = getattr(request, "param", "auto")
    want = _PATH_ENV[mode]
    old = {k: os.environ.get(k) for k in ("FBUS_LANE", "FBUS_LANE_GEN", "FBUS_LANE_FPC", "FBUS_SMALL_BATCH")}
    for k in old:
        os.environ.pop(k, None)
    os.environ.update(want)
    yield mode
    for k, v in old.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v
