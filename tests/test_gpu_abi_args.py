"""Memory kinds at the C ABI (include/fbus_ekf.h): a mem / out_mem / trace_mem argument or an fbus_imu_stream / fbus_det_frames
mem field other than FBUS_MEM_HOST or FBUS_MEM_DEVICE is rejected with FBUS_E_BADARG, names the call in fbus_last_error, leaves
the state alone and leaves the handle usable.  Every data pointer is a pinned host buffer, valid as a host and as a device
pointer, so no reading of a bad kind can fault."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

B, N_SOLVE, K = 4, 6, 4   # filters, items of the one-shot solves, frames stepped before the call under test

PAIRS = [("fbus_init_gravity_gyrobias", "imu.mem"), ("fbus_iir_prefilter", "imu.mem"), ("fbus_propagate", "imu.mem"),
         ("fbus_iir_prefilter", "out_mem"),
         ("fbus_step_windows", "imu.mem"), ("fbus_step_windows", "det.mem"), ("fbus_step_windows", "trace_mem"),
         ("fbus_init_position_quaternion", "det.mem"), ("fbus_update", "det.mem"), ("fbus_reset_state", "det.mem"),
         ("fbus_refract_solve", "mem"), ("fbus_inair_solve", "mem"), ("fbus_solve_to_detections", "mem"),
         ("fbus_undistort_fisheye", "mem"), ("fbus_refract_solve_gn", "mem"), ("fbus_marker_pose", "mem"),
         ("fbus_stats", "mem"), ("fbus_set_noise", "mem"), ("fbus_filter_errors", "mem"), ("fbus_filter_errors", "out_mem"),
         ("fbus_marker_project", "mem")]


def _pinned(a):
    """a pinned host copy of numpy array `a`, as (numpy view, address)"""
    import torch
    t = torch.empty(max(a.nbytes, 1), dtype=torch.uint8, pin_memory=True)
    v = t.numpy()[:a.nbytes].view(a.dtype).reshape(a.shape)
    v[...] = a
    return v, t.data_ptr(), t


class _Inputs:
    """the trajectory's streams and the arrays of every call, all in pinned host memory"""

    def __init__(self, cfg):
        from fbus_ekf_b200 import capi, synth
        traj = synth.truth_trajectory(cfg, duration=0.4)
        self.traj, self.W = traj, len(traj["t_frames"])
        rng = np.random.default_rng(3)
        det_id = np.zeros((self.W, 1, B), dtype=np.int32)
        det_id[K - 1, 0, 1:3] = -1   # filters 1 and 2 keep frame K-1's samples buffered for frame K: a continuation carries them
        arrays = {
            "t_imu": traj["t_imu"], "t_frames": traj["t_frames"],
            "imu": np.repeat(traj["base_imu"][:, :, None], B, axis=2),
            "det_id": det_id,
            "det_pose": np.repeat(traj["base_pose"][:, None, :, None], B, axis=3),
            "win_off": np.asarray(traj["win_off"], dtype=np.uint32),
            "trace": np.zeros((self.W, 17, B)), "iir_out": np.zeros(traj["base_imu"].shape[:1] + (6, B)),
            "corners": rng.uniform(-0.2, 0.2, (16, N_SOLVE)).astype(np.float32),
            "pose": np.repeat(traj["base_pose"][:1].T, N_SOLVE, axis=1),
            "corners3d": rng.uniform(-0.2, 0.2, (12, N_SOLVE)) + np.array([0, 0, 1.0] * 4)[:, None],
            "out_pose": np.zeros((7, N_SOLVE)), "out_c3d": np.zeros((12, N_SOLVE)), "out_f32": np.zeros((16, N_SOLVE), np.float32),
            "out_c16": np.zeros((16, N_SOLVE)), "cost": np.zeros(N_SOLVE), "valid": np.zeros(N_SOLVE, np.int32),
            "std_corners": rng.uniform(-0.2, 0.2, (16, 2 * B)).astype(np.float32), "std_ids": np.zeros((2, 1, B), np.int32),
            "std_id": np.zeros((2, 1, B), np.int32), "std_pose": np.zeros((2, 1, 7, B)),
            "truth_p": np.repeat(traj["base_pose"][-1, :3, None], B, axis=1), "truth_q": np.repeat(traj["base_pose"][-1, 3:, None], B, axis=1),
            "stats": np.zeros(capi.FBUS_NSTATS), "errors": np.zeros((4, B)), "noise": capi.noise_from_config(cfg, B),
        }
        self.v, self.p, self._keep = {}, {}, []
        for k, a in arrays.items():
            self.v[k], self.p[k], t = _pinned(np.ascontiguousarray(a))
            self._keep.append(t)

    def imu(self, mem):
        from fbus_ekf_b200 import capi
        return capi.make_imu_stream(self.v["t_imu"], self.p["imu"], B, mem)

    def det(self, mem):
        from fbus_ekf_b200 import capi
        return capi.make_det_frames(self.v["t_frames"], self.p["det_id"], self.p["det_pose"], B, 1, mem)


def _call(lib, f, x, call, param, kind):
    """`call` on handle f with `param` set to `kind` and every other memory kind FBUS_MEM_HOST"""
    from fbus_ekf_b200 import capi
    H = capi.FBUS_MEM_HOST
    m = lambda name: kind if param == name else H
    p, off, n_imu = x.p, x.v["win_off"], len(x.v["t_imu"])
    h = f._h
    if call == "fbus_init_gravity_gyrobias":
        return lib.fbus_init_gravity_gyrobias(h, C.byref(x.imu(m("imu.mem"))), 0, int(off[1]))
    if call == "fbus_iir_prefilter":
        return lib.fbus_iir_prefilter(h, C.byref(x.imu(m("imu.mem"))), 0, n_imu, p["iir_out"], m("out_mem"))
    if call == "fbus_propagate":
        return lib.fbus_propagate(h, C.byref(x.imu(m("imu.mem"))), int(off[K]), int(off[K + 1] - off[K]), float(x.v["t_frames"][K]))
    if call == "fbus_step_windows":
        return lib.fbus_step_windows(h, C.byref(x.imu(m("imu.mem"))), C.byref(x.det(m("det.mem"))),
                                     C.cast(p["win_off"], capi.c_uint32_p), K, x.W, p["trace"], m("trace_mem"))
    if call == "fbus_init_position_quaternion":
        return lib.fbus_init_position_quaternion(h, C.byref(x.det(kind)), K, int(off[K]))
    if call in ("fbus_update", "fbus_reset_state"):
        return getattr(lib, call)(h, C.byref(x.det(kind)), K)
    if call in ("fbus_refract_solve", "fbus_inair_solve"):
        return getattr(lib, call)(h, p["corners"], N_SOLVE, p["out_pose"], p["out_c3d"], p["valid"], kind)
    if call == "fbus_solve_to_detections":
        return lib.fbus_solve_to_detections(h, p["std_corners"], p["std_ids"], 2, 1, 1, 2, p["std_id"], p["std_pose"], kind)
    if call == "fbus_undistort_fisheye":
        return lib.fbus_undistort_fisheye(h, p["corners"], N_SOLVE, p["out_f32"], kind)
    if call == "fbus_refract_solve_gn":
        return lib.fbus_refract_solve_gn(h, p["corners"], 0, N_SOLVE, 2, p["out_pose"], p["cost"], p["valid"], kind)
    if call == "fbus_marker_pose":
        return lib.fbus_marker_pose(h, p["corners3d"], N_SOLVE, p["out_pose"], kind)
    if call == "fbus_stats":
        return lib.fbus_stats(h, p["truth_p"], p["truth_q"], kind, C.cast(p["stats"], capi.c_double_p), None)
    if call == "fbus_set_noise":
        return lib.fbus_set_noise(h, p["noise"], kind)
    if call == "fbus_filter_errors":
        return lib.fbus_filter_errors(h, p["truth_p"], p["truth_q"], m("mem"), p["errors"], m("out_mem"))
    if call == "fbus_marker_project":
        return lib.fbus_marker_project(h, p["pose"], N_SOLVE, 1, p["out_c16"], p["valid"], kind)
    raise AssertionError(call)


def _same_state(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), k


def _device_streams(x):
    """the trajectory's IMU and detection streams as device-resident descriptors (and the tensors that hold them)"""
    import torch
    from fbus_ekf_b200 import capi
    dev = [torch.from_numpy(np.array(x.v[k])).cuda() for k in ("imu", "det_id", "det_pose")]
    s = capi.make_imu_stream(x.traj["t_imu"], dev[0].data_ptr(), B, capi.FBUS_MEM_DEVICE)
    d = capi.make_det_frames(x.traj["t_frames"], dev[1].data_ptr(), dev[2].data_ptr(), B, 1, capi.FBUS_MEM_DEVICE)
    return s, d, dev


@pytest.mark.parametrize("bad", [2, -1])
@pytest.mark.parametrize("call,param", PAIRS)
def test_bad_memory_kind(cfg, call, param, bad):
    from fbus_ekf_b200 import BatchFilter, capi
    x = _Inputs(cfg)
    lib = capi.lib()
    f = BatchFilter(cfg, batch=B)
    f.StepWindows(x.imu(capi.FBUS_MEM_HOST), x.det(capi.FBUS_MEM_HOST), x.v["win_off"], 0, K)   # an initialised state
    before = f.GetState()
    assert _call(lib, f, x, call, param, bad) == capi.FBUS_E_BADARG
    assert call.encode() in lib.fbus_last_error(f._h)
    _same_state(before, f.GetState())
    assert _call(lib, f, x, call, param, capi.FBUS_MEM_HOST) == 0
    f.Synchronize()
    f.close()

    if call == "fbus_step_windows" and param in ("imu.mem", "trace_mem"):
        # a call rejected for these kinds does not end the continuation: [0, K), the rejected call, [K, W) equals [0, W)
        s, d, _dev = _device_streams(x)

        def run(rejected):
            g = BatchFilter(cfg, batch=B)
            if rejected is None:
                g.StepWindows(s, d, x.v["win_off"], 0, x.W)
            else:
                g.StepWindows(s, d, x.v["win_off"], 0, K)
                assert _call(lib, g, x, call, rejected, bad) == capi.FBUS_E_BADARG
                g.StepWindows(s, d, x.v["win_off"], K, x.W)
            st = g.GetState()
            g.close()
            return st

        whole = run(None)
        _same_state(whole, run(param))
        # a bad detection descriptor does end it; the samples buffered over frame K-1 then make the results differ
        assert not np.array_equal(whole["p"], run("det.mem")["p"])
