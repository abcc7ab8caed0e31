#!/usr/bin/env python
"""bench.py -- throughput of the batched FBUS-EKF hot path on B200 (see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the reference's own filter.cpp (oracle/_ref) on all host cores

Metric (BASELINE.json): filter-steps/sec (batched EKF, FP64).  1 filter-step = one IMU propagate (F1+F2) or one
marker-pose update (F4 incl. F5) for one filter.  Workload = BASELINE configs[4]: 1,048,576 Monte-Carlo filters per
GPU on synthetic 200 Hz IMU + 25 Hz marker poses; one bench "step" = one second of stream for every filter
(200 propagates + 25 updates per filter) through ONE launch of the fused window kernel.  The truth trajectory is
periodic in that second, so every step replays the same device-resident noisy streams with timestamps advanced by
one period: the filters keep running, nothing is reset or cached between steps.

--dump-outputs DIR writes, after the timed steps, what the timed path left its caller: the state of a fixed, seeded sample
of rank 0's filters and the statistics vector of the whole batch, as float64 DIR/<name>.npy (about 24 MB).  The inputs
depend only on the arguments, so two builds run with the same arguments can be compared output for output.

One JSON line on stdout (rank 0).  `value` = device-resident inputs; `e2e` = the same call with HOST (pinned)
buffers, i.e. host->device copies of every step's streams and a device->host read of the step's statistics inside
the timed region.  The host IMU stream of `e2e` is in the format the reference system receives it in -- the IMSEE SDK's
float32 samples in g and deg/s (FBUS_IMU_F32_SENSOR; converted on the device exactly as main.cpp:254 does, bit-identical
filter results) --; `e2e_f64_si` is the same with pre-converted doubles (twice the IMU bytes).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "filter-steps/sec (batched EKF, FP64)"
UNIT = "filter-steps/s"
# algorithmic work model (SURVEY.md 8d / BASELINE.md 3): FMA = 2 flops, structural zeros not counted, full 18x18 P
FLOP_IMU_STEP = 3050.0
FLOP_UPDATE = 8700.0
FLOP_SOLVE = 1900.0
BYTES_SOLVE = 124.0
PERIOD = 1.0  # seconds of stream per bench step
IMU_RATE, FRAME_RATE = 200.0, 25.0
DUMP_FILTERS = 8192  # filters whose whole state --dump-outputs writes: 363 doubles each, ~24 MB


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons of one GPU while the timed region runs"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax.append(float(r[1]))
            except ValueError:
                continue
            for nm, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def shifted(traj, k):
    """timestamps of bench step k (the trajectory is periodic with PERIOD)"""
    return traj["t_imu"] + k * PERIOD, traj["t_frames"] + k * PERIOD


# ------------------------------------------------------------------------------------------------------- CPU arm
def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_arm(cfg, traj, target_seconds=15.0, threads=None, max_filters=None):
    """The reference's CPU filter as independent copies on all host cores (threads pinned 1:1 to the cores the process may
    use).  oracle/_ref -- the reference's own C++/src/filter.cpp compiled unmodified against stand-in Eigen/glog/... headers
    (oracle/ref_build) -- when its prebuilt library is present ("kind": "reference"), else the oracle's dense scalar port
    ("kind": "port").  Bounded sample: `B` filters x `passes` seconds of the same synthetic stream."""
    import orc
    from fbus_ekf_b200 import capi  # ctypes struct definitions only: the product library is not loaded on this path
    threads = threads or host_threads()
    use_ref = orc.ref_available() and not os.environ.get("FBUS_BENCH_CPU_PORT")
    B = 32 * threads
    if max_filters:
        B = min(B, max_filters)
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    rng = np.random.default_rng(123)
    imu = np.ascontiguousarray(traj["base_imu"][:, :, None] + rng.normal(size=(N, 6, B)) * np.array([0.015] * 3 + [1e-3] * 3)[None, :, None])
    ids = np.zeros((W, 1, B), dtype=np.int32)
    pose = np.repeat(traj["base_pose"][:, None, :, None], B, axis=3) + rng.normal(size=(W, 1, 7, B)) * 2.5e-4
    pose[:, :, 3:7, :] /= np.linalg.norm(pose[:, :, 3:7, :], axis=2, keepdims=True)
    pose = np.ascontiguousarray(pose)
    fast = use_ref and orc.host_has_avx2() and os.path.exists(orc.REF_AVX2_LIB_PATH)
    o = ((orc.RefFast if fast else orc.Ref) if use_ref else orc.Oracle)(cfg, B)

    def one_pass(k):
        ti, tf = shifted(traj, k)
        s = capi.make_imu_stream(ti, imu, B)
        d = capi.make_det_frames(tf, ids, pose, B, 1)
        o.step_windows(s, d, traj["win_off"], 0, W, None, threads)

    t0 = time.perf_counter()
    one_pass(0)  # includes the pose initialisation frame; also calibrates the pass time
    t_pass = time.perf_counter() - t0
    passes = int(max(2, min(400, round(target_seconds / max(t_pass, 1e-3)))))
    t0 = time.perf_counter()
    for k in range(1, passes + 1):
        one_pass(k)
    dt = time.perf_counter() - t0
    steps = B * (N + W) * passes
    st = o.get_state(with_cov=False)
    finite = bool(np.isfinite(st["p"]).all())
    impl = ("oracle/_ref: the reference's own C++/src/filter.cpp compiled unmodified (g++ " + ("-O3 -mavx2" if fast else "-O2") + ") against stand-in Eigen/glog/yaml/opencv "
            "headers, one FBUSEKF::FILTER object per filter" if use_ref else "oracle/fbus_oracle.cpp (dense scalar port of filter.cpp)")
    return {"value": steps / dt, "unit": UNIT, "cores": threads, "kind": "reference" if use_ref else "port",
            "sample": f"{B} filters x {passes} s of the synthetic 200 Hz IMU + 25 Hz marker stream ({steps} filter-steps in {dt:.1f} s), "
                      f"{impl}, {threads} threads pinned 1:1", "finite": finite,
            "seconds": dt, "steps_per_pass": B * (N + W), "sample_filters": B, "sample_seconds_of_stream": passes}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on every host core, rank 0 only: oracle/_ref (the
    reference's own filter.cpp, prebuilt where /root/reference exists) or, without it, the oracle port.  Nothing of the
    product is built, loaded or called here: the configuration comes from the oracle's own restatement of the YAML files
    and the workload generator is plain NumPy."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    import orc
    orc.build()
    try:
        orc.build_ref()  # no-op without /root/reference (the GPU box uses the prebuilt oracle/_ref)
    except Exception as e:
        print(f"bench.py: oracle/_ref not built ({e}); falling back to the oracle port", file=sys.stderr)
    from fbus_ekf_b200 import synth
    cfg = orc.config_default()
    traj = synth.truth_trajectory(cfg, PERIOD, IMU_RATE, FRAME_RATE, periodic=True)
    threads = host_threads()
    k_total = max(1, args.steps)
    # each "step" = a bounded sample; whole run sized to a few minutes at most
    per_step_seconds = min(20.0, 120.0 / (k_total + args.warmup))
    for _ in range(args.warmup):
        cpu_arm(cfg, traj, target_seconds=min(2.0, per_step_seconds), threads=threads)
    vals, secs, cb = [], 0.0, None
    for _ in range(k_total):
        cb = cpu_arm(cfg, traj, target_seconds=per_step_seconds, threads=threads)
        vals.append(cb["value"])
        secs += cb["seconds"]
    v = float(np.mean(vals))
    cb["value"] = v
    conf = workload_config(env_int("FBUS_BENCH_BATCH", 1 << 20), max(1, args.gpus))
    conf["reference_sample"] = (f"each step times {cb['sample_filters']} independent filters (32 per host thread) of this workload x "
                                f"{cb['sample_seconds_of_stream']} s of stream; filters are independent, so the rate carries over to any batch")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * secs / k_total, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": conf, "cpu_baseline": cb,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), file=JSON_OUT or sys.stdout, flush=True)
    return 0


def workload_config(batch, world):
    return {"workload": "BASELINE configs[4]: 1,048,576 Monte-Carlo filters per GPU (perturbed noise seeds, Philox keyed by global "
                        "filter index) on synthetic 200 Hz IMU + 25 Hz marker poses; 1 bench step = 1 s of stream per filter",
            "filters_per_gpu": batch, "filters_total": batch * world, "imu_steps_per_filter_per_step": int(IMU_RATE * PERIOD),
            "updates_per_filter_per_step": int(FRAME_RATE * PERIOD), "state": "18-state error-state EKF, 7-row marker-pose update",
            "parallelism": f"independent filters sharded over {world} GPU(s), no hot-path collective",
            "l2": "inputs per step (imu+detections) are far larger than the 126 MB L2 at the default batch"}


# ------------------------------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local = env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        import __graft_entry__ as ge
        ge.build()
    if world > 1:
        dist.barrier()
    from fbus_ekf_b200 import BatchFilter, capi, synth

    B = env_int("FBUS_BENCH_BATCH", 1 << 20)
    K, Wm = args.steps, args.warmup
    if args.dump_outputs and rank == 0:
        # fbus_get_state reads the whole batch: host copy of every field + the library's staging of the packed covariance
        import psutil
        need = B * 8 * (sum(n for _, n, _ in capi.STATE_FIELDS) + 18 * 19 // 2)
        avail = psutil.virtual_memory().available
        if need > 0.8 * avail:
            raise SystemExit(f"bench.py: --dump-outputs reads the state of all {B} filters, {need / 1e9:.1f} GB of host memory; "
                             f"{avail / 1e9:.1f} GB are available")
    cfg = capi.config_default()
    traj = synth.truth_trajectory(cfg, PERIOD, IMU_RATE, FRAME_RATE, periodic=True)
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    steps_per_filter = N + W

    f = BatchFilter(cfg, batch=B, device=local)
    stream = torch.cuda.ExternalStream(f.stream, device=dev)
    imu_d = torch.empty((N, 6, B), dtype=torch.float64, device=dev)
    id_d = torch.empty((W, 1, B), dtype=torch.int32, device=dev)
    pose_d = torch.empty((W, 1, 7, B), dtype=torch.float64, device=dev)
    f.SynthStreams(synth.make_synth_spec(traj, seed=20260117 + 5, filter_offset=rank * B), imu_d.data_ptr(), id_d.data_ptr(),
                   pose_d.data_ptr())

    def gpu_step(k):
        ti, tf = shifted(traj, k)
        imu = capi.make_imu_stream(ti, imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE)
        det = capi.make_det_frames(tf, id_d.data_ptr(), pose_d.data_ptr(), B, 1, capi.FBUS_MEM_DEVICE)
        f.StepWindows(imu, det, traj["win_off"], 0, W)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    fp64_peak = f.MeasureFp64Peak()  # DFMA microbenchmark on this GPU: the FP64 roofline denominator (burst)

    for k in range(Wm):
        gpu_step(k)
    f.Synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    ev[0].record(stream)
    for k in range(K):
        gpu_step(Wm + k)
        ev[k + 1].record(stream)
    f.Synchronize()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = ev[0].elapsed_time(ev[K])
    launch_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(K)]
    tmax = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total_max = float(tmax.item())
    value = world * B * steps_per_filter * K / (ms_total_max * 1e-3)

    # ---- final statistics: local sums on the device, one NCCL all-reduce over NVLink (the only collective) ----------
    k_last = Wm + K - 1
    tp = torch.tensor(traj["truth_p"][-1], dtype=torch.float64, device=dev).reshape(3, 1).expand(3, B).contiguous()
    tq = torch.tensor(traj["truth_q"][-1], dtype=torch.float64, device=dev).reshape(4, 1).expand(4, B).contiguous()
    st_d = torch.zeros(capi.FBUS_NSTATS, dtype=torch.float64, device=dev)
    f.Stats(tp.data_ptr(), tq.data_ptr(), capi.FBUS_MEM_DEVICE, out_dev_ptr=st_d.data_ptr(), want_host=False)
    f.Synchronize()
    from fbus_ekf_b200 import shard
    shard.combine_stats(st_d, dist if world > 1 else None)  # SUM of the sums, MAX of the maximum
    stats_vec = st_d.cpu().numpy()
    stats = shard.summarize_stats(stats_vec)
    stats.update({"after_seconds_of_stream": (k_last + 1) * PERIOD, "allreduce": "nccl" if world > 1 else "single rank"})
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, f, stats_vec)  # before the e2e_montecarlo leg steps `f` further

    # ---- roofline of the dominant kernel (ekf_window_kernel) -------------------------------------------------------
    flop_launch = B * (N * FLOP_IMU_STEP + W * FLOP_UPDATE)
    bytes_launch = B * (N * 48.0 + W * 60.0 + 2.0 * (171 + 29) * 8.0 + 12.0)  # streams + state in/out + flags
    avg_launch_s = float(np.mean(launch_ms)) * 1e-3
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    # counters that only a profiler can give (DRAM traffic, executed FP64 instructions, pipe utilisation) come from the ncu
    # capture recorded in profiles/roofline_inputs.json.  They describe ONE build of the library: the file carries that build's
    # source hash, and they are reported only while the loaded library has the same hash (otherwise null + the reason).
    prof, prof_note = {}, None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "roofline_inputs.json")))
        lib_hash = open(os.path.join(ROOT, "fbus_ekf_b200", "libfbus_ekf.so.srchash")).read().strip()
        if prof.get("srchash") != lib_hash:
            prof_note = ("profiles/roofline_inputs.json was captured for library source hash %s, the loaded library has %s: "
                         "profiler-derived fields dropped" % (str(prof.get("srchash"))[:12], lib_hash[:12]))
            prof = {}
    except Exception as e:
        prof, prof_note = {}, f"no usable profiles/roofline_inputs.json ({e})"
    ach_tf = flop_launch / avg_launch_s / 1e12
    exe = None
    if "fp64_flop_executed_per_filter_per_launch" in prof:
        exe_tf = prof["fp64_flop_executed_per_filter_per_launch"] * B / avg_launch_s / 1e12
        exe = {"achieved": exe_tf, "frac": exe_tf / (fp64_peak / 1e12), "unit": "TFLOP/s",
               "flop_per_filter_per_launch": prof["fp64_flop_executed_per_filter_per_launch"],
               "what": "FP64 flops the kernel actually executes (ncu: 2 x DFMA + DMUL + DADD thread-level instructions of one launch of "
                       "this workload shape), divided by the launch time measured in THIS run: the structured kernel skips the "
                       "zeros and the symmetric half that the contract count includes"}
    roofline = {"kernel": "ekf_window_split_kernel<128>", "bound": "fp64", "achieved": ach_tf, "peak": fp64_peak / 1e12, "unit": "TFLOP/s",
                "frac": ach_tf / (fp64_peak / 1e12),
                "frac_executed": exe["frac"] if exe else None, "executed": exe,
                "peak_source": "DFMA-saturating microbenchmark measured live on this GPU (fbus_measure_fp64_peak, burst); "
                               "MEASURED_PEAKS.json has no FP64 entry; nominal 37.2 TFLOP/s",
                "algorithmic_flop_per_launch": flop_launch, "avg_launch_ms": avg_launch_s * 1e3,
                "fp64_pipe_busy_pct_ncu": prof.get("fp64_pipe_busy_pct_ncu"),
                "note": "achieved / frac use SURVEY 8d's algorithmic flop count (full 18x18 P, FMA = 2, zeros not counted) as the "
                        "contract defines them; frac_executed is the same launch measured by the FP64 instructions the kernel "
                        "really issues, the number to judge the kernel by",
                "profile_note": prof_note,
                "traffic": (prof["ekf_window_dram_bytes_per_filter_per_launch"] * B) if "ekf_window_dram_bytes_per_filter_per_launch" in prof else None,
                "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture at %d filters, scaled per filter "
                                  "(profiles/roofline_inputs.json)" % prof.get("measured_at_filters", 0) if prof else None,
                "hbm": {"achieved": bytes_launch / avg_launch_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": bytes_launch / avg_launch_s / 1e9 / hbm_peak, "algorithmic_bytes_per_launch": bytes_launch,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)"}}

    # ---- BASELINE configs[2]: 4 096 Monte-Carlo filters on one B200 (latency / occupancy case, 32-filter CTAs) ---------
    small = None
    small_1k = None
    if not args.no_solves:
        def small_run(Bs):
            fs = BatchFilter(cfg, batch=Bs, device=local)
            s_stream = torch.cuda.ExternalStream(fs.stream, device=dev)
            imu_s = torch.empty((N, 6, Bs), dtype=torch.float64, device=dev)
            id_s = torch.empty((W, 1, Bs), dtype=torch.int32, device=dev)
            pose_s = torch.empty((W, 1, 7, Bs), dtype=torch.float64, device=dev)
            fs.SynthStreams(synth.make_synth_spec(traj, seed=20260117 + 3, filter_offset=rank * Bs), imu_s.data_ptr(), id_s.data_ptr(),
                            pose_s.data_ptr())

            def small_step(kk):
                ti, tf = shifted(traj, kk)
                fs.StepWindows(capi.make_imu_stream(ti, imu_s.data_ptr(), Bs, capi.FBUS_MEM_DEVICE),
                               capi.make_det_frames(tf, id_s.data_ptr(), pose_s.data_ptr(), Bs, 1, capi.FBUS_MEM_DEVICE), traj["win_off"], 0, W)
            reps = max(K, 5) * 4
            for kk in range(3):
                small_step(kk)
            fs.Synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record(s_stream)
            for kk in range(reps):
                small_step(3 + kk)
            s1.record(s_stream)
            fs.Synchronize()
            fs.close()
            return world * Bs * steps_per_filter * reps / (s0.elapsed_time(s1) * 1e-3), s0.elapsed_time(s1) / reps
        v, ms = small_run(4096)
        small = {"workload": "BASELINE configs[2]: 4,096 Monte-Carlo filters, 1 s of 200 Hz IMU + 25 Hz marker poses per launch",
                 "value": v, "unit": UNIT, "ms_per_launch": ms,
                 "kernel": "ekf_window_split_kernel<32> (one thread per filter, 32-filter CTAs): 28 filters per SM, latency-bound"}
        v, ms = small_run(1024)
        small_1k = {"workload": "1,024 Monte-Carlo filters, same streams", "value": v, "unit": UNIT, "ms_per_launch": ms,
                    "kernel": "ekf_window_lane2_kernel (nine lanes per filter, 7 filters per CTA)"}

    # ---- the live use of the reference: ONE filter, one detection frame per call with host arrays (what the C++ shim does
    #      in SetDetectionResultUpdated): latency of a frame, H2D of its ~8 IMU samples and the synchronisation included ----
    single = None
    if not args.no_solves and rank == 0:
        f1 = BatchFilter(cfg, batch=1, device=local)
        imu1 = np.ascontiguousarray(traj["base_imu"][:, :, None])
        id1 = np.zeros((W, 1, 1), dtype=np.int32)
        pose1 = np.ascontiguousarray(traj["base_pose"][:, None, :, None])
        lat = []
        for kk in range(4):
            ti, tf = shifted(traj, kk)
            imu_v = capi.make_imu_stream(ti, imu1, 1)
            det_v = capi.make_det_frames(tf, id1, pose1, 1, 1)
            for w in range(W):
                t0 = time.perf_counter()
                f1.StepWindows(imu_v, det_v, traj["win_off"], w, w + 1)
                f1.Synchronize()
                if kk > 0:
                    lat.append(time.perf_counter() - t0)
        lat = np.sort(np.array(lat)) * 1e6
        single = {"workload": "one filter, one detection frame (8 IMU samples + 1 marker pose) per fbus_step_windows call, host arrays, "
                              "synchronised after every frame", "frames": int(lat.size), "median_us": float(np.median(lat)),
                  "p95_us": float(lat[int(0.95 * (lat.size - 1))]), "frame_period_of_the_camera_us": 1e6 / FRAME_RATE}
        f1.close()

    # ---- refractive solves/sec (second half of the metric): K3+K4 on 524,288 markers per launch ---------------------
    solves = bench_solves(f, cfg, dev, stream, K, Wm, world, fp64_peak, hbm_peak) if not args.no_solves else None

    config4 = bench_config4(cfg, dev, local, rank, world, K, Wm) if not args.no_solves else None
    config4_tol = bench_config4(cfg, dev, local, rank, world, K, Wm, gn_tol=1e-8) if not args.no_solves else None

    # ---- e2e: HOST buffers through the C ABI, H2D of every step's streams + D2H of the step's statistics -------------
    # The host IMU stream is in the format the reference system receives it in: the IMSEE SDK's float32 samples in g and deg/s
    # (indem::ImuData, driver/IMSEE-SDK/include/types.h:122-127; main.cpp:252-256 converts each sample before SetImuData).
    e2e = bench_e2e(cfg, traj, imu_d, id_d, pose_d, B, local, dev, world, K, Wm, tp, tq, sensor_f32=True) if not args.no_e2e else None
    # the same with the samples pre-converted to doubles on the host (IMUData's fields; twice the IMU bytes over PCIe)
    e2e_f64 = bench_e2e(cfg, traj, imu_d, id_d, pose_d, B, local, dev, world, K, Wm, tp, tq, sensor_f32=False) if not args.no_e2e else None
    # Monte-Carlo use: the host sends the shared base trajectory + a seed, the per-filter noisy streams are generated on the
    # device inside the timed region (fbus_synth_streams + fbus_step_windows + fbus_stats).  A different experiment, never a
    # replacement for `e2e`.
    e2e_mc = bench_e2e_montecarlo(f, cfg, traj, imu_d, id_d, pose_d, B, rank, dev, world, K, Wm, tp, tq) if not args.no_e2e else None
    strong = bench_strong(cfg, traj, local, rank, dev, world, K, Wm, value) if not args.no_solves or world > 1 else None

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu_baseline = cpu_arm(cfg, traj, target_seconds=12.0)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
                "ms_per_step": ms_total_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": workload_config(B, world), "e2e": e2e, "e2e_f64_si": e2e_f64,
                "e2e_montecarlo": e2e_mc, "strong_scaling": strong, "gpu_launches": K, "library_build": library_build_info(),
                "roofline": roofline, "cpu_baseline": cpu_baseline, "clocks": clocks, "stats": stats, "solves": solves,
                "small_batch": small, "small_batch_1024": small_1k, "single_filter": single, "config4": config4, "config4_gn_tol": config4_tol,
                "timing": "CUDA events on the library's stream, barrier + synchronize on both sides, max over ranks"}
        print(json.dumps(line), file=JSON_OUT or sys.stdout, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def bench_solves(f, cfg, dev, stream, K, Wm, world, fp64_peak, hbm_peak):
    import torch
    from fbus_ekf_b200 import capi, synth
    n_unique = 65536
    rng = np.random.default_rng(99)
    c = synth.random_marker_corners(cfg, n_unique, rng)
    n = n_unique * 8  # BASELINE configs[3]: 65,536 filters x 8 markers per frame
    reps = 32         # distinct corner sets so that successive launches stream new data (32 x 33.5 MB > L2)
    base = torch.from_numpy(c).to(dev)
    corners = torch.empty((reps, 16, n), dtype=torch.float32, device=dev)
    for r in range(reps):
        corners[r] = base.repeat(1, 8) + (1e-4 * (r + 1)) * torch.randn((16, n), device=dev, dtype=torch.float32)
    pose = torch.empty((7, n), dtype=torch.float64, device=dev)
    valid = torch.empty((n,), dtype=torch.int32, device=dev)
    iters = max(K * 8, 16)
    for i in range(max(Wm, 3)):
        f.RefractSolveDevice(corners[i % reps].data_ptr(), n, pose.data_ptr(), None, valid.data_ptr())
    f.Synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(iters):
        f.RefractSolveDevice(corners[i % reps].data_ptr(), n, pose.data_ptr(), None, valid.data_ptr())
    e1.record(stream)
    f.Synchronize()
    sec = e0.elapsed_time(e1) * 1e-3 / iters
    rate = n / sec
    # e2e: pinned host corners in, poses + flags out
    hc = torch.empty((16, n), dtype=torch.float32).pin_memory()
    hc.copy_(corners[0].cpu())
    hp = torch.empty((7, n), dtype=torch.float64).pin_memory()
    hv = torch.empty((n,), dtype=torch.int32).pin_memory()
    lib = capi.lib()

    def host_call():
        rc = lib.fbus_refract_solve(f._h, hc.data_ptr(), n, hp.data_ptr(), None, hv.data_ptr(), capi.FBUS_MEM_HOST)
        assert rc == 0
    for _ in range(3):
        host_call()
    t0 = time.perf_counter()
    for _ in range(max(K, 4)):
        host_call()
    e2e_rate = n * max(K, 4) / (time.perf_counter() - t0)
    # R3 (north_star): closed form + 5 Gauss-Newton iterations, same markers
    cost = torch.empty((n,), dtype=torch.float64, device=dev)
    lib.fbus_refract_solve_gn(f._h, corners[0].data_ptr(), 0, n, 5, pose.data_ptr(), cost.data_ptr(), valid.data_ptr(), capi.FBUS_MEM_DEVICE)
    f.Synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g_iters = max(K, 4)
    g0.record(stream)
    for i in range(g_iters):
        lib.fbus_refract_solve_gn(f._h, corners[i % reps].data_ptr(), 0, n, 5, pose.data_ptr(), cost.data_ptr(), valid.data_ptr(),
                                  capi.FBUS_MEM_DEVICE)
    g1.record(stream)
    f.Synchronize()
    gn_rate = n * g_iters / (g0.elapsed_time(g1) * 1e-3)
    # the same with the convergence stop (fbus_config.gn_tol = 1e-8, at most 5 iterations; north_star's pose tolerance is 1e-8): a second handle, same markers
    import copy
    from fbus_ekf_b200 import BatchFilter
    cfg_t = copy.copy(cfg)
    cfg_t.gn_tol = 1e-8
    ft = BatchFilter(cfg_t, batch=1, device=dev.index)
    t_stream = torch.cuda.ExternalStream(ft.stream, device=dev)
    pose_t = torch.empty_like(pose)
    for i in range(2):
        lib.fbus_refract_solve_gn(ft._h, corners[i % reps].data_ptr(), 0, n, 5, pose_t.data_ptr(), cost.data_ptr(), valid.data_ptr(), capi.FBUS_MEM_DEVICE)
    ft.Synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record(t_stream)
    for i in range(g_iters):
        lib.fbus_refract_solve_gn(ft._h, corners[i % reps].data_ptr(), 0, n, 5, pose_t.data_ptr(), cost.data_ptr(), valid.data_ptr(),
                                  capi.FBUS_MEM_DEVICE)
    g1.record(t_stream)
    ft.Synchronize()
    gn_tol_rate = n * g_iters / (g0.elapsed_time(g1) * 1e-3)
    gn_tol_diff = float((pose_t - pose).abs().max().item())  # same markers (last launch of both loops): converged vs 5 iterations
    ft.close()
    return {"metric": "refractive solves/sec", "value": rate * world, "gauss_newton_5it_solves_per_s": gn_rate * world,
            "gauss_newton_tol1e-8_max5it_solves_per_s": gn_tol_rate * world, "gauss_newton_tol_vs_5it_max_abs_diff": gn_tol_diff, "unit": "solves/s", "markers_per_launch": n,
            "ms_per_launch": sec * 1e3, "valid_fraction": float(valid.float().mean().item()),
            "e2e": {"value": e2e_rate * world, "unit": "solves/s", "h2d_bytes_per_step": 64 * n, "d2h_bytes_per_step": 60 * n},
            "roofline": {"kernel": "refract_kernel", "bound": "fp64", "achieved": rate * FLOP_SOLVE / 1e12, "peak": fp64_peak / 1e12,
                         "unit": "TFLOP/s", "frac": rate * FLOP_SOLVE / fp64_peak,
                         "hbm": {"achieved": rate * BYTES_SOLVE / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": rate * BYTES_SOLVE / 1e9 / hbm_peak}}}


def bench_config4(cfg, dev, local, rank, world, K, Wm, gn_tol=0.0):
    """BASELINE configs[3]: 65,536 filters, per frame 8 board markers x 4 corners x stereo -> refractive solve with 5
    Gauss-Newton iterations -> detection frames -> EKF (nearest of 8 markers), device-resident; one step = 1 s of stream."""
    import torch
    from fbus_ekf_b200 import BatchFilter, capi, synth
    B4, m, gn = env_int("FBUS_BENCH_BATCH4", 65536), 8, 5
    bcfg = synth.board_config(cfg)
    bcfg.gn_tol = gn_tol
    traj = synth.truth_trajectory(bcfg, PERIOD, IMU_RATE, FRAME_RATE, periodic=True, standoff=1.0)
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    base, ids, _ = synth.board_base_corners(bcfg, traj)
    f = BatchFilter(bcfg, batch=B4, device=local)
    stream = torch.cuda.ExternalStream(f.stream, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(4 + rank)
    n = W * m * B4
    corners = torch.from_numpy(base.astype(np.float32)).to(dev).reshape(16, W * m, 1).expand(16, W * m, B4).reshape(16, n).contiguous()
    corners += 2e-4 * torch.randn((16, n), device=dev, dtype=torch.float32, generator=g)
    mids = torch.from_numpy(ids).to(dev).reshape(W, m, 1).expand(W, m, B4).contiguous()
    det_id = torch.empty((W, m, B4), dtype=torch.int32, device=dev)
    det_pose = torch.empty((W, m, 7, B4), dtype=torch.float64, device=dev)
    imu_d = torch.from_numpy(traj["base_imu"]).to(dev).reshape(N, 6, 1).expand(N, 6, B4).contiguous()
    imu_d += torch.tensor([0.015] * 3 + [1e-3] * 3, device=dev, dtype=torch.float64).reshape(1, 6, 1) * \
        torch.randn((N, 6, B4), device=dev, dtype=torch.float64, generator=g)
    torch.cuda.synchronize(dev)

    def step(kk):
        ti, tf = shifted(traj, kk)
        f.SolveToDetections(corners.data_ptr(), mids.data_ptr(), W, m, True, gn, det_id.data_ptr(), det_pose.data_ptr(), capi.FBUS_MEM_DEVICE)
        f.StepWindows(capi.make_imu_stream(ti, imu_d.data_ptr(), B4, capi.FBUS_MEM_DEVICE),
                      capi.make_det_frames(tf, det_id.data_ptr(), det_pose.data_ptr(), B4, m, capi.FBUS_MEM_DEVICE), traj["win_off"], 0, W)
    for kk in range(max(Wm, 3)):
        step(kk)
    f.Synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = max(K, 3)
    e0.record(stream)
    for kk in range(reps):
        step(max(Wm, 3) + kk)
    e1.record(stream)
    f.Synchronize()
    sec = e0.elapsed_time(e1) * 1e-3 / reps
    st = f.GetState(with_cov=False)
    err = np.linalg.norm(st["p"] - traj["truth_p"][-1][:, None], axis=0)
    out = {"workload": "BASELINE configs[3]: 65,536 filters, 8 markers x 4 corners x stereo per frame, refractive solve + 5 GN "
                       "iterations -> detections -> EKF, 1 s of 200 Hz IMU + 25 Hz frames per step",
           "filters_per_gpu": B4, "ms_per_step": sec * 1e3, "filter_steps_per_s": world * B4 * (N + W) / sec,
           "refractive_gn_solves_per_s": world * n / sec, "rmse_pos_m": float(np.sqrt(np.mean(err ** 2))),
           "finite": bool(np.isfinite(st["p"]).all()), "gpu_launches_per_step": 2,
           "gn": "exactly 5 iterations" if gn_tol <= 0 else f"at most 5 iterations, a marker stops once an applied step is below {gn_tol:g} (fbus_config.gn_tol)"}
    f.close()
    return out


def bind_to_gpu_numa_node(local: int):
    """Pins this process to the CPUs of the NUMA node its GPU hangs off (sysfs: the PCI device's numa_node / local_cpulist), so
    that pinned host buffers allocated afterwards are first touched -- and therefore placed -- on that node and the H2D DMA
    does not cross the socket interconnect.  Returns what was done, for the bench line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        if all(hasattr(pr, a) for a in ("pci_domain_id", "pci_bus_id", "pci_device_id")):
            bus = f"{int(pr.pci_domain_id):04x}:{int(pr.pci_bus_id):02x}:{int(pr.pci_device_id):02x}.0"
        else:
            import pynvml
            pynvml.nvmlInit()
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local)).busId
            bus = (bus.decode() if isinstance(bus, bytes) else str(bus)).lower()
            if len(bus.split(":")[0]) == 8:  # NVML prints an 8-digit PCI domain, sysfs a 4-digit one
                bus = bus[4:]
        base = f"/sys/bus/pci/devices/{bus}"
        node = int(open(base + "/numa_node").read().strip())
        cpus = open(base + "/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            if "-" in part:
                a, b = part.split("-")
                ids.update(range(int(a), int(b) + 1))
            elif part:
                ids.add(int(part))
        allowed = os.sched_getaffinity(0)
        use = (ids & allowed) or allowed
        os.sched_setaffinity(0, use)
        n_nodes = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()])
        return {"gpu_pci": bus, "numa_node": node, "numa_nodes_on_host": n_nodes, "cpus_bound": len(use)}
    except Exception as e:
        return {"error": f"not bound ({e})"}


def bench_e2e(cfg, traj, imu_d, id_d, pose_d, B, local, dev, world, K, Wm, tp, tq, sensor_f32=False):
    """Same metric through the public API with HOST buffers: every step copies that step's per-filter streams from pinned
    host memory to the device and reads the step's statistics vector back.  sensor_f32: the IMU stream is handed over in
    the IMSEE sensor's own format (float32, g and deg/s; FBUS_IMU_F32_SENSOR) and converted on the device as the
    reference's IMU callback does -- half the bytes per sample, same doubles inside the filter."""
    import psutil
    import torch
    import torch.distributed as dist
    from fbus_ekf_b200 import BatchFilter, capi
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    per_filter = N * (24 if sensor_f32 else 48) + W * 60
    local_world = env_int("LOCAL_WORLD_SIZE", world)
    budget = 0.15 * psutil.virtual_memory().available / max(local_world, 1)
    Be = B
    while Be > 4096 and Be * per_filter > budget:
        Be //= 2
    Be = env_int("FBUS_BENCH_E2E_BATCH", Be)
    numa = bind_to_gpu_numa_node(local)  # pinned buffers are first touched below: allocate them on the GPU's own NUMA node
    f2 = BatchFilter(cfg, batch=Be, device=local)
    h_imu = torch.empty((N, 6, Be), dtype=torch.float32 if sensor_f32 else torch.float64).pin_memory()
    h_id = torch.empty((W, 1, Be), dtype=torch.int32).pin_memory()
    h_pose = torch.empty((W, 1, 7, Be), dtype=torch.float64).pin_memory()
    if sensor_f32:  # nearest sensor-unit sample of the synthetic SI stream (capi.si_to_sensor, on the device)
        raw = torch.empty((N, 6, Be), dtype=torch.float32, device=dev)
        raw[:, 0:3] = (imu_d[:, 0:3, :Be] / cfg.imu_g).float()
        raw[:, 3:6] = (imu_d[:, 3:6, :Be] * (180.0 / capi.REF_M_PI)).float()
        h_imu.copy_(raw)
        del raw
    else:
        h_imu.copy_(imu_d[:, :, :Be])
    h_id.copy_(id_d[:, :, :Be])
    h_pose.copy_(pose_d[:, :, :, :Be])
    tpe, tqe = tp[:, :Be].contiguous(), tq[:, :Be].contiguous()
    lib = capi.lib()
    import ctypes as C
    off = np.ascontiguousarray(traj["win_off"], dtype=np.uint32)

    def step(k):
        ti, tf = shifted(traj, k)
        imu = capi.make_imu_stream(ti, h_imu.data_ptr(), Be, capi.FBUS_MEM_HOST,
                                   fmt=capi.FBUS_IMU_F32_SENSOR if sensor_f32 else capi.FBUS_IMU_F64_SI)
        det = capi.make_det_frames(tf, h_id.data_ptr(), h_pose.data_ptr(), Be, 1, capi.FBUS_MEM_HOST)
        rc = lib.fbus_step_windows(f2._h, C.byref(imu), C.byref(det), capi.dptr(off, capi.c_uint32_p), 0, W, None, 0)
        assert rc == 0
        return f2.Stats(tpe.data_ptr(), tqe.data_ptr(), capi.FBUS_MEM_DEVICE)  # 64-byte D2H, synchronises

    for k in range(max(Wm, 1)):
        step(k)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for k in range(K):
        last = step(Wm + k)
    torch.cuda.synchronize(dev)
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    sec = float(dt.item())
    f2.close()
    return {"value": world * Be * (N + W) * K / sec, "unit": UNIT, "h2d_bytes_per_step": int(Be * per_filter + (N + 2 * W + 1) * 8),
            "d2h_bytes_per_step": 64, "filters_per_gpu": Be, "ms_per_step": 1e3 * sec / K, "host_numa": numa,
            "h2d_gb_per_s_per_gpu": Be * per_filter * K / sec / 1e9,
            "api": "fbus_step_windows(FBUS_MEM_HOST streams in pinned memory%s) + fbus_stats -> host"
                   % (", IMU samples as float32 sensor units (FBUS_IMU_F32_SENSOR), converted on the device as main.cpp:254 does" if sensor_f32 else ""),
            "rmse_pos_m_last_step": float(np.sqrt(last[0] / max(last[3], 1.0)))}


def bench_e2e_montecarlo(f, cfg, traj, imu_d, id_d, pose_d, B, rank, dev, world, K, Wm, tp, tq):
    """Monte-Carlo experiment end to end: per step the host hands over only the shared noise-free trajectory (base IMU,
    base marker poses: a few KB) and a seed; the B per-filter noisy streams are generated on the device (Philox keyed by the
    global filter index), filtered, and the statistics vector is read back -- all inside the timed region."""
    import torch
    import torch.distributed as dist
    from fbus_ekf_b200 import capi, synth
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]

    def step(k):
        spec = synth.make_synth_spec(traj, seed=20260117 + 100 + k, filter_offset=rank * B)
        f.SynthStreams(spec, imu_d.data_ptr(), id_d.data_ptr(), pose_d.data_ptr())
        ti, tf = shifted(traj, k)
        f.StepWindows(capi.make_imu_stream(ti, imu_d.data_ptr(), B, capi.FBUS_MEM_DEVICE),
                      capi.make_det_frames(tf, id_d.data_ptr(), pose_d.data_ptr(), B, 1, capi.FBUS_MEM_DEVICE), traj["win_off"], 0, W)
        return f.Stats(tp.data_ptr(), tq.data_ptr(), capi.FBUS_MEM_DEVICE)  # 64-byte D2H, synchronises

    base = Wm + K + 8  # continue after the device-resident run's timestamps
    for k in range(2):
        step(base + k)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for k in range(K):
        last = step(base + 2 + k)
    torch.cuda.synchronize(dev)
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    sec = float(dt.item())
    return {"value": world * B * (N + W) * K / sec, "unit": UNIT, "h2d_bytes_per_step": int((N * 6 + W * 7 + N + 2 * W + 1) * 8),
            "d2h_bytes_per_step": 64, "filters_per_gpu": B, "ms_per_step": 1e3 * sec / K, "gpu_launches_per_step": 3,
            "api": "fbus_synth_streams(base trajectory + seed) + fbus_step_windows(device streams) + fbus_stats -> host",
            "rmse_pos_m_last_step": float(np.sqrt(last[0] / max(last[3], 1.0)))}


def bench_strong(cfg, traj, local, rank, dev, world, K, Wm, weak_value):
    """BASELINE configs[4] as worded: 1,048,576 filters IN TOTAL sharded over the ranks (strong scaling), next to the weak
    `value` of the line (1,048,576 per GPU).  Shards are contiguous global index ranges (shard.shard_range), the Philox
    streams are keyed by the global index, so the union of the shards is the N = 1 batch bit for bit."""
    import torch
    import torch.distributed as dist
    from fbus_ekf_b200 import BatchFilter, capi, shard, synth
    total = env_int("FBUS_BENCH_TOTAL", 1 << 20)
    N, W = traj["base_imu"].shape[0], traj["base_pose"].shape[0]
    if world == 1 and total == env_int("FBUS_BENCH_BATCH", 1 << 20):
        return {"filters_total": total, "filters_per_gpu": total, "value": weak_value, "unit": UNIT,
                "note": "at N = 1 the strong and the weak workload are the same launch: value repeated"}
    lo, hi = shard.shard_range(total, rank, world)
    Bs = hi - lo
    f = BatchFilter(cfg, batch=Bs, device=local)
    stream = torch.cuda.ExternalStream(f.stream, device=dev)
    imu_d = torch.empty((N, 6, Bs), dtype=torch.float64, device=dev)
    id_d = torch.empty((W, 1, Bs), dtype=torch.int32, device=dev)
    pose_d = torch.empty((W, 1, 7, Bs), dtype=torch.float64, device=dev)
    f.SynthStreams(synth.make_synth_spec(traj, seed=20260117 + 5, filter_offset=lo), imu_d.data_ptr(), id_d.data_ptr(), pose_d.data_ptr())

    def step(k):
        ti, tf = shifted(traj, k)
        f.StepWindows(capi.make_imu_stream(ti, imu_d.data_ptr(), Bs, capi.FBUS_MEM_DEVICE),
                      capi.make_det_frames(tf, id_d.data_ptr(), pose_d.data_ptr(), Bs, 1, capi.FBUS_MEM_DEVICE), traj["win_off"], 0, W)
    for k in range(max(Wm, 3)):
        step(k)
    f.Synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    reps = max(K, 5) * 2
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(reps):
        step(max(Wm, 3) + k)
    e1.record(stream)
    f.Synchronize()
    if world > 1:
        dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / reps
    f.close()
    v = total * (N + W) / (ms * 1e-3)
    return {"filters_total": total, "filters_per_gpu": Bs, "value": v, "unit": UNIT, "ms_per_step": ms,
            "vs_weak_per_gpu_rate": v / weak_value if weak_value else None,
            "note": "value / (weak value of this line) = strong-scaling efficiency against N x the single-GPU rate at 1,048,576 "
                    "filters per GPU; CUDA events on each rank's stream, barrier both sides, max over ranks"}


def dump_outputs(out_dir, f, stats_vec):
    """--dump-outputs: the state fbus_get_state returns after the last timed step (every field, covariance included) for
    DUMP_FILTERS filters (FBUS_BENCH_DUMP_FILTERS) drawn with a fixed seed (all of them for a smaller batch), their indices,
    and the statistics vector of the whole batch; all as float64 .npy files."""
    n = env_int("FBUS_BENCH_DUMP_FILTERS", DUMP_FILTERS)
    st = f.GetState()
    if f.batch <= n:
        idx = np.arange(f.batch)
    else:
        idx = np.sort(np.random.default_rng(0).choice(f.batch, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "filter_index.npy"), idx.astype(np.float64))
    for name, a in st.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a[..., idx], dtype=np.float64))
    np.save(os.path.join(out_dir, "stats.npy"), np.asarray(stats_vec, dtype=np.float64))


def library_build_info():
    """which build of the CUDA library ran: its source hash, and whether this process compiled it or found it prebuilt"""
    try:
        from fbus_ekf_b200 import build as b
        return {"srchash": open(b.HASH_FILE).read().strip()[:16], "mode": b.LAST_MODE, "built_with": b.built_with()}
    except Exception as e:
        return {"error": str(e)}


JSON_OUT = None  # the process's real stdout, kept for the one JSON line


def main():
    # stdout carries the ONE JSON line and nothing else: whatever libraries print at the C level (NCCL's version banner
    # under NCCL_DEBUG=VERSION ignores NCCL_DEBUG_FILE, make, nvcc) is sent to stderr by pointing fd 1 at fd 2
    global JSON_OUT
    sys.stdout.flush()
    JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-solves", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the state after the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm times bounded CPU samples")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
