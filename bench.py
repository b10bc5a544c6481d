#!/usr/bin/env python3
"""bench.py -- robot-instance control steps/s of the full controller tick on N B200s (BASELINE.json configs[4]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload full|vehicle]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch.
  --workload full (default; BASELINE.json configs[4]): the full controller tick -- vehicle at 1 kHz, IMU
      update + arm tick at 100 Hz, coupled through the IMU yaw -- over `--total` robots (2^24)
      batch-sharded across the GPUs (strong scaling), run in chunks of `--chunk` robots x `--ticks` fused ticks.
      The configs[1] / [2] / [3] module numbers ride along under "modules".
  --workload vehicle (BASELINE.json configs[1]): one launch of the fused rollout kernel over
      `--instances` vehicles per GPU x `--ticks` 1 kHz control ticks, closed loop through the
      integer motor plant.  Weak scaling (per-GPU batch fixed).
Rank 0 prints ONE JSON line (see DESIGN.md "Measurement").

  value        whole-job instance-steps/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e          the same metric through the C-ABI starting from HOST memory: per chunk a 48-byte stream
               descriptor (seed, first robot, distribution parameters) is copied H2D, the rk_stream_* kernels
               expand it into the command / sensor tables on the device, the rollout runs, the per-robot cost
               vector is copied D2H -- all inside the timed region
  roofline     algorithmic FP32 flops of the dominant kernel (183 per vehicle tick, SURVEY.md App. B) / its
               slot of the timed region, against the FP32 FFMA peak measured live by rk_probe_fp32
               (MEASURED_PEAKS.json carries no FP32 entry); HBM figures of the step under roofline["step"]
  cpu_baseline the reference's own sources compiled for x86 (oracle/_ref) -- or the plain-C port
               if the prebuilt .so is absent -- on the box's host cores, bounded sample
  --impl reference   times only that CPU implementation and prints the same JSON shape
The parity spot check (sampled robots of the exact bench launch against the oracle) runs on EVERY rank.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

FLOP_PER_TICK = 183        # SURVEY.md Appendix B (83 add/sub + 93 mul + 7 div), + 8 FP64 mul
STATE_BYTES = 448          # include/robotick.h RK_VS_WORDS * 4
METRIC = "robot-instance control steps/sec"
UNIT = "instance-steps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="full", choices=["vehicle", "full"])
    ap.add_argument("--instances", type=int, default=1 << 20, help="vehicles per GPU (workload vehicle)")
    ap.add_argument("--total", type=int, default=1 << 24, help="robots over all GPUs (workload full)")
    ap.add_argument("--chunk", type=int, default=1 << 20, help="robots per rk_tick_rollout call (workload full)")
    ap.add_argument("--slow-period", type=int, default=10, help="vehicle ticks per IMU/arm tick (workload full)")
    ap.add_argument("--lanes", type=int, default=2, help="CUDA streams the chunks of a pass alternate over (workload full)")
    ap.add_argument("--ticks", type=int, default=1000, help="fused control ticks per launch")
    ap.add_argument("--seg-len", type=int, default=125)
    ap.add_argument("--yaw-period", type=int, default=10)
    ap.add_argument("--cpu-seconds", type=float, default=4.0, help="wall budget of the cpu_baseline leg")
    ap.add_argument("--occupancy", type=int, default=0, help="RK_OPT_FAST_OCCUPANCY override (tuning)")
    ap.add_argument("--packed", type=int, default=-1, help="RK_OPT_FAST_PACKED override (tuning; -1 = library default)")
    ap.add_argument("--ffsat", type=int, default=-1, help="RK_OPT_FAST_FFSAT override (tuning; -1 = library default)")
    ap.add_argument("--gen-ctas", type=int, default=2, help="e2e: RK_OPT_STREAM_CTAS while the stream generators run beside the rollout")
    ap.add_argument("--side-ctas", type=int, default=-1, help="RK_OPT_TICK_SIDE_CTAS override (tuning; -1 = library default)")
    ap.add_argument("--no-modules", action="store_true", help="workload full: skip the configs[1..3] module measurements")
    ap.add_argument("--no-yaw-column", action="store_true", help="workload full: the vehicle reads the yaw from the IMU register cells instead of the 2-byte Yaw column")
    ap.add_argument("--e2e-tables", action="store_true", help="workload full: the e2e path materialises the IMU register table instead of drawing the samples inside the IMU update")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-skip", default="", help="tuning only: comma list of gen,reset,d2h left out of the e2e pass (its number is then not an e2e number)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (a fixed, seeded sample of at most "
                         f"{DUMP_ROBOTS} robots per rank) to DIR/<name>.npy")
    return ap.parse_args()


DUMP_ROBOTS = 32768  # ~56 MB for the full tick: cost + vehicle, IMU and arm state words as float64


def dump_outputs(out_dir, n_rank, lo, rank, world, parts):
    """Write a seeded sample of this rank's robots to out_dir/<name>.npy.  parts: [(robots, cost, {name: (state, words)})], one
    per batch of `robots` consecutive robots (a chunk), holding device tensors.  State blocks are SoA ([words/4, robots, 4]); each
    sampled robot's words are written as float64 (every uint32 word is exact there).  The sample depends only on the robot count,
    so two builds run with the same arguments dump the same robots."""
    import torch

    m = min(DUMP_ROBOTS, n_rank)
    pick = np.sort(np.random.default_rng(0x5EED).choice(n_rank, m, replace=False))
    out, base = {"robot": [], "cost": []}, 0
    for robots, cost, states in parts:
        idx = pick[(pick >= base) & (pick < base + robots)] - base
        it = torch.from_numpy(idx).to(cost.device)
        out["robot"].append((idx + base + lo).astype(np.float64))
        out["cost"].append(cost[it].cpu().numpy().astype(np.float32))
        for name, (st, words) in states.items():
            w = st.view(words // 4, robots, 4)[:, it].permute(1, 0, 2).reshape(len(idx), words)
            out.setdefault(name, []).append(w.cpu().numpy().view(np.uint32).astype(np.float64))
        base += robots
    os.makedirs(out_dir, exist_ok=True)
    sfx = f"_rank{rank}" if world > 1 else ""
    for name, arrs in out.items():
        np.save(os.path.join(out_dir, f"{name}{sfx}.npy"), np.concatenate(arrs))


def workload_name(a):
    if a.workload == "full":
        return (f"configs[4]: full controller tick, {a.total} robots batch-sharded over {a.gpus} GPU(s) x {a.ticks} fused 1 kHz "
                f"vehicle ticks (closed loop through the integer motor plant, command every {a.seg_len} ticks) + WT901 IMU "
                f"update and 5-axis arm tick every {a.slow_period} ticks, IMU yaw -> vehicle as VD_task_main.cpp:368; "
                f"chunks of {a.chunk} robots")
    return (f"configs[1]: {a.instances} mecanum vehicles/GPU x {a.ticks} fused 1 kHz ticks "
            f"(rx_callback + FK/odometry + 3x const-jerk target + IK + 4x FF_PI_D + current saturation), "
            f"closed loop through the integer motor plant, command every {a.seg_len} ticks, yaw every {a.yaw_period}"
            " as the WT901C Yaw register (int16)")


# ------------------------------------------------------------------------------------------
# CPU arm: the reference's own code (oracle/_ref) or the C port, all host threads
# ------------------------------------------------------------------------------------------
def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class CpuArm:
    def __init__(self, a):
        import oracle_lib as ol
        import workloads as wl
        from roboken_fmskf_robot_controller_b200 import _cabi

        self.ol, self.wl, self._cabi = ol, wl, _cabi
        self.a = a
        self.threads = host_threads()
        self.kind = "reference" if os.path.exists(os.path.join(ol.ORACLE, "_ref", "libref_vdt.so")) else "port"
        self._inp = {}

    def _run(self, n, threads=None):
        a = self.a
        threads = threads or self.threads
        if n not in self._inp:
            from roboken_fmskf_robot_controller_b200 import streams

            n_seg, n_yaw = (a.ticks + a.seg_len - 1) // a.seg_len, (a.ticks + a.yaw_period - 1) // a.yaw_period
            inp = dict(cmd=streams.vehicle_commands_v2(n, n_seg, 0x5EED, 0), yaw=streams.vehicle_yaw_reg_v2(n, n_yaw, 0x5EED, 0))
            ro = self.ol.HostRollout(n, a.ticks, self._cabi.RK_SENSOR_PLANT, inp["cmd"], a.seg_len, inp["yaw"], a.yaw_period)
            self._inp[n] = (inp, ro)
        _, ro = self._inp[n]
        t0 = time.perf_counter()
        if self.kind == "reference":
            self.ol.run_ref(None, n, ro, nthreads=threads)
        else:
            self.ol.run_port(None, n, ro, nthreads=threads)
        return time.perf_counter() - t0

    def calibrate(self, step_budget_s):
        """Pick the per-step sample (instances) so that one step takes about step_budget_s."""
        n0 = 64 * self.threads
        self._run(n0)  # warm caches / page in
        dt = self._run(n0)
        rate = n0 * self.a.ticks / dt
        n = int(rate * step_budget_s / self.a.ticks)
        n = max(self.threads * 16, min(n, self.a.instances))
        return (n // self.threads) * self.threads

    def sample_desc(self, n):
        return (f"{n} of {self.a.instances} instances x {self.a.ticks} ticks per step, same seeded command/yaw "
                f"streams and plant, {self.threads} host threads over instances")


# ---- full tick on the CPU: per-module oracles composed exactly as tests/oracle_lib.full_tick ----
_FULL_CACHE = {}


def _full_cpu_worker(job):
    """One host process = one slice of instances through vehicle + IMU + arm (the reference keeps its
    IMU / arm objects in static storage, so parallelism is across processes, one per core)."""
    kind, n, first, ticks, slow, seg_len, seed = job
    import oracle_lib as ol
    from roboken_fmskf_robot_controller_b200 import layout, streams

    key = (n, first, ticks, slow, seg_len, seed)
    if key not in _FULL_CACHE:
        n_seg, n_slow = (ticks + seg_len - 1) // seg_len, (ticks + slow - 1) // slow
        cmd = streams.vehicle_commands_v2(n, n_seg, seed, first)
        regs, have = streams.imu_samples_v2(n, n_slow + 1, seed=seed, first=first, drop_every=64)
        seq = layout.aos_to_soa(streams.arm_sequences_v2(n, seed=seed, first=first, seq_id=1, max_len=32))
        _FULL_CACHE.clear()
        _FULL_CACHE[key] = (cmd, regs, have, seq)
    cmd, regs, have, seq = _FULL_CACHE[key]
    v = np.zeros(layout.VS_WORDS * n, dtype=np.uint32)
    i = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    ar = np.zeros(layout.AS_WORDS * n, dtype=np.uint32)
    tb = np.zeros(layout.ACMD_WORDS * n, dtype=np.uint32)
    (ol.imu_port if kind == "port" else ol.imu_ref)(i, n, regs[:1], None, do_init=True)
    t0 = time.perf_counter()
    ol.arm_batch(kind, "init", ar, tb, n)
    ol.arm_batch(kind, "push", ar, tb, n, seq=seq)
    ol.full_tick(kind, n, ticks, slow, cmd, seg_len, regs[1:], have[1:], v, i, ar, tb)
    return time.perf_counter() - t0


class CpuArmFull:
    def __init__(self, a):
        import concurrent.futures as cf
        import multiprocessing as mp

        import oracle_lib as ol

        self.a = a
        self.threads = host_threads()
        have = all(os.path.exists(os.path.join(ol.ORACLE, "_ref", f)) for f in ("libref_vdt.so", "libref_imu.so", "libref_arm.so"))
        self.kind = "reference" if have else "port"
        self.pool = cf.ProcessPoolExecutor(max_workers=self.threads, mp_context=mp.get_context("fork"))

    def _run(self, n):
        """n instances split over the worker processes; wall time of the whole pass."""
        a, per = self.a, max(1, n // self.threads)
        jobs = [("ref" if self.kind == "reference" else "port", per, w * per, a.ticks, a.slow_period, a.seg_len, 0x5EED)
                for w in range(self.threads)]
        t0 = time.perf_counter()
        list(self.pool.map(_full_cpu_worker, jobs))
        return time.perf_counter() - t0

    def calibrate(self, step_budget_s):
        n0 = 8 * self.threads
        self._run(n0)
        dt = self._run(n0)
        n = int(n0 / dt * step_budget_s)
        n = max(self.threads * 4, min(n, self.a.total))
        return (n // self.threads) * self.threads

    def sample_desc(self, n):
        return (f"{n} of {self.a.total} robots x {self.a.ticks} vehicle ticks (+ IMU and arm every {self.a.slow_period}) per step, "
                f"same seeded streams, {self.threads} host processes over instances (the reference keeps IMU/arm objects static)")

    def close(self):
        self.pool.shutdown()


def make_cpu_arm(a):
    return CpuArmFull(a) if a.workload == "full" else CpuArm(a)


def run_reference(a):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    arm = make_cpu_arm(a)
    budget = min(2.0, 90.0 / max(1, a.steps + a.warmup))
    n = arm.calibrate(budget)
    for _ in range(a.warmup):
        arm._run(n)
    t = 0.0
    for _ in range(a.steps):
        t += arm._run(n)
    value = n * a.ticks * a.steps / t
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * t / a.steps, "higher_is_better": True, "scaling": "strong" if a.workload == "full" else "weak",
        "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "instances_per_step": n, "ticks_per_launch": a.ticks},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.threads, "kind": arm.kind, "sample": arm.sample_desc(n)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------
# clocks sampler (NVML) -- runs DURING the timed regions
# ------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {
        0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
        0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
        0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting",
    }

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self.ok = [], set(), None, False
        self._stop = threading.Event()
        self._active = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False
        self.th = threading.Thread(target=self._loop, daemon=True)
        if self.ok:
            self.th.start()

    def _loop(self):
        while not self._stop.is_set():
            if self._active.is_set():
                try:
                    self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                    r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    for bit, name in self.REASONS.items():
                        if r & bit and name != "gpu_idle":
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.02)

    def start(self):
        self._active.set()

    def pause(self):
        self._active.clear()

    def result(self):
        self._stop.set()
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"], "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------
# roofline denominators
# ------------------------------------------------------------------------------------------
def fp32_probes(lib, local_rank, dev, stream):
    """FP32 peaks measured live (MEASURED_PEAKS.json has no FP32 entry): dense FFMA and dense
    non-fused FMUL/FADD issue throughput, TFLOP/s, best of 3 after one warm-up."""
    import torch

    from roboken_fmskf_robot_controller_b200 import _cabi

    sm, khz = C.c_int(), C.c_int()
    _cabi.check(lib.rk_device_info(local_rank, C.byref(sm), C.byref(khz), None))
    probe_out = torch.zeros(4, dtype=torch.float32, device=dev)

    def probe(fused):
        fl, best = C.c_double(), 0.0
        for it in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            _cabi.check(lib.rk_probe_fp32(fused, sm.value * 32, 4096, probe_out.data_ptr(), C.byref(fl), C.c_void_p(stream.cuda_stream)))
            e1.record(stream)
            torch.cuda.synchronize()
            if it:
                best = max(best, fl.value / (e0.elapsed_time(e1) * 1e-3))
        return best / 1e12

    return probe(1), probe(0), sm.value


def hbm_peak_measured():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        try:
            return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
# helpers shared by the GPU arms
# ------------------------------------------------------------------------------------------
def timed_launches(fn, stream, reps, warm=2):
    """Average duration (ms) of fn() over `reps` back-to-back calls on `stream`, CUDA events on that stream."""
    import torch

    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def all_ranks_ok(ok, dev):
    """True iff `ok` on every rank."""
    import torch
    import torch.distributed as dist

    if not dist.is_initialized():
        return bool(ok)
    t = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item() > 0.5)


def oracle_kind():
    import oracle_lib as ol

    have = all(os.path.exists(os.path.join(ol.ORACLE, "_ref", f)) for f in ("libref_vdt.so", "libref_imu.so", "libref_arm.so"))
    return ("ref", "the reference's own sources compiled for x86 (oracle/_ref)") if have else ("port", "the plain-C port (oracle/)")


def vehicle_module(a, lib, dev, stream, peaks):
    """BASELINE configs[1] on this GPU: 2^20 vehicles x 1000 fused ticks, device-resident inputs; the dominant kernel alone."""
    import torch

    from roboken_fmskf_robot_controller_b200 import _cabi
    from roboken_fmskf_robot_controller_b200.devstreams import DeviceStreams
    from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch

    n, T = a.instances, a.ticks
    n_seg, n_yaw = (T + a.seg_len - 1) // a.seg_len, (T + a.yaw_period - 1) // a.yaw_period
    ds = DeviceStreams(dev, seed=0x5EED, first=0)
    cmd = ds.vehicle_commands(torch.empty((n_seg, n, 4), dtype=torch.int32, device=dev))
    yaw = ds.vehicle_yaw_reg(torch.empty((n_yaw, n), dtype=torch.int16, device=dev))
    vb = VehicleBatch(n, dev)
    args = vb.make_args(T, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=cmd, seg_len=a.seg_len, yaw=yaw, yaw_period=a.yaw_period)
    ms = timed_launches(lambda: vb.rollout_args(args, stream=stream), stream, 5)
    ffma, issue = peaks
    tf = FLOP_PER_TICK * n * T / (ms * 1e-3) / 1e12
    return {"workload": f"configs[1]: {n} vehicles x {T} fused 1 kHz ticks, closed loop through the integer plant, Yaw-register input",
            "kernel": "rk::vdt_rollout_fast_kernel", "value": n * T / (ms * 1e-3), "unit": UNIT, "ms_per_launch": ms,
            "roofline": {"bound": "fp32", "achieved": tf, "peak": ffma, "unit": "TFLOP/s", "frac": tf / ffma,
                         "frac_of_nonfused_issue_peak": tf / issue, "algorithmic_flop_per_tick": FLOP_PER_TICK}}


def imu_module(a, dev, stream, hbm):
    """BASELINE configs[2]: 2^20 IMUs x 64 fused updates with the full Data page written back per update."""
    import torch

    from roboken_fmskf_robot_controller_b200.devstreams import DeviceStreams
    from roboken_fmskf_robot_controller_b200.imu import ImuBatch

    n, K = a.instances, 64
    ds = DeviceStreams(dev, seed=3, first=0)
    regs, have = ds.imu_samples(torch.empty((K, 2, n, 8), dtype=torch.int16, device=dev), torch.empty((K, n), dtype=torch.uint8, device=dev))
    ib = ImuBatch(n, dev)
    ib.update(regs[:1].contiguous(), None, None, do_init=True)
    out = torch.empty((K, 4, n, 4), dtype=torch.float32, device=dev)
    ms = timed_launches(lambda: ib.update(regs, have, out), stream, 5)
    nbytes = n * (K * (32 + 1 + 64) + 2 * 96)
    peak, src = hbm
    return {"workload": f"configs[2]: {n} WT901 IMUs x {K} fused updates, Data page written per update", "kernel": "rk::imt_update_kernel",
            "value": n * K / (ms * 1e-3), "unit": "IMU updates/s", "ms_per_launch": ms,
            "roofline": {"bound": "hbm", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": nbytes / (ms * 1e-3) / 1e9 / peak, "peak_source": src, "algorithmic_bytes_per_update": 97}}


def arm_module(a, dev, stream):
    """BASELINE configs[3]: 2^20 arms x 1000 fused 100 Hz ticks, one PosCmdSeq each."""
    import torch

    from roboken_fmskf_robot_controller_b200 import layout
    from roboken_fmskf_robot_controller_b200.arm import ArmBatch
    from roboken_fmskf_robot_controller_b200.devstreams import DeviceStreams

    n, K = a.instances, 1000
    ds = DeviceStreams(dev, seed=0xC4, first=0, arm_seq_id=9)
    seq = ds.arm_sequences(torch.empty(layout.ACMD_SLOT_WORDS * n, dtype=torch.int32, device=dev))
    ab = ArmBatch(n, dev)

    def setup():
        ab.mode_init(stream=stream)
        ab.push_cmdseq(seq, stream=stream)

    def full():
        setup()
        ab.update(K, stream=stream)

    ms = timed_launches(full, stream, 5) - timed_launches(setup, stream, 5)
    return {"workload": f"configs[3]: {n} 5-axis arms x {K} fused 100 Hz ticks, one PosCmdSeq each", "kernel": "rk::adt_update_kernel",
            "value": n * K / (ms * 1e-3), "unit": "arm ticks/s", "ms_per_launch": ms,
            "roofline": {"bound": "issue", "achieved": 46 * n * K / (ms * 1e-3) / 1e12, "unit": "TFLOP/s", "algorithmic_flop_per_tick": 46}}


# ------------------------------------------------------------------------------------------
# GPU arm, workload "vehicle" (BASELINE configs[1], weak scaling)
# ------------------------------------------------------------------------------------------
def run_ours(a):
    import torch

    import roboken_fmskf_robot_controller_b200 as rk
    from roboken_fmskf_robot_controller_b200 import _cabi, layout, sharding, streams
    from roboken_fmskf_robot_controller_b200.devstreams import DeviceStreams
    from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch

    lib = rk.load()  # raises if the CUDA library is not built: no fallback
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU fallback)")
    rank, local_rank, world = sharding.init("nccl")
    assert world == a.gpus, f"--gpus {a.gpus} but WORLD_SIZE={world} (launch with torchrun for N>1)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _cabi.check(lib.rk_set_device(local_rank))
    if a.occupancy:
        _cabi.check(lib.rk_set_option(_cabi.RK_OPT_FAST_OCCUPANCY, a.occupancy))
    if a.packed >= 0:
        _cabi.check(lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, a.packed))
    if a.ffsat >= 0:
        _cabi.check(lib.rk_set_option(_cabi.RK_OPT_FAST_FFSAT, a.ffsat))
    n, K, W, T = a.instances, a.steps, a.warmup, a.ticks
    first = rank * n  # contiguous slice of the global instance index space
    n_seg = (T + a.seg_len - 1) // a.seg_len
    n_yaw = (T + a.yaw_period - 1) // a.yaw_period
    stream = torch.cuda.current_stream(dev)
    clocks = ClockSampler(local_rank)

    # ---- synthetic inputs, generated on the device from a 48-byte descriptor ----------------
    seed = 0x5EED
    ds = DeviceStreams(dev, seed=seed, first=first)
    cmd_d = ds.vehicle_commands(torch.empty((n_seg, n, 4), dtype=torch.int32, device=dev))
    yaw_d = ds.vehicle_yaw_reg(torch.empty((n_yaw, n), dtype=torch.int16, device=dev))
    goal_d = torch.zeros((n, 2), dtype=torch.float32, device=dev)
    cost_d = torch.zeros(n, dtype=torch.float32, device=dev)
    vb = VehicleBatch(n, dev)
    args = vb.make_args(T, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=cmd_d, seg_len=a.seg_len, yaw=yaw_d,
                        yaw_period=a.yaw_period, goal=goal_d, cost=cost_d)

    # ---- parity spot check of the exact bench launch (first pass, power-on state), every rank -----
    vb.rollout_args(args)
    torch.cuda.synchronize()
    import oracle_lib as ol

    idx = np.unique(np.concatenate([[0, n - 1], np.random.default_rng(rank).integers(0, n, 62)]))
    gidx = idx.astype(np.uint64) + np.uint64(first)
    ro = ol.HostRollout(len(idx), T, _cabi.RK_SENSOR_PLANT, streams.vehicle_commands_v2(0, n_seg, seed, inst=gidx), a.seg_len,
                        streams.vehicle_yaw_reg_v2(0, n_yaw, seed, inst=gidx), a.yaw_period)
    exp = np.zeros(layout.VS_WORDS * len(idx), dtype=np.uint32)
    kind, kind_desc = oracle_kind()
    (ol.run_ref if kind == "ref" else ol.run_port)(exp, len(idx), ro, nthreads=min(8, host_threads()))
    got = layout.soa_to_aos(vb.state.cpu().numpy().view(np.uint32), n, layout.VS_WORDS)[idx]
    same = all_ranks_ok(np.array_equal(got, layout.soa_to_aos(exp, len(idx), layout.VS_WORDS)), dev)
    spot = f"{len(idx)} sampled instances x {T} ticks on each of {world} rank(s) {'bit-exact' if same else 'MISMATCH'} vs {kind_desc}"
    if not same:
        raise SystemExit("bench parity spot check failed: " + spot)

    # ---- value: inputs resident in HBM -----------------------------------------------------
    for _ in range(max(W - 1, 0)):
        vb.rollout_args(args)
    torch.cuda.synchronize()
    sharding.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clocks.start()
    ev0.record(stream)
    for _ in range(K):
        vb.rollout_args(args)
    ev1.record(stream)
    torch.cuda.synchronize()
    clocks.pause()
    sharding.barrier()
    ms_local = ev0.elapsed_time(ev1)
    ms = sharding.max_over_ranks(ms_local, dev)
    value = world * n * T * K / (ms * 1e-3)
    launches = K
    if a.dump_outputs:  # before the e2e passes below reset and rerun the vehicles
        dump_outputs(a.dump_outputs, n, first, rank, world, [(n, cost_d, {"vehicle_state": (vb.state, layout.VS_WORDS)})])

    ffma_tflops, issue_tflops, sm_count = fp32_probes(lib, local_rank, dev, stream)
    hbm_peak, hbm_src = hbm_peak_measured()
    launch_s = ms_local * 1e-3 / K
    achieved_tflops = FLOP_PER_TICK * n * T / launch_s / 1e12
    alg_bytes = n * (2 * STATE_BYTES + n_seg * 16 + n_yaw * 2 + 8 + 4)  # state ld+st, cmd, yaw, goal, cost
    roofline = {
        "bound": "fp32",
        "achieved": achieved_tflops, "peak": ffma_tflops, "unit": "TFLOP/s", "frac": achieved_tflops / ffma_tflops,
        "peak_source": "rk_probe_fp32 FFMA chains, measured live in this run (no FP32 entry in MEASURED_PEAKS.json)",
        "nonfused_issue_peak": issue_tflops,
        "frac_of_nonfused_issue_peak": achieved_tflops / issue_tflops,
        "algorithmic_flop_per_tick": FLOP_PER_TICK,
        "kernel": "rk::vdt_rollout_fast_kernel",
        "launch_ms": launch_s * 1e3,
        "traffic": traffic_note("vdt_rollout_plant_bytes_per_launch"),
        "hbm": {"achieved": alg_bytes / launch_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": alg_bytes / launch_s / 1e9 / hbm_peak, "peak_source": hbm_src,
                "algorithmic_bytes_per_launch": alg_bytes},
        "sm_count": sm_count,
    }

    # ---- e2e: descriptor in (pinned host -> device), tables expanded on the device, costs out ----
    e2e = None
    if not a.no_e2e:
        gen_s, comp_s, back_s = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        bufs = []
        for b in range(2):
            c, y = torch.empty_like(cmd_d), torch.empty_like(yaw_d)
            co = torch.zeros(n, dtype=torch.float32, device=dev)
            bufs.append(dict(cmd=c, yaw=y, cost=co, cost_h=torch.empty(n, dtype=torch.float32).pin_memory(),
                             ds=DeviceStreams(dev, seed=seed, first=first),
                             args=vb.make_args(T, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=c, seg_len=a.seg_len, yaw=y,
                                               yaw_period=a.yaw_period, goal=goal_d, cost=co, reset_state=True),
                             up=torch.cuda.Event(), done=torch.cuda.Event(), down=torch.cuda.Event()))
        h2d, d2h = DeviceStreams.NBYTES, n * 4

        def e2e_pass(s):
            b = bufs[s % 2]
            with torch.cuda.stream(gen_s):
                gen_s.wait_event(b["done"])  # buffer free again (previous use computed)
                b["ds"].upload(gen_s)
                b["ds"].vehicle_commands(b["cmd"], gen_s)
                b["ds"].vehicle_yaw_reg(b["yaw"], gen_s)
                b["up"].record(gen_s)
            with torch.cuda.stream(comp_s):
                comp_s.wait_event(b["up"])
                comp_s.wait_event(b["down"])  # cost buffer drained
                vb.rollout_args(b["args"], stream=comp_s)  # reset_state: every rollout starts from the power-on state
                b["done"].record(comp_s)
            with torch.cuda.stream(back_s):
                back_s.wait_event(b["done"])
                b["cost_h"].copy_(b["cost"], non_blocking=True)
                b["down"].record(back_s)

        for s in range(max(W, 2)):
            e2e_pass(s)
        torch.cuda.synchronize()
        sharding.barrier()
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks.start()
        t0e.record(stream)
        for st_ in (gen_s, back_s, comp_s):
            st_.wait_stream(stream)
        for s in range(K):
            e2e_pass(s)
        for st_ in (gen_s, back_s, comp_s):
            stream.wait_stream(st_)
        t1e.record(stream)
        torch.cuda.synchronize()
        clocks.pause()
        sharding.barrier()
        ms_e = sharding.max_over_ranks(t0e.elapsed_time(t1e), dev)
        e2e = {"value": world * n * T * K / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": ms_e / K,
               "path": "per step: 48-byte stream descriptor pinned host -> device, rk_stream_vehicle_commands + "
                       "rk_stream_vehicle_yaw_reg expand it on the device, state reset to power-on, rk_vdt_rollout() via "
                       "ctypes, cost vector D2H; double-buffered on three streams"}

    # ---- optional NCCL gather of the summary costs (outside the timed regions) --------------
    gather_ms = None
    if world > 1:
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sharding.gather_costs(cost_d)
        torch.cuda.synchronize()
        g0.record(stream)
        allc = sharding.gather_costs(cost_d)
        g1.record(stream)
        torch.cuda.synchronize()
        gather_ms = sharding.max_over_ranks(g0.elapsed_time(g1), dev)
        assert allc.numel() == world * n

    clk = clocks.result()

    # ---- CPU baseline (rank 0, N=1 only) ------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        arm = CpuArm(a)
        nc = arm.calibrate(a.cpu_seconds / 3.0)
        t = min(arm._run(nc) for _ in range(2))
        cpu = {"value": nc * T / t, "unit": UNIT, "cores": arm.threads, "kind": arm.kind, "sample": arm.sample_desc(nc)}
        n1 = max(64, nc // (4 * arm.threads))  # the single-core figure SURVEY 8d asks for, on a quarter of one thread's share
        arm._run(n1, threads=1)
        cpu["single_core_value"] = n1 * T / arm._run(n1, threads=1)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(a), "instances_per_gpu": n, "ticks_per_launch": T,
                       "l2": f"inputs larger than L2: {n * STATE_BYTES >> 20} MiB state + "
                             f"{(cmd_d.numel() * 4 + yaw_d.numel() * 2) >> 20} MiB tables per pass vs 126 MB L2",
                       "parity_spot_check": spot},
            "clocks": clk, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
        }
        if gather_ms is not None:
            line["cost_gather_ms"] = gather_ms
        emit(line)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


def traffic_note(key):
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(path)).get(key)
    except Exception:
        return None


# ------------------------------------------------------------------------------------------
# GPU arm, workload "full" (BASELINE configs[4], the default)
# ------------------------------------------------------------------------------------------
FLOP_PER_FULL_STEP = 183 + 1 + (55 + 46) / 10.0  # SURVEY.md 8d: vehicle + deg2rad + (IMU + arm) at 1/10 rate
FULL_BYTES_PER_ROBOT = 4  # filled in run_ours_full


def run_ours_full(a):
    import torch

    import roboken_fmskf_robot_controller_b200 as rk
    from roboken_fmskf_robot_controller_b200 import _cabi, layout, sharding, streams
    from roboken_fmskf_robot_controller_b200.devstreams import DeviceStreams
    from roboken_fmskf_robot_controller_b200.robot import RobotBatch

    lib = rk.load()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU fallback)")
    rank, local_rank, world = sharding.init("nccl")
    assert world == a.gpus, f"--gpus {a.gpus} but WORLD_SIZE={world} (launch with torchrun for N>1)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _cabi.check(lib.rk_set_device(local_rank))
    if a.occupancy:
        _cabi.check(lib.rk_set_option(_cabi.RK_OPT_FAST_OCCUPANCY, a.occupancy))
    if a.side_ctas >= 0:
        _cabi.check(lib.rk_set_option(_cabi.RK_OPT_TICK_SIDE_CTAS, a.side_ctas))
    if a.ffsat >= 0:
        _cabi.check(lib.rk_set_option(_cabi.RK_OPT_FAST_FFSAT, a.ffsat))
    K, W, T, slow = a.steps, a.warmup, a.ticks, a.slow_period
    lo, hi = sharding.shard_range(a.total, rank, world)
    n_rank = hi - lo
    n = min(a.chunk, n_rank)
    assert n_rank % n == 0 and a.total % world == 0, "--total / --gpus must be a multiple of --chunk"
    n_chunks = n_rank // n
    n_seg, n_slow = (T + a.seg_len - 1) // a.seg_len, (T + slow - 1) // slow
    stream = torch.cuda.current_stream(dev)
    clocks = ClockSampler(local_rank)
    seed = 0x5EED

    # ---- synthetic inputs: every chunk's tables expanded on the device from its 48-byte descriptor; resident in HBM
    # for the `value` region (distinct per chunk when they fit, else one set replayed by every chunk) ----------------
    per_robot_in = n_seg * 16 + n_slow * (33 if a.no_yaw_column else 35) + layout.ACMD_SLOT_WORDS * 4
    free_b, _ = torch.cuda.mem_get_info(dev)
    distinct = n_chunks * n * (per_robot_in + 4 * (layout.VS_WORDS + layout.IS_WORDS + layout.AS_WORDS)) + 4 * n * (per_robot_in + 4 * layout.ACMD_WORDS) < 0.85 * free_b

    def alloc_tables():
        return dict(cmd=torch.empty((n_seg, n, 4), dtype=torch.int32, device=dev),
                    regs=torch.empty((n_slow, 2, n, 8), dtype=torch.int16, device=dev),
                    have=torch.empty((n_slow, n), dtype=torch.uint8, device=dev),
                    yawc=None if a.no_yaw_column else torch.empty((n_slow, n), dtype=torch.int16, device=dev),
                    seq=torch.empty(layout.ACMD_SLOT_WORDS * n, dtype=torch.int32, device=dev))

    def generate(ds, tb, st=None):
        ds.vehicle_commands(tb["cmd"], st)
        ds.imu_samples(tb["regs"], tb["have"], st, yaw_reg=tb["yawc"])  # + the Yaw register as a 2-byte column for the vehicle
        ds.arm_sequences(tb["seq"], st)

    def chunk_desc(c):
        return DeviceStreams(dev, seed=seed, first=lo + c * n, first_update=1, arm_seq_id=1)

    goal_d = torch.zeros((n, 2), dtype=torch.float32, device=dev)
    lanes = max(1, min(a.lanes, 4))
    lane_s = [torch.cuda.Stream(dev) for _ in range(lanes)]
    yaws = [torch.zeros(n, dtype=torch.float32, device=dev) for _ in range(lanes)]
    rings = [torch.zeros(layout.ACMD_WORDS * n, dtype=torch.int32, device=dev) for _ in range(lanes)]
    tables, chunks = [], []
    boot = torch.empty((1, 2, n, 8), dtype=torch.int16, device=dev)
    for c in range(n_chunks):
        ds = chunk_desc(c)
        if distinct or c == 0:
            tb = alloc_tables()
            generate(ds, tb)
            tables.append(tb)
        tb = tables[c if distinct else 0]
        rb = RobotBatch(n, dev, arm_cmdtab=rings[c % lanes])
        DeviceStreams(dev, seed=seed, first=lo + c * n, first_update=0).imu_samples(boot, None)
        rb.imu.update(boot, None, None, do_init=True)  # IMU_IF_WT901C::init() at boot consumes sample 0
        cost = torch.zeros(n, dtype=torch.float32, device=dev)
        args = rb.make_args(T, slow, cmd=tb["cmd"], seg_len=a.seg_len, regs=tb["regs"], have_quat=tb["have"], yaw_reg=tb["yawc"], yaw=yaws[c % lanes],
                            goal=goal_d, cost=cost)
        chunks.append(dict(rb=rb, cost=cost, args=args, tb=tb, ds=ds))
    torch.cuda.synchronize()

    def fork():
        for ls in lane_s:
            ls.wait_stream(stream)

    def join():
        for ls in lane_s:
            stream.wait_stream(ls)

    def one_pass(fork_join=True):
        """All chunks of this rank: arm bring-up + one command sequence pushed, then the fused tick.  The lanes fork from
        and join the current stream, so events recorded on it bracket the work; inside a timed region of several passes
        only the first forks and the last joins (a chunk always runs on the same lane, which orders its passes)."""
        if fork_join:
            fork()
        for c, ch in enumerate(chunks):
            ls = lane_s[c % lanes]
            ch["rb"].arm.mode_init(stream=ls)
            ch["rb"].arm.push_cmdseq(ch["tb"]["seq"], stream=ls)
            ch["rb"].rollout_args(ch["args"], stream=ls)
        if fork_join:
            join()

    # ---- parity spot check of the exact bench launch (first pass), on EVERY rank: robots sampled from the first,
    # a middle and the last chunk of the rank against the oracle on host-generated copies of their streams ----------
    one_pass()
    torch.cuda.synchronize()
    import oracle_lib as ol

    kind, kind_desc = oracle_kind()
    same, m_total = True, 0
    for c in sorted({0, n_chunks // 2, n_chunks - 1}):
        rbc = chunks[c]["rb"]
        idx = np.unique(np.concatenate([[0, n - 1], np.random.default_rng(1000 * rank + c).integers(0, n, 30)]))
        gidx = idx.astype(np.uint64) + np.uint64(lo + (c if distinct else 0) * n)
        m = len(idx)
        m_total += m
        cmd_np = streams.vehicle_commands_v2(0, n_seg, seed, inst=gidx)
        regs_np, have_np = streams.imu_samples_v2(0, n_slow + 1, seed, inst=gidx)
        if not distinct:  # boot samples are per chunk even when the tables are shared
            regs_np[:1] = streams.imu_samples_v2(0, 1, seed, inst=idx.astype(np.uint64) + np.uint64(lo + c * n))[0]
        seq_np = streams.arm_sequences_v2(0, seed, inst=gidx, seq_id=1)
        v, i_, ar, tb_ = (np.zeros(w * m, dtype=np.uint32) for w in (layout.VS_WORDS, layout.IS_WORDS, layout.AS_WORDS, layout.ACMD_WORDS))
        (ol.imu_ref if kind == "ref" else ol.imu_port)(i_, m, regs_np[:1], None, do_init=True)
        ol.arm_batch(kind, "init", ar, tb_, m)
        ol.arm_batch(kind, "push", ar, tb_, m, seq=layout.aos_to_soa(seq_np))
        _, _, _, cost_np = ol.full_tick(kind, m, T, slow, cmd_np, a.seg_len, np.ascontiguousarray(regs_np[1:]), np.ascontiguousarray(have_np[1:]),
                                        v, i_, ar, tb_, goal=np.zeros((m, 2), dtype=np.float32), nthreads=min(8, host_threads()))
        for got, exp, words in ((rbc.vehicle.state, v, layout.VS_WORDS), (rbc.imu.state, i_, layout.IS_WORDS), (rbc.arm.state, ar, layout.AS_WORDS)):
            g = layout.soa_to_aos(got.cpu().numpy().view(np.uint32), n, words)[idx]
            same &= np.array_equal(g, layout.soa_to_aos(exp, m, words))
        cost_np = np.asarray(cost_np, dtype=np.float32)
        same &= np.array_equal(chunks[c]["cost"].cpu().numpy()[idx].view(np.uint32), cost_np.view(np.uint32))
        if c == n_chunks - 1:
            # What the e2e path must hand back for this chunk: every e2e rollout starts from the power-on vehicle and a freshly
            # initialised arm, while the IMU carries on from the end of the previous rollout over the same samples (its last
            # yaw is what the vehicle holds while the first samples of the table carry no quaternion frame).
            v2, ar2, tb2 = (np.zeros(w * m, dtype=np.uint32) for w in (layout.VS_WORDS, layout.AS_WORDS, layout.ACMD_WORDS))
            i2 = i_.copy()
            ol.arm_batch(kind, "init", ar2, tb2, m)
            ol.arm_batch(kind, "push", ar2, tb2, m, seq=layout.aos_to_soa(seq_np))
            _, _, _, cost2 = ol.full_tick(kind, m, T, slow, cmd_np, a.seg_len, np.ascontiguousarray(regs_np[1:]), np.ascontiguousarray(have_np[1:]),
                                          v2, i2, ar2, tb2, goal=np.zeros((m, 2), dtype=np.float32), nthreads=min(8, host_threads()))
            spot_last = (idx, np.asarray(cost2, dtype=np.float32))
    same = all_ranks_ok(same, dev)
    spot = (f"{m_total} sampled robots x {T} ticks (vehicle + IMU + arm state, rollout cost) on each of {world} rank(s) "
            f"{'bit-exact' if same else 'MISMATCH'} vs {kind_desc}")
    if not same:
        raise SystemExit("bench parity spot check failed: " + spot)

    # ---- value: inputs resident in HBM -----------------------------------------------------------
    for _ in range(max(W - 1, 0)):
        one_pass()
    torch.cuda.synchronize()
    sharding.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clocks.start()
    ev0.record(stream)
    fork()
    for _ in range(K):
        one_pass(fork_join=False)
    join()
    ev1.record(stream)
    torch.cuda.synchronize()
    clocks.pause()
    sharding.barrier()
    ms_local = ev0.elapsed_time(ev1)
    ms = sharding.max_over_ranks(ms_local, dev)
    value = a.total * T * K / (ms * 1e-3)
    launches = K * n_chunks * 6  # mode_init, push, yaw snapshot, IMU update, arm update, vehicle rollout
    if a.dump_outputs:  # before the roofline and e2e passes below run chunk 0 again
        dump_outputs(a.dump_outputs, n_rank, lo, rank, world,
                     [(n, ch["cost"], {"vehicle_state": (ch["rb"].vehicle.state, layout.VS_WORDS),
                                       "imu_state": (ch["rb"].imu.state, layout.IS_WORDS),
                                       "arm_state": (ch["rb"].arm.state, layout.AS_WORDS)}) for ch in chunks])

    # ---- roofline of the dominant kernel: its share of the timed region, and timed alone -----------------------------
    ffma_tflops, issue_tflops, sm_count = fp32_probes(lib, local_rank, dev, stream)
    hbm = hbm_peak_measured()
    step_s = ms_local * 1e-3 / K
    chunk_s = step_s / n_chunks  # one chunk's slot of the timed region: its vehicle rollout with the IMU / arm kernels in its shadow
    rb0 = chunks[0]["rb"]
    vargs = rb0.vehicle.make_args(T, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=chunks[0]["tb"]["cmd"], seg_len=a.seg_len, goal=goal_d,
                                  cost=chunks[0]["cost"])
    vargs.d_imu_regs, vargs.d_imu_have_quat = chunks[0]["tb"]["regs"].data_ptr(), chunks[0]["tb"]["have"].data_ptr()
    vargs.d_imu_yaw0_deg, vargs.n_yaw, vargs.yaw_period = yaws[0].data_ptr(), n_slow, slow
    alone_ms = timed_launches(lambda: rb0.vehicle.rollout_args(vargs, stream=stream), stream, 5)
    achieved = FLOP_PER_TICK * n * T / chunk_s / 1e12
    step_bytes = n_rank * (2 * 4 * (layout.VS_WORDS + layout.IS_WORDS + layout.AS_WORDS) + n_seg * 16 + n_slow * (33 + 16 + 1) +
                           2 * 4 * layout.ACMD_SLOT_WORDS + 8 + 4 + 8)
    roofline = {
        "bound": "fp32", "achieved": achieved, "peak": ffma_tflops, "unit": "TFLOP/s", "frac": achieved / ffma_tflops,
        "peak_source": "rk_probe_fp32 FFMA chains, measured live in this run (no FP32 entry in MEASURED_PEAKS.json)",
        "nonfused_issue_peak": issue_tflops, "frac_of_nonfused_issue_peak": achieved / issue_tflops,
        "algorithmic_flop_per_tick": FLOP_PER_TICK,
        "kernel": "rk::vdt_rollout_fast_kernel (dominant kernel)",
        "launch_ms": chunk_s * 1e3,
        "launch_ms_note": "timed region / vehicle launches in it: the kernel's slot including the IMU, arm and ring-push kernels that "
                          "run in its shadow (CUDA events on the launching streams' parent)",
        "launch_ms_alone": alone_ms, "frac_alone": FLOP_PER_TICK * n * T / (alone_ms * 1e-3) / 1e12 / ffma_tflops,
        "traffic": traffic_note("vdt_rollout_imu_regs_bytes_per_launch" if a.no_yaw_column else "vdt_rollout_yaw_column_bytes_per_launch"),
        "step": {"algorithmic_flop_per_robot_step": FLOP_PER_FULL_STEP,
                 "achieved_tflops": FLOP_PER_FULL_STEP * n_rank * T / step_s / 1e12,
                 "frac_of_ffma_peak": FLOP_PER_FULL_STEP * n_rank * T / step_s / 1e12 / ffma_tflops,
                 "algorithmic_bytes": step_bytes, "hbm_gbs": step_bytes / step_s / 1e9,
                 "hbm_frac": step_bytes / step_s / 1e9 / hbm[0], "hbm_peak_source": hbm[1]},
        "sm_count": sm_count,
    }

    # ---- e2e: per chunk a 48-byte descriptor in, tables expanded on the device, costs out, through rk_tick_rollout ----
    e2e = None
    if not a.no_e2e:
        gen_s, back_s = torch.cuda.Stream(dev, priority=-1), torch.cuda.Stream(dev)
        _cabi.check(lib.rk_set_option(_cabi.RK_OPT_STREAM_CTAS, a.gen_ctas))  # the generators trickle beside the rollout
        # table sets: one being generated, one per compute lane in flight
        NB = lanes + 1
        skip = set(x for x in a.e2e_skip.split(",") if x)
        fused = not (a.e2e_tables or a.no_yaw_column)  # the IMU update draws its samples from the descriptor in registers
        bufs = []
        for b in range(NB):
            d = alloc_tables()
            d.update(cost=torch.zeros(n, dtype=torch.float32, device=dev), cost_h=torch.empty(n, dtype=torch.float32).pin_memory(),
                     up=torch.cuda.Event(), done=torch.cuda.Event(), down=torch.cuda.Event())
            bufs.append(d)
        h2d, d2h = n_chunks * DeviceStreams.NBYTES, n_chunks * n * 4
        argcache = {}

        def e2e_pass(s):
            """Like one_pass, with every chunk's tables expanded on the device first (generation stream, beside the rollouts)
            and its cost vector read back (copy stream)."""
            for c, ch in enumerate(chunks):
                g = s * n_chunks + c
                b = bufs[g % NB]
                rb, ls = ch["rb"], lane_s[c % lanes]
                with torch.cuda.stream(gen_s):
                    gen_s.wait_event(b["done"])  # the rollout that last used this table set has finished
                    ch["ds"].upload(gen_s)
                    if "gen" not in skip or s < 0:
                        if fused:  # commands, the two IMU columns the vehicle reads, arm waypoints; the IMU samples are drawn in the update
                            ch["ds"].vehicle_commands(b["cmd"], gen_s)
                            ch["ds"].imu_columns(b["yawc"], b["have"], gen_s)
                            ch["ds"].arm_sequences(b["seq"], gen_s)
                        else:
                            generate(ch["ds"], b, gen_s)
                    b["up"].record(gen_s)
                with torch.cuda.stream(ls):
                    ls.wait_event(b["up"])
                    ls.wait_event(b["down"])  # the cost buffer has been drained
                    rb.arm.mode_init(stream=ls)
                    rb.arm.push_cmdseq(b["seq"], stream=ls)
                    key = (c, g % NB)
                    if key not in argcache:  # reset_vehicle: every rollout starts from the power-on vehicle
                        argcache[key] = rb.make_args(T, slow, cmd=b["cmd"], seg_len=a.seg_len, regs=None if fused else b["regs"],
                                                     imu_desc=ch["ds"] if fused else None, have_quat=b["have"], yaw_reg=b["yawc"],
                                                     yaw=yaws[c % lanes], goal=goal_d, cost=b["cost"], reset_vehicle="reset" not in skip)
                    rb.rollout_args(argcache[key], stream=ls)
                    b["done"].record(ls)
                with torch.cuda.stream(back_s):
                    back_s.wait_event(b["done"])
                    if "d2h" not in skip:
                        b["cost_h"].copy_(b["cost"], non_blocking=True)
                    b["down"].record(back_s)

        e2e_pass(-1)  # (the first pass always generates)
        for s in range(2):
            e2e_pass(s)
        torch.cuda.synchronize()
        sharding.barrier()
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        clocks.start()
        t0e.record(stream)
        for st_ in [gen_s, back_s] + lane_s:
            st_.wait_stream(stream)
        for s in range(K):
            e2e_pass(s)
        for st_ in [gen_s, back_s] + lane_s:
            stream.wait_stream(st_)
        t1e.record(stream)
        torch.cuda.synchronize()
        clocks.pause()
        sharding.barrier()
        ms_e = sharding.max_over_ranks(t0e.elapsed_time(t1e), dev)
        _cabi.check(lib.rk_set_option(_cabi.RK_OPT_STREAM_CTAS, 0))
        # the costs the last e2e rollout copied back == the oracle's for the sampled robots of that chunk
        b_last = bufs[((K - 1) * n_chunks + n_chunks - 1) % NB]
        e2e_same = all_ranks_ok(np.array_equal(b_last["cost_h"].numpy()[spot_last[0]].view(np.uint32), spot_last[1].view(np.uint32)), dev)
        if not e2e_same and not skip:
            raise SystemExit("bench e2e parity check failed: costs returned through the end-to-end path differ from the oracle")
        e2e = {"value": a.total * T * K / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": ms_e / K,
               "path": ("per chunk: 48-byte stream descriptor pinned host -> device; rk_stream_vehicle_commands / rk_stream_imu_samples_yaw / "
                        "rk_stream_arm_sequences expand it on the device into the command table, the two IMU columns the vehicle reads (Yaw "
                        "register, quaternion-frame flag) and the arm-sequence table; the IMU update draws its 100 register snapshots per "
                        "robot from the same descriptor in registers (rk_tick_rollout_t::d_imu_desc: 3.2 KB per robot neither written nor "
                        "read); rk_adt_mode_init + rk_adt_push_cmdseq + rk_tick_rollout (vehicles from power-on) via ctypes; cost vector D2H; "
                        "generation (high-priority stream, capped grid), compute (the lanes of the value path) and D2H overlap") if fused else
                       ("per chunk: 48-byte stream descriptor pinned host -> device; rk_stream_vehicle_commands / rk_stream_imu_samples / "
                        "rk_stream_arm_sequences expand it into the command, IMU-register and arm-sequence tables on the device (4.5 KB per "
                        "robot that never cross PCIe); rk_adt_mode_init + rk_adt_push_cmdseq + rk_tick_rollout (vehicles from power-on) via "
                        "ctypes; cost vector D2H; generation (high-priority stream, capped grid), compute (the lanes of the value path) and D2H overlap"),
               "parity": "costs copied back by the last rollout bit-exact vs the oracle on the sampled robots of that chunk, every rank"}

    # ---- the module configurations (BASELINE configs[1..3]) on this GPU, outside the timed regions ----------------------
    modules = None
    if rank == 0 and not a.no_modules:
        for ch in chunks[1:]:
            ch.clear()  # release the chunk tables before the modules allocate theirs
        del chunks[1:], tables[1:]
        torch.cuda.empty_cache()
        modules = {"vehicle": vehicle_module(a, lib, dev, stream, (ffma_tflops, issue_tflops)), "imu": imu_module(a, dev, stream, hbm),
                   "arm": arm_module(a, dev, stream)}

    clk = clocks.result()
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        arm = CpuArmFull(a)
        nc = arm.calibrate(a.cpu_seconds / 3.0)
        t = min(arm._run(nc) for _ in range(2))
        cpu = {"value": nc * T / t, "unit": UNIT, "cores": arm.threads, "kind": arm.kind, "sample": arm.sample_desc(nc)}
        arm.close()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(a), "robots_total": a.total, "robots_per_gpu": n_rank, "chunk": n, "lanes": lanes, "ticks_per_launch": T,
                       "tables": "distinct per chunk" if distinct else "one chunk's tables replayed by every chunk (HBM budget)",
                       "l2": f"inputs larger than L2: {n * per_robot_in >> 20} MiB tables + {n * 848 >> 20} MiB state per chunk vs 126 MB L2",
                       "parity_spot_check": spot},
            "clocks": clk, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "modules": modules,
        }
        emit(line)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


_JSON_FD = None


def emit(line):
    """The ONE JSON line of the contract, on the process's real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    a = parse()
    # Libraries print to stdout on their own (NCCL's version banner when NCCL_DEBUG is set, for one); keep the real
    # stdout for the JSON line and send everything else to stderr.
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if a.impl == "reference":
        if a.dump_outputs:
            raise SystemExit("--dump-outputs writes what the GPU path computed: use it with --impl ours")
        run_reference(a)
    elif a.workload == "full":
        run_ours_full(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
