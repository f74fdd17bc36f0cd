#!/usr/bin/env python
"""bench.py — scan-to-map registrations/sec (100k-pt scan vs 1M-pt map) on B200, per BASELINE.json.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload headline|c2|c1|c3|c4|c5]
                  [--dump-outputs DIR]

One "step" = one NDT registration (pcl::Registration::align semantics) of a synthetic 64-ring scan (~100k points)
against a 1M-point map, resolution 2.0, DIRECT7, transformation_epsilon 0.01, max 35 iterations, identity guess —
the steady state apps/align.cpp:32-36 calls "10times" (target already set).

 * value     : registrations/s with the scans already resident in HBM (setInputSourceDevice + align per step)
 * e2e       : the same through the public API with HOST buffers: setInputSource(numpy) + align + 4x4 read-back
 * roofline  : the solver kernel's algorithmic bytes (SURVEY.md §8d: per evaluation N_src*16 + N_src*7*8 +
               N_hit*48 + 224) / its CUDA-event duration on the launching stream, vs MEASURED_PEAKS.json hbm_gbs
 * cpu_baseline: the CPU oracle (restatement of the reference's OpenMP path) on the same workload, bounded sample
 * --impl reference: times that CPU path alone (the reference needs PCL/Eigen/FLANN and cannot be built here)
 * --dump-outputs DIR: after the timed steps, what the timed path returned for each of them (poses, iteration counts, ...)
               as DIR/<name>.npy; the inputs are seeded, so two builds run with the same arguments compare output for output
               (to rounding, not bit for bit: the target's voxel moments are summed with f64 atomics in arrival order)
N > 1: one process per GPU (torchrun), each rank registers its own K scans (replicas — a single alignment does not
shard, SURVEY.md §8e) and ONE NCCL all-gather of the K 4x4 poses closes the timed region; value = N*K / max time.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (synth config, resolution, description)
    "headline": ("headline", 2.0, "NDT align, 64-ring scan (~100k pts) vs 1M-pt map, res 2.0, DIRECT7, eps 0.01, max_iter 35"),
    "c2": ("c2", 2.0, "NDT align, 32-ring scan (~60k pts) vs 500k-pt map, res 2.0, DIRECT7, eps 0.01, max_iter 35"),
    "c1": ("c1", 5.0, "NDT align, 16-ring scan (~10k pts) vs 50k-pt map, res 5.0, DIRECT7, eps 0.01, max_iter 35"),
}
N_SCANS = 4  # ray-cast base scans; every step gets its own copy with an independent sensor-noise draw (step_scans)


def make_workload(name: str, rank: int):
    from lidarslam_ros2_b200 import synth

    cfg, res, desc = WORKLOADS[name]
    src0, tgt, T_gt = synth.registration_pair(cfg, res)
    rings, azim = {"headline": (64, 1563), "c2": (32, 1875), "c1": (16, 625)}[name]
    scene = synth.make_scene()
    scans = [src0]
    d = np.pi / 180.0
    for k in range(1, N_SCANS):  # nearby sensor poses → different scans, same map; every rank gets the same poses
        s = 1.0 + 0.15 * k        # (same work per GPU: weak scaling) with its own noise stream
        T = synth.pose_matrix((0.40 * s, -0.25 * s, 0.06), (0.4 * d, -0.3 * d * s, 1.5 * d * s))
        scans.append(synth.make_scan(scene, rings, azim, synth.sensor_pose(T), stream=9000 + 10 * k + 100 * rank))
    return scans, tgt, res, desc


def step_scans(base, n_steps: int, rank: int):
    """One scan per step: base scan k mod N_SCANS plus an independent 3 mm isotropic sensor-noise draw (seeded by rank and
    step), so that no two steps of a run read the same input buffer. Deterministic; the CPU legs get the same arrays."""
    out = []
    for k in range(n_steps):
        rng = np.random.default_rng(77_000 + 1000 * rank + k)
        b = base[k % len(base)]
        out.append((b + rng.normal(0.0, 0.003, size=b.shape)).astype(np.float32))
    return out


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe) by a NATIVE thread
    (tools/clock_sampler.c: NVML through dlopen; one sample before the region, one 400 us into it — while the batched kernel runs
    and the host only waits — then at a backing-off period, one after the region: NVML queries contend with CUDA / NCCL calls).
    Round 1 polled NVML from a Python thread: eight such pollers fighting eight launch loops for their GILs cost one
    rank 6.5 ms inside a 3.8 ms timed region on the 8-GPU box. If the native sampler is unavailable the clocks are
    read once before and once after the region through nvidia_ml_py (never from a polling Python thread)."""

    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))
    LIB = os.path.join(ROOT, "tools", "libclocksampler.so")

    def __init__(self, gpu_index: int, period_us: int = 400):
        self.gpu, self.period_us = gpu_index, int(os.environ.get("BENCH_CLK_PERIOD_US", period_us))
        self.native = None
        self.nvml = None
        self.sm, self.mask, self.mx = [], 0, None
        self.acc_sm, self.acc_mask, self.acc_mx, self.used_native = [], 0, None, False

    def _uuid(self):
        try:
            import torch
            u = str(torch.cuda.get_device_properties(self.gpu).uuid)
            return u if u.startswith("GPU-") else "GPU-" + u
        except Exception:
            return None

    def _one_shot(self):
        try:
            import pynvml
            if self.nvml is None:
                pynvml.nvmlInit()
                u = self._uuid()
                self.h = pynvml.nvmlDeviceGetHandleByUUID(u) if u else pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
                self.nvml = pynvml
                self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.sm.append(float(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM)))
            try:
                self.mask |= int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                self.mask |= int(self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
        except Exception:
            pass

    def start(self):
        import ctypes as C
        try:
            if os.environ.get("BENCH_NO_NVML"):
                raise RuntimeError("disabled")
            L = C.CDLL(self.LIB)
            L.b200clk_start.argtypes = [C.c_char_p, C.c_int, C.c_int]
            L.b200clk_stop.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
            L.b200clk_arm.restype = None
            u = self._uuid()
            if L.b200clk_start(u.encode() if u else None, self.gpu, self.period_us) == 0:
                self.native = L
                return
        except Exception:
            self.native = None
        self._one_shot()

    def arm(self):
        if self.native is not None:
            self.native.b200clk_arm()

    def pause(self):
        """End of one timed region: collect its samples; start() may be called again for the next region."""
        import ctypes as C
        if self.native is not None:
            cap = 65536
            sm = (C.c_uint * cap)()
            rs = (C.c_ulonglong * cap)()
            mx = C.c_uint(0)
            n = self.native.b200clk_stop(sm, rs, cap, C.byref(mx))
            self.acc_sm += [float(sm[i]) for i in range(n)]
            for i in range(n):
                self.acc_mask |= int(rs[i])
            self.acc_mx = float(mx.value) or self.acc_mx
            self.native = None
            self.used_native = True
        else:
            self._one_shot()

    def stop(self) -> dict:
        if self.native is not None or not getattr(self, "used_native", False):
            self.pause()
        if getattr(self, "used_native", False):
            vals, mask, n = self.acc_sm, self.acc_mask, len(self.acc_sm)
            mx = type("M", (), {"value": self.acc_mx or 0.0})()
            return {"sm_mhz": float(np.median(vals)) if vals else None, "sm_max_mhz": float(mx.value) or None, "samples": n,
                    "reasons": sorted(name for bit, name in self.REASONS if mask & bit),
                    "source": f"nvml from a native thread: one sample before the timed region, one {self.period_us} us into it, then every "
                              "4 / 8 / 16 / 20 ms, one after it"}
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx, "samples": len(self.sm),
                "reasons": sorted(name for bit, name in self.REASONS if self.mask & bit),
                "source": "nvml, one sample before and one after the timed region (native sampler unavailable)"}


def pin_host_thread(local_rank: int):
    """Keep the launching thread on a few cores of its GPU's NUMA node for the timed regions (the 8-GPU box has two
    sockets; a migrating launch thread is one of the host-jitter sources the round-1 record showed). Returns the
    previous affinity so that the CPU baseline can have all cores back."""
    try:
        prev = os.sched_getaffinity(0)
    except Exception:
        return None
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        u = str(torch.cuda.get_device_properties(local_rank).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(u if u.startswith("GPU-") else "GPU-" + u)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = sorted(c for c in (w * 64 + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1) if c in prev)
        if len(cpus) >= 8:
            base = (local_rank * 8 + 4) % (len(cpus) - 4)
            os.sched_setaffinity(0, set(cpus[base:base + 4]))
    except Exception:
        pass
    return prev


def cpu_info() -> dict:
    info = {"cpus": os.cpu_count()}
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    info["model"] = line.split(":", 1)[1].strip()
                    break
        out = subprocess.run(["lscpu"], capture_output=True, text=True, timeout=5).stdout
        for line in out.splitlines():
            k = line.split(":", 1)[0].strip()
            if k in ("Socket(s)", "NUMA node(s)", "Thread(s) per core", "Core(s) per socket", "CPU max MHz"):
                info[k] = line.split(":", 1)[1].strip()
        with open("/sys/devices/system/cpu/cpu0/cpufreq/scaling_governor") as f:
            info["governor"] = f.read().strip()
    except Exception:
        pass
    return info


def ncu_traffic(n_registrations: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of the solver kernel for a launch of n_registrations, from the committed
    ncu --set full capture of the batched launch (profiles/r2_ndt_solver_traffic.json holds the bytes per registration of
    that capture; bench.py itself never runs under a profiler)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_ndt_solver_traffic.json")) as f:
            t = json.load(f)
        return float(t["dram_bytes_per_registration"]) * n_registrations
    except Exception:
        return None


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def synchronized_start(world: int, device):
    """Barrier, then a common wall-clock deadline: the ranks of ONE node share CLOCK_MONOTONIC, so rank 0 announces
    'now + 3 ms' and every rank spins until then — the start skew of the timed region drops from the barrier's exit skew
    (tens of microseconds, paid again as waiting time inside the closing all-gather) to about a microsecond."""
    import torch
    import torch.distributed as dist

    if world <= 1:
        torch.cuda.synchronize()
        return
    dist.barrier()
    torch.cuda.synchronize()
    if os.environ.get("BENCH_SYNC_START") == "0":  # developer switch: barrier only
        return
    t = torch.tensor([time.monotonic() + 0.003], dtype=torch.float64, device=device)
    dist.broadcast(t, src=0)
    deadline = float(t.item())
    while time.monotonic() < deadline:
        pass


def host_threads() -> int:
    """Hardware threads the CPU legs may use (torchrun exports OMP_NUM_THREADS=1, which is not a property of the box)."""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_thread_candidates():
    hw = host_threads()
    return sorted({c for c in (hw, max(1, hw // 2), 32, 16, 8) if c <= hw}, reverse=True)


def workload_config(name: str, scans, tgt) -> dict:
    """The `config` object — identical in the GPU arm and in the reference arm (same workload, same inputs)."""
    desc = WORKLOADS[name][2]
    return {"workload": desc, "n_source": int(len(scans[0])), "n_target": int(len(tgt)), "guess": "identity",
            "distinct_scans": len(scans),
            "l2": "GPU arm: 256 MiB memset evicts L2 before every timed region (and between the steps of the single_align leg); "
                  "inside the batched region every step reads its own scan buffer, the 0.5 MB voxel map of the fixed target "
                  "stays cache-resident by design (steady-state registration against one map); CPU arm: not applicable"}


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays: dict):
    """--dump-outputs: every array as <out_dir>/<name>.npy, float32 arrays as they are and all others as float64 (exact for
    the integer counters and flags). Nothing is written when no directory was given."""
    if not out_dir:
        return
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed {DUMP_MAX_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def make_cpu_ndt(res, threads):
    import oracle

    return oracle.NDT(resolution=res, transformation_epsilon=0.01, max_iterations=35, search_method=oracle.DIRECT7, num_threads=threads)


def best_cpu_threads(scans, tgt, res):
    """Thread count the CPU path runs fastest with on this box: all hardware threads, one per physical core (SMT siblings
    often hurt this cache-bound loop), or fewer (the std::map walks stop scaling early). One probe align each."""
    cand = cpu_thread_candidates()
    best = None
    for c in cand:
        n = make_cpu_ndt(res, c)
        n.set_target(tgt)
        n.set_source(scans[0])
        n.align()  # builds the lazy target kd-tree like PCL's first align
        t0 = time.perf_counter()
        n.align()
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, c)
    return best[1], cand


def time_cpu(scans, tgt, res, max_seconds: float, max_aligns: int, threads: int):
    """CPU oracle on the same workload. Returns (registrations/s, n_aligns, poses)."""
    n = make_cpu_ndt(res, threads)
    n.set_target(tgt)
    n.set_source(scans[0])
    n.align()  # warm-up (also builds the lazy target kd-tree like PCL's first align)
    poses, t_total, k = [], 0.0, 0
    while k < max_aligns and (k < 2 or t_total < max_seconds):
        n.set_source(scans[k % len(scans)])
        t0 = time.perf_counter()
        poses.append(n.align())
        t_total += time.perf_counter() - t0
        k += 1
    return k / t_total, k, poses


def cpu_thread_sweep(scans, tgt, res, counts):
    """registrations/s of the CPU path at a few thread counts (two aligns each; BASELINE.md quotes the reference's README at
    1 and 8 threads)."""
    out = {}
    for c in counts:
        n = make_cpu_ndt(res, c)
        n.set_target(tgt)
        n.set_source(scans[0])
        n.align()
        t0 = time.perf_counter()
        for k in range(2):
            n.set_source(scans[k % len(scans)])
            n.align()
        out[str(c)] = 2.0 / (time.perf_counter() - t0)
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU (OpenMP) path for this hot path, timed on the box's host cores with every
    hardware thread it can use (the reference itself needs PCL/Eigen/FLANN and cannot be built here: kind = port)."""
    if rank != 0:
        return
    base, tgt, res, desc = make_workload(args.workload, 0)
    scans = step_scans(base, max(args.steps, args.warmup, 1), 0)  # the very scans the GPU arm registers, step by step
    import oracle

    oracle.build()
    nt, cand = best_cpu_threads(scans, tgt, res)
    n = make_cpu_ndt(res, nt)
    n.set_target(tgt)
    for w in range(args.warmup):
        n.set_source(scans[w % len(scans)])
        n.align()
    t_total, poses = 0.0, []
    for k in range(args.steps):
        n.set_source(scans[k % len(scans)])
        t0 = time.perf_counter()
        T = n.align()
        t_total += time.perf_counter() - t0
        poses.append(T)
    v = args.steps / t_total
    sweep = cpu_thread_sweep(scans, tgt, res, sorted({1, min(8, host_threads())}))
    sweep[str(nt)] = v
    line = {
        "impl": "reference", "metric": "scan-to-map registrations/sec", "value": v, "unit": "registrations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 pair math / f64 reduction",
        "data": "synthetic",
        "config": workload_config(args.workload, base, tgt),
        "cpu_baseline": {"value": v, "unit": "registrations/s", "cores": nt, "kind": "port",
                         "sample": f"{args.steps} full align() calls, {nt} OpenMP threads (fastest of {cand}), "
                                   f"host has {os.cpu_count()} cpus",
                         "threads_sweep": sweep, "host": cpu_info(),
                         "note": "reference cannot be compiled here (PCL/Eigen/FLANN absent): CPU restatement oracle/"},
        "e2e": {"value": v, "unit": "registrations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    dump_outputs(args.dump_outputs, {"pose": np.stack(poses)})


def run_c5(args, rank, local_rank, world, m):
    """BASELINE config 5: streaming scan-to-growing-map. `--frames` synthetic frames of a drive down the canyon (0.5 m per
    frame, 32 rings x 1875 azimuths ~ 50k points), per frame the reference's frontend callback: VoxelGrid(0.2) +
    setInputSource + NDT align (res 5.0 as lidarslam.yaml / sm.cpp:28) from the previous pose, map update every 1.5 m
    (VoxelGrid(0.1), transform, concatenation of the last 10 submaps, setInputTarget). Host buffers in, pose out:
    this workload is end to end by construction. Inherently sequential -> 1 GPU (rank 0 only)."""
    import torch

    from lidarslam_ros2_b200 import synth
    from lidarslam_ros2_b200.scanmatcher import ScanMatcher

    if rank != 0:
        return
    rings, azim = 32, 1875
    frames = list(synth.drive_stream(args.frames, rings=rings, azimuths=azim, step=0.5, workers=min(32, os.cpu_count() or 1)))
    kw = dict(ndt_resolution=5.0, vg_size_for_input=0.2, vg_size_for_map=0.1, trans_for_mapupdate=1.5, num_targeted_cloud=10)
    warm = ScanMatcher(device=local_rank, **kw)
    for scan, _ in frames[:8]:  # warm-up on a throw-away session (allocations, first-launch costs)
        warm.receiveCloud(scan)
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.arm()
    passes = []
    for rep in range(3):  # three passes over the stream, each on a fresh session; the MEDIAN pass is reported
        sm = ScanMatcher(device=local_rank, **kw)
        launches0 = sm.registration.stats()["kernel_launches"]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        t0 = time.perf_counter()
        errs, n_upd, bytes_in, outs = [], 0, 0, []
        for scan, T_gt in frames:
            pose, final, upd = sm.receiveCloud(scan)
            n_upd += int(upd)
            bytes_in += scan.shape[0] * scan.shape[1] * 4
            errs.append(synth.pose_error(final, T_gt)[0])
            outs.append((pose, final, upd))
        e1.record()
        torch.cuda.synchronize()
        passes.append({"ms": e0.elapsed_time(e1), "wall": time.perf_counter() - t0, "errs": errs, "n_upd": n_upd, "bytes_in": bytes_in,
                       "outs": outs,
                       "st": sm.stats(), "launches": int(sm.registration.stats()["kernel_launches"] - launches0 + sm.stats()["kernel_launches"])})
    clocks = sampler.stop()
    passes.sort(key=lambda p: p["ms"])
    mid = passes[1]
    ms, wall, errs, n_upd, bytes_in, st = mid["ms"], mid["wall"], mid["errs"], mid["n_upd"], mid["bytes_in"], mid["st"]
    # CPU restatement of the same callback on a bounded prefix of the same stream
    import oracle
    import oracle.scanmatcher as osm

    oracle.build()
    best = None
    for c in cpu_thread_candidates():  # fastest thread count for this callback on this box (three probe frames each)
        op = osm.ScanMatcher(num_threads=c, **kw)
        c0 = time.perf_counter()
        for scan, _ in frames[:3]:
            op.receive_cloud(scan)
        dtc = time.perf_counter() - c0
        if best is None or dtc < best[0]:
            best = (dtc, c)
    cpu_threads = best[1]
    o = osm.ScanMatcher(num_threads=cpu_threads, **kw)
    n_cpu, t_cpu, dpose = 0, 0.0, 0.0
    g2 = ScanMatcher(device=local_rank, **kw)
    for scan, _ in frames[:min(len(frames), args.cpu_frames)]:
        c0 = time.perf_counter()
        po, To, _u = o.receive_cloud(scan)
        t_cpu += time.perf_counter() - c0
        n_cpu += 1
        pg, Tg, _u2 = g2.receiveCloud(scan)
        dpose = max(dpose, synth.pose_error(Tg, To)[0])
    v = len(frames) / (ms * 1e-3)
    line = {
        "metric": "streaming scan-to-growing-map frames/sec", "value": v, "unit": "frames/s", "n_gpus": 1, "steps": len(frames),
        "warmup": 4, "ms_per_step": ms / len(frames), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 pair math / f64 reduction", "data": "synthetic",
        "config": {"workload": f"c5: {len(frames)}-frame drive, {rings}x{azim} rays (~{int(np.mean([len(f[0]) for f in frames]))} pts/frame), "
                               "VoxelGrid 0.2 + NDT res 5.0 per frame, map update every 1.5 m (VoxelGrid 0.1, last 10 submaps)",
                   "map_updates": n_upd, "submaps": st["n_submaps"], "targeted_points": st["n_targeted"],
                   "trajectory_error_m": {"max": float(np.max(errs)), "final": float(errs[-1])},
                   "l2": "every frame is a new host buffer (one H2D copy per frame)",
                   "passes_ms_per_frame": [p["ms"] / len(frames) for p in passes]},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": int(bytes_in / len(frames)), "d2h_bytes_per_step": 56 + 64 + 456,
                "wall_s": wall},
        "gpu_launches": mid["launches"],
        "clocks": clocks,
        "roofline": None,
        "cpu_baseline": {"value": n_cpu / t_cpu if t_cpu > 0 else None, "unit": "frames/s", "cores": cpu_threads, "kind": "port",
                         "sample": f"first {n_cpu} frames of the same stream through oracle/scanmatcher.py", "pose_parity_max_m": dpose},
    }
    print(json.dumps(line), flush=True)
    pose7, final, updated = zip(*mid["outs"])  # per frame of the reported pass: what receiveCloud returned
    dump_outputs(args.dump_outputs, {"pose7": np.stack(pose7), "final_transformation": np.stack(final), "map_updated": np.array(updated)})


def run_c3(args, rank, local_rank, world, m):
    """BASELINE config 3: GICP align, 64-ring scan (~100k pts) vs 1M-pt map, corr_dist_threshold 5.0, transformation_epsilon
    1e-8 (scanmatcher_component.cpp:118-119), k = 20 (replicas per rank). Host buffers in, pose out. The target's 1M 20-NN
    covariances are computed once by the first align (reported separately); the timed steps are setInputSource + align."""
    import torch

    base, tgt, res, desc = make_workload("headline", rank)
    K = args.steps
    scans = step_scans(base, K, rank)
    g = m.GeneralizedIterativeClosestPoint(device=local_rank)
    g.setMaxCorrespondenceDistance(5.0)
    g.setTransformationEpsilon(1e-8)
    t0 = time.perf_counter()
    g.setInputTarget(tgt)
    g.setInputSource(scans[0])
    g.align()  # first align computes the target covariances (1M points, k = 20) once
    first_s = time.perf_counter() - t0
    g.setInputSource(scans[1 % K])
    g.align()
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.arm()
    launches0 = g.stats()["kernel_launches"]
    e = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    poses, inner_ms, pair_evals, its, evs = [], 0.0, 0.0, [], []
    torch.cuda.synchronize()
    for k in range(K):
        e[k][0].record()
        g.setInputSource(scans[k])
        poses.append(g.align())
        e[k][1].record()
        st = g.stats()
        inner_ms += st["gicp_inner_ms"]
        pair_evals += st["gicp_pair_evaluations"]
        its.append(st["iterations"])
        evs.append(st["evaluations"])
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = float(np.sum([a.elapsed_time(b) for a, b in e]))
    if rank != 0:
        return
    peak, which = hbm_peak()
    alg_bytes = pair_evals * (16 + 16 + 36 + 4)  # per correspondence and evaluation: moved point, target point, Mahalanobis 3x3, index
    achieved = alg_bytes / (inner_ms * 1e-3) / 1e9 if inner_ms > 0 else 0.0
    line = {"metric": "GICP scan-to-map registrations/sec", "value": K / (ms * 1e-3), "unit": "registrations/s", "n_gpus": 1,
            "steps": K, "warmup": 2, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 residuals / f64 covariances and sums", "data": "synthetic",
            "config": {"workload": "c3: GICP align, 64-ring scan (~100k pts) vs 1M-pt map, corr_dist 5.0, eps 1e-8, k=20",
                       "n_source": int(len(scans[0])), "n_target": int(len(tgt)),
                       "l2": "every step uploads its own scan (host buffers); the 1M-point target and its covariances stay resident"},
            "details": {"first_align_incl_target_covariances_s": first_s, "outer_iterations": its, "evaluations": evs},
            "e2e": {"value": K / (ms * 1e-3), "unit": "registrations/s", "h2d_bytes_per_step": int(len(scans[0]) * 12), "d2h_bytes_per_step": 64},
            "gpu_launches": int(g.stats()["kernel_launches"] - launches0), "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "gicp_inner_kernel (persistent: BFGS + all cost / gradient evaluations of one outer iteration)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": which, "traffic": None,
                         "alg_bytes_per_step": alg_bytes / K, "inner_kernel_ms_per_step": inner_ms / K,
                         "share_of_step": inner_ms / ms if ms > 0 else None,
                         "us_per_evaluation": 1e3 * inner_ms / max(1.0, float(np.sum(evs)))}}
    if not args.no_cpu_baseline:
        import oracle

        from lidarslam_ros2_b200 import synth

        oracle.build()
        o = oracle.GICP(max_correspondence_distance=5.0, transformation_epsilon=1e-8)
        o.set_target(tgt)
        o.set_source(scans[0])
        c0 = time.perf_counter()
        o.align()  # includes the 1.1M 20-NN covariances, like the GPU's first align
        first_cpu = time.perf_counter() - c0
        o.set_source(scans[1 % K])
        c0 = time.perf_counter()
        To = o.align()
        t_cpu = time.perf_counter() - c0
        g.setInputSource(scans[1 % K])
        dt, dr = synth.pose_error(g.align(), To)
        line["cpu_baseline"] = {"value": 1.0 / t_cpu, "unit": "registrations/s", "cores": host_threads(), "kind": "port",
                                "sample": "1 align() of step 1 (after the first align, which computes the target covariances: "
                                          f"{first_cpu:.1f} s on the CPU, {first_s:.2f} s on the GPU)",
                                "pose_parity": {"dt_m": dt, "dr_rad": dr}, "host": cpu_info()}
    print(json.dumps(line), flush=True)
    dump_outputs(args.dump_outputs, {"pose": np.stack(poses), "iterations": np.array(its), "evaluations": np.array(evs)})


def c4_generate(pairs: int, mine: list[int]):
    """The (scan, submap) pairs of the loop-closure sweep owned by this rank, generated in worker processes (before CUDA
    is touched: fork). Pair i is reproducible on its own (synth.loop_closure_pairs), so every N sees the same 64 pairs."""
    from concurrent.futures import ProcessPoolExecutor

    world = max(1, int(os.environ.get("WORLD_SIZE", "1")))
    workers = max(1, min(len(mine), host_threads() // world, 32))
    if workers <= 1 or len(mine) <= 1:
        return {i: _c4_pair((pairs, i)) for i in mine}
    with ProcessPoolExecutor(max_workers=workers) as ex:
        return dict(zip(mine, ex.map(_c4_pair, [(pairs, i) for i in mine])))


def _c4_pair(arg):
    from lidarslam_ros2_b200 import synth

    pairs, i = arg
    _, src, tgt, T_rel = next(iter(synth.loop_closure_pairs(pairs, first=i, count=1)))
    return src, tgt, T_rel


def c4_sweep(args, rank, local_rank, world, m, data, with_cpu: bool, comm=None):
    """BASELINE config 4 inside the default line: the loop-closure candidate sweep — args.pairs independent scan<->submap
    registrations (32-ring scan ~56k pts vs 200k-pt local map, NDT res 2.0, max_iter 100 as graph_based_slam_component.
    cpp:66), the SAME pairs at every N, pair i -> rank i mod N, per pair the node's sequence setInputTarget +
    setInputSource + align + getFitnessScore (gbs.cpp:181, 227-231) from HOST buffers, and ONE all-gather of the result
    rows INSIDE the timed region. Strong scaling: value = pairs / max-over-ranks time. Returns (the line's object, the
    gathered results) on rank 0 and (None, None) on the other ranks."""
    import torch
    import torch.distributed as dist

    from lidarslam_ros2_b200 import batch, synth

    mine = batch.shard_pairs(args.pairs, rank, world)
    prev_aff = pin_host_thread(local_rank)  # the sweep's host threads inherit the mask (cores of the GPU's NUMA node)
    sweep = batch.LoopSweep(m, device=local_rank, resolution=2.0, max_iterations=100)
    dev = torch.device("cuda", local_rank)
    if comm is None and world > 1:
        comm = batch.RowComm(rank, world, local_rank)  # ncclAllGather issued by libb200reg.so (b200comm.h)
    if mine:  # warm-up: one untimed pass over this rank's pairs — every engine of the sweep reaches its final buffer sizes
        sweep.run([data[i][0] for i in mine], [data[i][1] for i in mine], mine)
    for _ in range(8):  # NCCL warm-up (its channels come up lazily over the first few calls)
        batch.gather_rows(np.full((len(mine), batch.ROW), -1.0, dtype=np.float32), args.pairs, rank, world, device=dev, comm=comm)
    launches0 = sweep.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    synchronized_start(world, dev)
    e0.record()
    rows = sweep.run([data[i][0] for i in mine], [data[i][1] for i in mine], mine)
    res = batch.gather_rows(rows, args.pairs, rank, world, device=dev, comm=comm)  # the one collective: ncclAllGather of the rows
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    allms = [t.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(allms, t)
    per_rank_ms = [float(x.item()) for x in allms] if world > 1 else [ms]
    ms_max = max(per_rank_ms)
    if prev_aff:
        os.sched_setaffinity(0, prev_aff)  # the CPU leg below gets every core back
    if rank != 0:
        return None, None
    errs = [synth.pose_error(res["pose"][k], data[int(i)][2]) for k, i in enumerate(res["index"]) if int(i) in data]
    out = {
        "metric": "loop-closure candidate registrations/sec (64 scan<->submap pairs, sharded)", "value": args.pairs / (ms_max * 1e-3),
        "unit": "registrations/s", "n_gpus": world, "pairs": args.pairs, "ms_per_pair": ms_max / args.pairs, "ms_total": ms_max,
        "warmup": "one untimed pass over the same pairs",
        "per_rank_ms": per_rank_ms, "scaling": "strong", "collective": "ONE ncclAllGather of 20-float result rows, issued from C (b200comm_all_gather_rows), inside the timed region",
        "workload": f"c4: {args.pairs} independent NDT pairs, 32-ring scan (~56k) vs 200k-pt submap, res 2.0, max_iter 100, DIRECT7, "
                    "setInputTarget+setInputSource+align+getFitnessScore per pair from host buffers; pair i -> rank i mod N",
        "h2d_bytes_per_pair": int(np.mean([16 * (len(data[i][0]) + len(data[i][1])) for i in mine])) if mine else 0,
        "gpu_launches": int(sweep.kernel_launches() - launches0),
        "converged": int(res["converged"].sum()), "mean_iterations": float(res["iterations"].mean()),
        "mean_fitness": float(res["fitness"].mean()),
        "pose_error_vs_truth_max": [float(max(e[0] for e in errs)), float(max(e[1] for e in errs))] if errs else None,
    }
    if with_cpu:
        try:  # the reference's CPU path on a bounded sample of the same pairs (rank 0's first two)
            import oracle

            best = None
            for c in cpu_thread_candidates():  # the thread count this path runs fastest with on this box (one probe pair each)
                o = oracle.NDT(resolution=2.0, transformation_epsilon=0.01, max_iterations=100, search_method=oracle.DIRECT7, num_threads=c)
                c0 = time.perf_counter()
                o.set_target(data[mine[0]][1])
                o.set_source(data[mine[0]][0])
                o.align()
                o.fitness()
                dtc = time.perf_counter() - c0
                if best is None or dtc < best[0]:
                    best = (dtc, c)
            nt = best[1]
            o = oracle.NDT(resolution=2.0, transformation_epsilon=0.01, max_iterations=100, search_method=oracle.DIRECT7, num_threads=nt)
            t_cpu, n_cpu, dmax, rmax = 0.0, 0, 0.0, 0.0
            for i in mine[:2]:
                c0 = time.perf_counter()
                o.set_target(data[i][1])
                o.set_source(data[i][0])
                To = o.align()
                o.fitness()
                t_cpu += time.perf_counter() - c0
                n_cpu += 1
                k = int(np.where(res["index"] == i)[0][0])
                e = synth.pose_error(res["pose"][k], To)
                dmax, rmax = max(dmax, e[0]), max(rmax, e[1])
            out["cpu_baseline"] = {"value": n_cpu / t_cpu, "unit": "registrations/s", "cores": nt, "kind": "port",
                                   "sample": f"{n_cpu} of the pairs (setInputTarget + setInputSource + align + getFitnessScore)",
                                   "pose_parity_max": {"dt_m": dmax, "dr_rad": rmax}}
        except Exception as e:  # the GPU numbers must not depend on the CPU leg
            out["cpu_baseline"] = {"value": None, "error": str(e)}
    return out, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="headline", choices=sorted(WORKLOADS) + ["c3", "c4", "c5"])
    ap.add_argument("--pairs", type=int, default=64, help="loop-closure sweep: number of candidate pairs (strong scaling)")
    ap.add_argument("--frames", type=int, default=200, help="c5: frames of the synthetic drive (BASELINE config: 1000)")
    ap.add_argument("--cpu-frames", type=int, default=6, help="c5: frames of the stream the CPU restatement is timed on")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the loop-closure sweep object of the headline line")
    ap.add_argument("--slots", type=int, default=3, help="registrations in flight per batched launch (1..3)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path returned for each step as DIR/<name>.npy")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    args.warmup = max(args.warmup, 3)
    K, W = args.steps, args.warmup
    # ---- inputs first (worker processes fork before CUDA exists) --------------------------------------------------
    c4_data = None
    if args.workload in ("headline", "c4") and not (args.workload == "headline" and args.no_c4):
        from lidarslam_ros2_b200 import batch as _batch

        c4_data = c4_generate(args.pairs, _batch.shard_pairs(args.pairs, rank, world))

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the registration engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import lidarslam_ros2_b200 as m

    if args.workload in ("c3", "c5"):
        {"c3": run_c3, "c5": run_c5}[args.workload](args, rank, local_rank, world, m)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.workload == "c4":
        sampler = ClockSampler(local_rank)
        sampler.start()
        sampler.arm()
        c4, c4_res = c4_sweep(args, rank, local_rank, world, m, c4_data, with_cpu=False)
        clocks = sampler.stop()
        if rank == 0:
            c4["clocks"] = clocks
            print(json.dumps(c4), flush=True)
            dump_outputs(args.dump_outputs, c4_res)
        if world > 1:
            dist.destroy_process_group()
        return

    base, tgt, res, desc = make_workload(args.workload, rank)
    scans = step_scans(base, max(K, W), rank)

    ndt = m.NormalDistributionsTransform(device=local_rank)
    ndt.setResolution(res)
    ndt.setTransformationEpsilon(0.01)
    ndt.setMaximumIterations(35)
    ndt.setNeighborhoodSearchMethod(m.DIRECT7)
    ndt.setBatchSlots(args.slots)
    ndt.setInputTarget(tgt)  # first call: allocations
    t0 = time.perf_counter()
    ndt.setInputTarget(tgt)  # H2D + voxel map build (reported separately)
    set_target_ms = 1e3 * (time.perf_counter() - t0)
    target_build_ms = ndt.stats()["target_build_ms"]
    tgt_pinned = torch.from_numpy(np.ascontiguousarray(tgt)).pin_memory().numpy()
    ndt.setInputTarget(tgt_pinned)
    t0 = time.perf_counter()
    ndt.setInputTarget(tgt_pinned)
    set_target_pinned_ms = 1e3 * (time.perf_counter() - t0)

    # scans resident in HBM as float4 (plumbing: torch owns the device memory), and in pinned / pageable host memory
    dev_scans = [torch.from_numpy(np.concatenate([x, np.ones((len(x), 1), dtype=np.float32)], axis=1)).cuda() for x in scans]
    pinned_scans = [torch.from_numpy(np.ascontiguousarray(x)).pin_memory() for x in scans]
    pageable_scans = [np.ascontiguousarray(x).copy() for x in scans]
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    from lidarslam_ros2_b200 import batch as _b
    comm = _b.RowComm(rank, world, local_rank) if world > 1 else None  # the collective is issued by libb200reg.so (b200comm.h)
    # N > 1: the poses of the sharded batch are exchanged by the solver kernel itself (pose board: peer-memory stores over
    # NVLink as each registration converges, include/b200comm.h); BENCH_POSE_EXCHANGE=nccl keeps round 1's form — one
    # ncclAllGather behind the batch call — and is also the fallback when the boards cannot be mapped (said in the line).
    board, board_why = None, None
    if world > 1 and os.environ.get("BENCH_POSE_EXCHANGE", "board") == "board":
        try:
            board = comm.create_board(max(K, 1))
        except Exception as e:  # collective: fails on every rank or on none
            board_why = str(e)
    ptrs = [d.data_ptr() for d in dev_scans]
    counts = [int(d.shape[0]) for d in dev_scans]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def flush():
        if not args.no_flush:
            flush_buf.zero_()  # evict L2 (126 MB); excluded from the timing
            torch.cuda.synchronize()

    def timed(fn):
        """barrier + sync, CUDA events around fn() (synchronous engine call) + the pose all-gather, sync; max over ranks"""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        flush()
        sampler.start()  # one sample now (before the region); the sampling thread parks until arm()
        synchronized_start(world, torch.device("cuda", local_rank))
        sampler.arm()  # the next sample comes 400 us from here
        e0.record()
        w0 = time.perf_counter()
        r = fn()
        w1 = time.perf_counter()
        if board is not None:  # all ranks' poses arrived with the call (stored by the peers' kernels): r["gathered"]
            assert r["gathered"].shape[0] == world
        elif world > 1:  # fallback: ncclAllGather of the 4x4 poses behind the call, from C
            r["gathered"] = comm.all_gather_rows(r["pose"].reshape(-1, 16)[:K]).reshape(world, -1, 4, 4)
        w1b = time.perf_counter()
        e1.record()
        w1c = time.perf_counter()
        e1.synchronize()
        w2 = time.perf_counter()
        sampler.pause()
        barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms, 1e3 * (w1 - w0), 1e3 * (w2 - w1), 1e3 * (w1b - w1), 1e3 * (w1c - w1b), 1e3 * (w2 - w1c)], dtype=torch.float64,
                         device="cuda")
        allt = [t.clone() for _ in range(world)]
        if world > 1:
            dist.all_gather(allt, t)
        rows = [[float(v) for v in x.tolist()] for x in allt] if world > 1 else [[float(v) for v in t.tolist()]]
        per = [{"step_ms_sum": x[0], "engine_call_ms": x[1], "pose_gather_ms": x[2],
                "tail_ms": {"poses_out": x[3], "event_record": x[4], "event_sync": x[5]}} for x in rows]
        return r, max(x[0] for x in rows), per

    # ---- warm-up: W single aligns, one batch of W from HBM, one from host --------------------------------------
    for k in range(W):
        ndt.setInputSourceDevice(ptrs[k], counts[k])
        ndt.align()
    ndt.alignBatchDevice(ptrs[:W], counts[:W])
    ndt.alignBatch([p.numpy() for p in pinned_scans[:K]])  # full size: the staging / device buffers reach their final size here
    ndt.alignBatch(pageable_scans[:K])
    if board is not None:
        barrier()  # attached batch calls are collective: enter the first one together
        ndt.attachPoseBoard(board)
        for _ in range(2):
            ndt.alignBatchDevice(ptrs[:K], counts[:K])
            ndt.alignBatch([p.numpy() for p in pinned_scans[:K]])
            ndt.gatheredPoses()
        wb = ndt.prepareBatchDevice(ptrs[:W], counts[:W])
        for _ in range(3):
            wb()
    if world > 1:
        for _ in range(8):  # NCCL sets its channels up lazily over the first few calls (measured: 195, 123, 118, 42, 38 us ...)
            comm.all_gather_rows(np.zeros((K, 16), dtype=np.float32))

    prev_aff = pin_host_thread(local_rank)
    sampler = ClockSampler(local_rank)
    # ---- timed (value): K registrations of HBM-resident scans, ONE batched launch ---------------------------------
    launches0 = ndt.stats()["kernel_launches"]
    wall0 = time.perf_counter()
    rb, total_ms_max, per_rank_ms = timed(ndt.prepareBatchDevice(ptrs[:K], counts[:K]))
    wall = time.perf_counter() - wall0
    st = ndt.stats()
    launches = st["kernel_launches"] - launches0
    kernel_ms = float(st["solve_ms"])
    evals, hits = rb["evaluations"].astype(np.int64), rb["hits_total"].astype(np.int64)
    n_pts = np.array(counts[:K], dtype=np.int64)
    alg_bytes = float(np.sum(evals * (n_pts * 16 + n_pts * 7 * 8 + 224)) + np.sum(hits) * 48)
    # ---- timed (e2e): the same K registrations from HOST buffers through the public call ---------------------------
    re, e2e_ms_max, _ = timed(ndt.prepareBatch([p.numpy() for p in pinned_scans[:K]]))
    rp, e2e_pg_ms_max, _ = timed(ndt.prepareBatch(pageable_scans[:K]))
    clocks = sampler.stop()
    exchange_checked = None
    if world > 1:  # outside the timing: what the timed region gathered == an ncclAllGather of the ranks' own results
        exchange_checked = True
        for res_k in (rb, re, rp):
            ref = comm.all_gather_rows(res_k["pose"].reshape(-1, 16)[:K]).reshape(world, K, 4, 4)
            exchange_checked = exchange_checked and bool(np.array_equal(np.asarray(res_k["gathered"])[:, :K], ref))
    if board is not None:  # every rank unmaps the peers' boards while all of them are still alive (rank 0 runs CPU legs later)
        ndt.attachPoseBoard(None)
        barrier()
        board.close()

    # ---- single_align leg: one b200reg_align per step (latency-bound: round 1's headline), L2 flushed between steps ----
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    single_solve_ms, single_poses = [], []
    barrier()
    for k in range(K):
        flush()
        ev[k][0].record()
        ndt.setInputSourceDevice(ptrs[k], counts[k])
        single_poses.append(ndt.align())
        ev[k][1].record()
        single_solve_ms.append(ndt.stats()["solve_ms"])
    barrier()
    single_ms = float(np.sum([a.elapsed_time(b) for a, b in ev]))
    if prev_aff:
        os.sched_setaffinity(0, prev_aff)
    bitwise = all(np.array_equal(rb["pose"][k], single_poses[k]) for k in range(K)) and \
        all(np.array_equal(rb["pose"][k], re["pose"][k]) and np.array_equal(rb["pose"][k], rp["pose"][k]) for k in range(K))

    # ---- the loop-closure sweep (BASELINE config 4) rides in the same line ---------------------------------------
    c4, c4_res = None, None
    if c4_data is not None:
        c4, c4_res = c4_sweep(args, rank, local_rank, world, m, c4_data, with_cpu=not args.no_cpu_baseline, comm=comm)

    if rank == 0:
        peak, which = hbm_peak()
        achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0
        n_evals = int(np.sum(evals))
        line = {
            "metric": "scan-to-map registrations/sec", "value": world * K / (total_ms_max * 1e-3), "unit": "registrations/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": total_ms_max / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 pair math / f64 reduction", "data": "synthetic",
            "config": workload_config(args.workload, base, tgt),
            "details": {"n_voxels": int(st["n_voxels"]), "grid_ctas": st["grid_ctas"], "block_threads": st["block_threads"],
                        "index_in_smem": st["index_in_smem"], "slots_in_flight": args.slots,
                        "step": "the K steps are K independent registrations (own scan buffer each) issued as ONE "
                                f"b200reg_ndt_align_batch_device call = one persistent launch, {args.slots} registrations in flight",
                        "parallelism": ("1 GPU" if world == 1 else
                                        f"replicas x{world}, poses exchanged inside the timed region by the solver kernel itself: "
                                        "peer-memory stores into every rank's pose board over NVLink as each registration converges "
                                        "(b200reg_ndt_attach_pose_board)" if board is not None else
                                        f"replicas x{world} + ONE ncclAllGather of the poses (b200comm_all_gather_rows) inside the "
                                        f"timed region (pose board not used: {board_why or 'BENCH_POSE_EXCHANGE=nccl'})"),
                        "pose_exchange": None if world == 1 else ("pose_board" if board is not None else "nccl_all_gather"),
                        "pose_exchange_equals_nccl_all_gather": exchange_checked,
                        "batch_bitwise_equals_single_align": bool(bitwise),
                        "mean_iterations": float(rb["iterations"].mean()), "converged": int(rb["converged"].sum())},
            "e2e": {"value": world * K / (e2e_ms_max * 1e-3), "unit": "registrations/s",
                    "h2d_bytes_per_step": int(np.mean([p.numel() * 4 for p in pinned_scans[:K]])), "d2h_bytes_per_step": 448,
                    "ms_per_step": e2e_ms_max / K, "host_memory": "pinned",
                    "pageable": {"value": world * K / (e2e_pg_ms_max * 1e-3), "ms_per_step": e2e_pg_ms_max / K,
                                 "note": "pcl::PointCloud storage is pageable: staged through a pinned buffer with memcpy"}},
            "single_align": {"value": world * K / (single_ms * 1e-3), "unit": "registrations/s", "ms_per_step": single_ms / K,
                             "kernel_ms_per_step": float(np.mean(single_solve_ms)),
                             "note": "one b200reg_align per step (setInputSourceDevice + align, L2 flushed between steps): the "
                                     "latency of ONE registration; rank 0's own time"},
            "gpu_launches": int(launches),
            "per_rank": per_rank_ms,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": f"ndt_solver_kernel<DIRECT7> (persistent: all evaluations of {K} registrations, "
                                                   f"{args.slots} in flight)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": which,
                         "traffic": ncu_traffic(K), "alg_bytes_per_launch": alg_bytes,
                         "launch_ms": kernel_ms, "evaluations_per_launch": n_evals,
                         "us_per_evaluation": 1e3 * kernel_ms / max(1, n_evals),
                         "hits_per_point": float(np.sum(hits)) / max(1.0, float(np.sum(evals * n_pts)))},
            "target_build": {"set_input_target_ms": set_target_ms, "set_input_target_pinned_ms": set_target_pinned_ms,
                             "voxel_build_device_ms": target_build_ms,
                             "note": "wall clock of setInputTarget for the 1M-point map from pageable / pinned host memory "
                                     "(12 MB upload + build) and the device time of the voxel-map build alone"},
            "wall_s_timed_region": wall,
        }
        if c4 is not None:
            line["c4"] = c4
        if not args.no_cpu_baseline:
            import oracle

            oracle.build()
            nt, cand = best_cpu_threads(scans, tgt, res)
            v, k_done, cpu_poses = time_cpu(scans, tgt, res, max_seconds=15.0, max_aligns=min(K, 40), threads=nt)
            from lidarslam_ros2_b200 import synth

            errs = [synth.pose_error(rb["pose"][i], cpu_poses[i]) for i in range(min(len(cpu_poses), K))]
            sweep = cpu_thread_sweep(scans, tgt, res, sorted({1, min(8, host_threads())}))
            sweep[str(nt)] = v
            line["cpu_baseline"] = {"value": v, "unit": "registrations/s", "cores": nt, "kind": "port",
                                    "sample": f"{k_done} full align() calls of the same steps, {nt} OpenMP threads "
                                              f"(fastest of {cand}; host reports {os.cpu_count()} cpus)",
                                    "threads_sweep": sweep, "host": cpu_info(),
                                    "pose_parity_max": {"dt_m": max(e[0] for e in errs), "dr_rad": max(e[1] for e in errs)}}
        print(json.dumps(line), flush=True)
        # the value leg's batch result (one row per step) and, when it ran, the loop-closure sweep's gathered rows
        dump_outputs(args.dump_outputs, {**rb, **{"c4_" + k: v for k, v in (c4_res or {}).items()}})
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
