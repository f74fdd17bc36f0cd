#!/usr/bin/env python
"""Batched GICP (b200reg_gicp_align_batch) against K sequential setInputSource + align() calls on BASELINE config 3: 64-ring
scans (~94k points) against the 1M-point map, corr_dist 5.0, transformation_epsilon 1e-8, k = 20 (bench.py --workload c3).

  python tools/gicp_batch_bench.py [--ks 1,4,8,20] [--reps 3] [--slots 3] [--out FILE]

After a warm-up (the target covariances, both paths, the largest K) every repetition times, with CUDA events and a device
synchronise, (a) K sequential aligns from host buffers and then (b) alignBatch over the same K host buffers (for the largest
K also alignBatchDevice over float4 copies already in HBM); (a) and (b) alternate, the spread is the min / max over the
repetitions. One JSON line per K: registrations/s and ms per registration of every form (median), us per inner evaluation
(gicp_inner_ms / evaluations), the batched inner kernel's algorithmic bytes (gicp_pair_evaluations x 72 B: moved point,
target point, Mahalanobis 3x3, index — as bench.py's c3 roofline counts them) over its device time against the HBM peak,
whether every batched result is bitwise the sequential one, and the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (its main() is guarded)

PAIR_BYTES = 16 + 16 + 36 + 4


def gpu_name_and_power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = (x.strip() for x in out.split(",", 1))
        return name, limit
    except Exception:
        import torch

        return torch.cuda.get_device_name(0), None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="1,4,8,20")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--slots", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("gicp_batch_bench needs a CUDA device (there is no CPU fallback)")
    import lidarslam_ros2_b200 as m

    ks = [int(x) for x in args.ks.split(",")]
    kmax = max(ks)
    base, tgt, _, _ = bench.make_workload("headline", 0)
    scans = bench.step_scans(base, kmax, 0)
    dev = [torch.from_numpy(np.concatenate([s[:, :3], np.ones((len(s), 1), np.float32)], axis=1)).cuda() for s in scans]
    g = m.GeneralizedIterativeClosestPoint()
    g.setMaxCorrespondenceDistance(5.0)
    g.setTransformationEpsilon(1e-8)
    g.setCorrespondenceRandomness(20)
    g.setBatchSlots(args.slots)
    g.setInputTarget(tgt)
    g.setInputSource(scans[0])
    g.align()  # the 1M target covariances, once
    g.alignBatch(scans)
    g.alignBatchDevice([d.data_ptr() for d in dev], [d.shape[0] for d in dev])
    torch.cuda.synchronize()
    name, power_limit = gpu_name_and_power_limit()
    peak, peak_source = bench.hbm_peak()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        torch.cuda.synchronize()
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    def sequential(K):
        poses, its, evs, inner_ms = [], [], [], 0.0
        for k in range(K):
            g.setInputSource(scans[k])
            poses.append(g.align())
            st = g.stats()
            its.append(st["iterations"])
            evs.append(st["evaluations"])
            inner_ms += st["gicp_inner_ms"]
        return {"pose": np.stack(poses), "iterations": np.array(its), "evaluations": np.array(evs), "inner_ms": inner_ms}

    def batched(K, device):
        if device:
            r = g.alignBatchDevice([d.data_ptr() for d in dev[:K]], [d.shape[0] for d in dev[:K]])
        else:
            r = g.alignBatch(scans[:K])
        st = g.stats()
        r["inner_ms"], r["inner_launches"], r["pair_evaluations"] = st["gicp_inner_ms"], st["gicp_inner_launches"], st["gicp_pair_evaluations"]
        return r

    for K in ks:
        forms = ["sequential", "batch_host"] + (["batch_device"] if K == kmax else [])
        ms = {f: [] for f in forms}
        last = {}
        for _ in range(args.reps):  # alternate the forms inside every repetition
            for f in forms:
                t, out = timed(lambda: sequential(K) if f == "sequential" else batched(K, f == "batch_device"))
                ms[f].append(t)
                last[f] = out
        ref = last["sequential"]
        equal = all(np.array_equal(last[f]["pose"], ref["pose"]) and np.array_equal(last[f]["iterations"], ref["iterations"])
                    and np.array_equal(last[f]["evaluations"], ref["evaluations"]) and np.all(last[f]["status"] == 0)
                    for f in forms[1:])
        line = {"tool": "gicp_batch_bench", "K": K, "slots": args.slots, "reps": args.reps, "gpu": name, "power_limit": power_limit,
                "config": "c3: GICP, 64-ring scan vs 1M-pt map, corr_dist 5.0, eps 1e-8, k=20; host scans except batch_device",
                "n_source_mean": float(np.mean([len(s) for s in scans[:K]])), "bitwise_equal_to_single": bool(equal),
                "outer_iterations": [int(x) for x in ref["iterations"]], "evaluations": int(np.sum(ref["evaluations"]))}
        for f in forms:
            t = float(np.median(ms[f]))
            evals = float(np.sum(last[f]["evaluations"]))
            entry = {"registrations_per_s": K / (t * 1e-3), "ms_per_registration": t / K,
                     "ms_spread": [float(np.min(ms[f])), float(np.max(ms[f]))],
                     "us_per_inner_evaluation": 1e3 * last[f]["inner_ms"] / max(evals, 1.0), "inner_kernel_ms": last[f]["inner_ms"]}
            if f != "sequential":
                achieved = last[f]["pair_evaluations"] * PAIR_BYTES / (last[f]["inner_ms"] * 1e-3) / 1e9 if last[f]["inner_ms"] > 0 else 0.0
                entry.update({"inner_launches": int(last[f]["inner_launches"]), "inner_alg_gbs": achieved, "hbm_peak_gbs": peak,
                              "hbm_peak_source": peak_source, "inner_hbm_frac": achieved / peak})
            line[f] = entry
        line["speedup_batch_host"] = line["batch_host"]["registrations_per_s"] / line["sequential"]["registrations_per_s"]
        s = json.dumps(line)
        print(s, flush=True)
        if args.out:
            with open(args.out, "a") as fh:
                fh.write(s + "\n")


if __name__ == "__main__":
    main()
