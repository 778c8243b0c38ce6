"""Throughput of the batched disk statistics (epid_disk_roi_stats) on a device-resident batch of 512 x 1024 x 1024 uint16 frames.

Two layouts a phantom module would sample:
  qc3  11 disks of r ~ 19 px (a planar QC-3-like pattern), median + std per disk
  ct   8 disks of r ~ 60 px and one of r ~ 150 px (a CT-slice-like pattern; the large disk does not fit the shared-memory stage and
       takes the re-read path)
Each call is synchronous (it returns once the statistics are in host memory), so the wall time of a call, taken with a host clock, is
the end-to-end time a caller sees; the kernel time alone comes from torch.profiler (CUDA activities) in a separate pass.  The card
name and power limit are read in the same run.  Prints one JSON line.

    python tools/bench_disk_roi.py [--frames 512] [--reps 10] [--warmup 3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from pylinac_b200 import _native as nat  # noqa: E402


def layouts():
    qc3 = [(512 + 260 * np.cos(a), 512 + 260 * np.sin(a)) for a in np.linspace(0, 2 * np.pi, 11, endpoint=False)]
    ct = [(512 + 330 * np.cos(a), 512 + 330 * np.sin(a)) for a in np.linspace(0, 2 * np.pi, 8, endpoint=False)] + [(512.0, 512.0)]
    return {"qc3": (qc3, [19.0] * 11), "ct": (ct, [60.0] * 8 + [150.0])}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception as e:          # reported, not fatal: the timing stands without it
        return f"unknown ({e})", "unknown"


def kernel_ms(ctx, b, centres, radii, pcts, reps):
    """Mean device time of k_disk_roi_stats per call from torch.profiler, or None when the profiler sees no such kernel."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
    except ImportError:
        return None
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            nat.disk_roi_stats(ctx, b, centres, radii, pcts)
    us = sum(e.device_time_total for e in prof.key_averages() if "k_disk_roi_stats" in e.key)
    return us / 1e3 / reps if us > 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if nat.device_count() < 1:
        raise SystemExit("bench_disk_roi needs a CUDA device")
    ctx = nat.Context.default()
    rng = np.random.default_rng(0)
    block = rng.normal(20000, 900, (8, 1024, 1024)).clip(0, 65535).astype(np.uint16)
    frames = np.tile(block, (args.frames // 8, 1, 1))
    b = nat.Batch.upload(ctx, frames)
    del frames
    name, power = card()
    res = {"tool": "bench_disk_roi", "gpu": name, "power_limit": power, "frames": args.frames, "frame_shape": [1024, 1024],
           "dtype": "uint16", "reps": args.reps}
    try:
        for lay, (centres, radii) in layouts().items():
            for _ in range(args.warmup):
                nat.disk_roi_stats(ctx, b, centres, radii)
            ts = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                nat.disk_roi_stats(ctx, b, centres, radii)
                ts.append(time.perf_counter() - t0)
            t = float(np.median(ts))
            k = kernel_ms(ctx, b, centres, radii, (), min(args.reps, 5))
            res[lay] = {"disks_per_frame": len(radii), "call_ms_median": t * 1e3, "call_ms_min": min(ts) * 1e3,
                        "frames_per_s": args.frames / t, "disks_per_s": args.frames * len(radii) / t, "kernel_ms": k}
    finally:
        b.free()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
