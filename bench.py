#!/usr/bin/env python
"""Benchmark of the hot path named by BASELINE.json: EPID frames/s (1024x1024) through PicketFence.analyze().

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...            # the reference algorithm on the host CPU cores (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results to DIR/*.npy

A "step" is one pass of the whole PicketFence pipeline over one batch of synthetic frames (config.workload); every PicketFence leg
below times exactly K steps.  The frames are generated from fixed seeds, so two builds given the same arguments analyse the same
inputs and their --dump-outputs files can be compared array for array.
  value    : whole-job frames/s with the batch already resident in HBM (CUDA events around exactly K back-to-back passes, max over ranks)
  e2e      : the same metric through the public API `pylinac_b200.picketfence.analyze_batch` with HOST frames in page-locked memory --
             chunked H2D copies and the D2H of the results are inside the timed region; `e2e_pageable` is the same call on an
             ordinary numpy array (what a drop-in user passes)
  roofline : the kernel with the largest share of the step (CUDA-event marks between the kernels INSIDE the timed region) against the
             measured HBM copy bandwidth, on SURVEY.md 8(d)'s algorithmic bytes (one read of every uint16 frame per step);
             `pipeline` is the whole step on the same bytes, `kernels` lists every stage
  cpu_baseline: the oracle port (numpy/scipy restatement of the reference, bit-identical to it on the golden cases) on all host
             cores for a bounded sample of the same frames: wall-clock throughput, with the cgroup CPU quota next to the core count
  mixed_noisy_5pct / modules: the per-frame-fallback workload and configs[2..4] (Winston-Lutz, Starshot, FieldAnalysis), measured in
             the same run (single-GPU runs only)
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAME_SHAPE = (1024, 1024)
DPMM = 2.56
PER_GPU_FRAMES = 512          # BASELINE.json configs[1]
DUMP_LIMIT = 60_000_000      # array bytes written by --dump-outputs (with the .npy headers the files stay under 64 MB)
METRIC = "EPID frames/sec (1024x1024) through PicketFence.analyze()"
_SHARED_FRAMES = None         # frames handed to forked CPU workers


def _gen_frame(i):
    from oracle import synth

    return synth.bench_pf_frame(i, FRAME_SHAPE)


def _oracle_shared(k):
    import warnings

    from oracle import pf_oracle

    a = _SHARED_FRAMES[k]
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        r = pf_oracle.pf_analyze(a, DPMM)
    return time.perf_counter() - t0, r["n_meas"]


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cgroup_cpu_quota():
    """CPUs the cgroup may use (cpu.max quota / period), or None when unlimited / unknown."""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else float(q) / float(p)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            return None if q <= 0 else q / p
        except Exception:
            return None


class CpuReference:
    """The CPU restatement of the reference on `cores` forked processes over a fixed sample of pre-generated frames (one pool for
    the whole run; frames reach the workers through fork, so a timed step is analysis only)."""

    def __init__(self, n_frames: int, cores: int, start: int = 0):
        global _SHARED_FRAMES
        for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
            os.environ[k] = "1"
        self.cores = cores
        self.n = n_frames
        ctx = mp.get_context("fork")
        with ctx.Pool(min(cores, n_frames)) as pool:
            _SHARED_FRAMES = pool.map(_gen_frame, range(start, start + n_frames), chunksize=1)
        self.pool = ctx.Pool(cores)
        self.pool.map(_oracle_shared, range(min(cores, n_frames)))          # warm the workers (imports, first-touch)

    def step(self):
        """-> (wall-clock frames/s, mean in-worker seconds per frame)"""
        t0 = time.perf_counter()
        res = self.pool.map(_oracle_shared, range(self.n), chunksize=1)
        wall = time.perf_counter() - t0
        return self.n / wall, sum(r[0] for r in res) / self.n

    def close(self):
        global _SHARED_FRAMES
        self.pool.close()
        self.pool.join()
        _SHARED_FRAMES = None


def generate_frames(n: int, start: int, cores: int) -> np.ndarray:
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        frames = pool.map(_gen_frame, range(start, start + n), chunksize=4)
    return np.stack(frames)


def _cpu_baseline_job(sample: int, cores: int):
    ref = CpuReference(sample, cores, start=2000)
    fps, per = ref.step()
    fps2, per2 = ref.step()
    ref.close()
    return max(fps, fps2), min(per, per2)


def _isolated_entry(conn, func, args, chunked):
    try:
        out = func(*args)
        if chunked:      # a large ndarray: 64 leading entries per message (a pipe message is limited to 2 GiB)
            conn.send(("shape", (out.shape, str(out.dtype))))
            for i in range(0, out.shape[0], 64):
                conn.send(("chunk", out[i:i + 64]))
            conn.send(("ok", None))
        else:
            conn.send(("ok", out))
    except BaseException as e:       # noqa: BLE001 -- reported to the parent
        conn.send(("err", repr(e)))
    finally:
        conn.close()


def _isolated(func, *args, chunked: bool = False):
    """Run `func` in a freshly spawned interpreter and return its result.  The CPU baseline and the frame generator fork up to 128
    worker processes; measured on the B200 hosts (profiles/r2m_summary.md), a process that has done that stages pageable frames 1.5 x
    slower afterwards (44.8 vs 29.9 ms per 512-frame step), so the GPU process of this benchmark never forks a pool itself."""
    ctx = mp.get_context("spawn")
    parent, child = ctx.Pipe(duplex=False)
    proc = ctx.Process(target=_isolated_entry, args=(child, func, args, chunked), daemon=False)
    proc.start()
    child.close()
    out, filled = None, 0
    while True:
        kind, val = parent.recv()
        if kind == "shape":
            out = np.empty(val[0], np.dtype(val[1]))
        elif kind == "chunk":
            out[filled:filled + len(val)] = val
            filled += len(val)
        elif kind == "ok":
            result = out if chunked else val
            break
        else:
            proc.join()
            raise RuntimeError(f"{func.__name__} failed in the isolated process: {val}")
    proc.join()
    return result


def dump_outputs(path, summary, meas):
    """What analyze_batch returned in the last timed end-to-end step, one float64 array per field: summary_<field>.npy [n, ...] and
    meas_<field>.npy [n, m, ...], where m is the largest measurement count of a frame (a frame's rows past its own count are zero),
    and frame_index.npy, the batch index of every row.  A batch whose arrays exceed DUMP_LIMIT is written as a fixed seeded sample
    of its frames."""
    n, m = len(summary), int(summary["n_meas"].max())
    width = lambda dt: sum(int(np.prod(dt[f].shape)) for f in dt.names)      # float64 values per row
    per_frame = 8 * (1 + width(summary.dtype) + m * width(meas.dtype))
    k = min(n, DUMP_LIMIT // per_frame)
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "frame_index.npy"), idx.astype(np.float64))
    for f in summary.dtype.names:
        np.save(os.path.join(path, f"summary_{f}.npy"), summary[f][idx].astype(np.float64))
    for f in meas.dtype.names:
        np.save(os.path.join(path, f"meas_{f}.npy"), meas[f][idx, :m].astype(np.float64))


def _gen_module_frames(kind_i):
    from oracle import synth

    kind, i = kind_i
    rng = np.random.default_rng(7000 + i)
    if kind == "star":
        return synth.starshot_frame(synth.epid1024(), offsets_mm=[tuple(rng.uniform(-0.5, 0.5, 2)) for _ in range(6)], noise_sigma=0.002, seed=100 + i)
    if kind == "field":
        return synth.openfield_frame(synth.as1200(1000.0), cax_offset_mm=tuple(rng.uniform(-3, 3, 2)), seed=200 + i)
    return synth.winstonlutz_frame(synth.epid1024(), offset_mm_left=rng.uniform(-1, 1), offset_mm_up=rng.uniform(-1, 1),
                                   offset_mm_in=rng.uniform(-1, 1), gantry=22.5 * i, couch=(0, 45, 90, 270, 315)[i % 5] if i % 4 == 0 else 0,
                                   noise_sigma=0.002, seed=300 + i)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend="gloo", rank=rank, world_size=world)   # plumbing only: barrier + max(time)
        return dist, world, rank, local
    return None, 1, 0, 0


def run_reference(args):
    # under torchrun only rank 0 measures (the host cores are shared by all ranks); no process group is needed for that
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    cores = host_cores()
    sample = cores                      # one frame per process and step: a step lasts one single-core frame analysis (~0.3 - 1.6 s)
    ref = CpuReference(sample, cores, start=1000)
    for _ in range(args.warmup):
        ref.step()
    fps_all, times, per = [], [], []
    for _ in range(args.steps):
        fps, sec = ref.step()
        fps_all.append(fps)
        per.append(sec)
        times.append(sample / fps * 1e3)
    ref.close()
    fps = statistics.mean(fps_all)
    out = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": statistics.mean(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"PicketFence.analyze() on synthetic 1024x1024 MLC picket frames; each step = {sample} frames "
                               f"on {cores} host processes (bounded sample of the {PER_GPU_FRAMES}-frame batch)"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "cgroup_cpu_quota": cgroup_cpu_quota(), "kind": "port",
                         "sample": f"{sample} pre-generated frames per step; wall-clock throughput of the analysis; "
                                   f"{statistics.mean(per) * 1e3:.0f} ms per frame inside a worker"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))
    return 0


def bench_modules(ctx, nat, peak, cores):
    """configs[2..4] in the same run: device-resident and end-to-end frames/s of the Winston-Lutz, Starshot and FieldAnalysis batch
    pipelines (frames tiled from 16 unique synthetic frames each), with the one-read HBM fraction (SURVEY.md 8(d) bytes)."""
    from pylinac_b200 import field_analysis as fa
    from pylinac_b200 import starshot as ss
    from pylinac_b200 import winston_lutz as wlm

    mctx = mp.get_context("fork")
    out = {}
    specs = [("winston_lutz_2d", "wl", 2048, lambda: wlm.make_params(2.56), nat.wl2d_analyze, "configs[2]: 2048 synthetic BB + field frames, 1024x1024"),
             ("starshot", "star", 256, lambda: ss.make_params(2.56), nat.starshot_analyze, "configs[3]: 256 synthetic star images, 1024x1024"),
             ("field_analysis", "field", 4096, lambda: fa.make_params(1 / 0.336), nat.field_analyze, "configs[4]: 4096 open-field frames, 1280x1280")]
    for name, kind, count, mk, fn, what in specs:
        try:
            with mctx.Pool(min(cores, 16)) as pool:
                uniq = np.stack(pool.map(_gen_module_frames, [(kind, i) for i in range(16)], chunksize=1))
        except Exception as e:       # forking after CUDA initialisation is not always possible: generate in-process
            uniq = np.stack([_gen_module_frames((kind, i)) for i in range(16)])
        frames = nat.pinned_empty((count,) + uniq.shape[1:], np.uint16)
        for k in range(0, count, 16):
            frames[k:k + 16] = uniq
        params = mk()
        b = nat.Batch.upload(ctx, frames)
        fn(ctx, b, params)
        ctx.sync()
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            rows = fn(ctx, b, params)
        ctx.sync()
        dev_s = (time.perf_counter() - t0) / reps
        b.free()
        t0 = time.perf_counter()
        for _ in range(2):
            bb = nat.Batch.upload(ctx, frames)
            rows2 = fn(ctx, bb, params)
            bb.free()
        ctx.sync()
        e2e_s = (time.perf_counter() - t0) / 2
        out[name] = {"workload": what, "frames": count, "device_resident_fps": count / dev_s, "e2e_fps": count / e2e_s,
                     "ms_per_batch": dev_s * 1e3, "status_ok": int((rows["status"] == 0).sum()),
                     "one_read_frac": frames.nbytes / dev_s / 1e9 / peak, "h2d_bytes": int(frames.nbytes),
                     "note": "device-resident time includes the D2H of the result rows"}
        del frames
    # VMAT (DRGS): image pairs, 1280 x 1280; algorithmic bytes = one read of BOTH frames of a pair
    try:
        from pylinac_b200 import vmat as vm

        pairs = [_gen_vmat_pair(i) for i in range(4)]
        count = 1024
        f1 = nat.pinned_empty((count,) + pairs[0][0].shape, np.uint16)
        f2 = nat.pinned_empty((count,) + pairs[0][0].shape, np.uint16)
        for k in range(count):
            f1[k], f2[k] = pairs[k % 4][k % 2], pairs[k % 4][1 - k % 2]      # either order: the open image is identified per pair
        params = vm._make_params(1 / 0.336, 1.5, (5, 100), [-60, -40, -20, 0, 20, 40, 60], True, True, False)
        b1, b2 = nat.Batch.upload(ctx, f1), nat.Batch.upload(ctx, f2)
        nat.vmat_analyze(ctx, b1, b2, params)
        ctx.sync()
        t0 = time.perf_counter()
        for _ in range(3):
            rows = nat.vmat_analyze(ctx, b1, b2, params)
        ctx.sync()
        dev_s = (time.perf_counter() - t0) / 3
        b1.free()
        b2.free()
        out["vmat_drgs"] = {"workload": "1024 synthetic DRGS (open, DMLC) pairs, 1280x1280, 7 segments", "pairs": count,
                            "device_resident_pairs_per_s": count / dev_s, "ms_per_batch": dev_s * 1e3, "status_ok": int((rows["status"] == 0).sum()),
                            "one_read_frac": (f1.nbytes + f2.nbytes) / dev_s / 1e9 / peak,
                            "note": "one read of both frames of a pair is the algorithmic traffic; time includes the D2H of the result rows"}
        del f1, f2
    except Exception as e:
        out["vmat_drgs"] = {"error": repr(e)}
    return out


def _gen_vmat_pair(i):
    from oracle import synth

    o = synth.as1200(1000.0)
    o.add_filtered_field((150, 150), alpha=0.6)
    o.gaussian(2.0)
    o.noise(0.002, seed=400 + i)
    d = synth.as1200(1000.0)
    for off, a in zip((-60, -40, -20, 0, 20, 40, 60), (0.30, 0.302, 0.299, 0.30, 0.301, 0.298, 0.30)):
        d.add_filtered_field((150, 18), cax_offset_mm=(0, off), alpha=a)
    d.gaussian(1.5)
    d.noise(0.002, seed=500 + i)
    return o.image, d.image


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--frames", type=int, default=PER_GPU_FRAMES, help="frames per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-modules", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed end-to-end step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    dist, world, rank, local = dist_setup()
    cores = host_cores()
    n = args.frames
    warmup = max(args.warmup, 3)
    # ---- everything that forks happens BEFORE the CUDA context exists
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample = cores
        fps, per = _isolated(_cpu_baseline_job, sample, cores)
        cpu_base = {"value": fps, "unit": "frames/s", "cores": cores, "cgroup_cpu_quota": cgroup_cpu_quota(), "kind": "port",
                    "sample": f"{sample} of the batch's frames on {cores} processes, wall-clock throughput of the analysis (best of 2 "
                              f"passes); {per * 1e3:.0f} ms per frame inside a worker"}
    gen_cores = max(1, cores // world)
    frames_np = _isolated(generate_frames, n, rank * n, gen_cores, chunked=True)

    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    ndev = nat.device_count()
    if ndev == 0:
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    ctx = nat.Context.default(local % ndev)
    from pylinac_b200 import parallel as par

    numa = par.bind_host_to_gpu(local % ndev)      # before the page-locked buffers exist: first touch puts them on the GPU's node
    params = pf.make_params(DPMM, FRAME_SHAPE)
    pinned = nat.pinned_empty(frames_np.shape, np.uint16)
    pinned[...] = frames_np
    # an ordinary numpy array, what a drop-in user passes -- allocated (first touch) AFTER the rank bound itself to the GPU's NUMA node,
    # like the page-locked buffer above; the generator's array was assembled before the binding and may sit on the other socket
    pageable = np.array(pinned, copy=True)
    del frames_np
    batch = nat.Batch.upload(ctx, pinned)

    if world > 1:
        par.init_comm(ctx, dist)

    def barrier():
        if dist is not None:
            dist.barrier()

    def gather(res):
        if world > 1:   # the job's only exchange: all ranks' summary rows (fixed size) to every rank
            allsum = np.zeros(world * n, nat.PF_SUMMARY_DTYPE)
            nat.check(nat.lib().epid_gather_results(ctx.handle, res.summary.ctypes.data, res.summary.nbytes, allsum.ctypes.data))

    # ---- warm-up (also grows the scratch arenas)
    nat.pf_bench(ctx, batch, params, warmup)
    for _ in range(warmup):
        res = pf.analyze_batch(pinned, DPMM, meas_cap=1024)
        gather(res)
    pf.analyze_batch(pageable, DPMM, meas_cap=1024)

    # ---- timed: device-resident, CUDA-event marks between the kernels inside the timed region
    clocks = ClockSampler(local % ndev)
    clocks.start()
    barrier()
    ctx.sync()
    total_ms, stage_ms, launches_timed, _ = nat.pf_bench_timed(ctx, batch, params, args.steps)
    ctx.sync()
    barrier()
    # ---- timed: end to end through the public API, host (pinned) frames in, host results out
    meas_cap = 1024
    summ_bytes = nat.PF_SUMMARY_DTYPE.itemsize * n
    meas_bytes = nat.PF_MEAS_DTYPE.itemsize * n * meas_cap
    barrier()
    ctx.sync()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = pf.analyze_batch(pinned, DPMM, meas_cap=meas_cap)
        gather(res)
    ctx.sync()
    e2e_s = time.perf_counter() - t0
    barrier()
    clk = clocks.stop()
    assert all(int(s) == 0 for s in res.summary["status"]), "pipeline reported a failed frame"
    # ---- the same call on pageable memory
    psteps = args.steps
    barrier()
    t0 = time.perf_counter()
    for _ in range(psteps):
        resp = pf.analyze_batch(pageable, DPMM, meas_cap=meas_cap)
        gather(resp)
    ctx.sync()
    e2e_page_s = (time.perf_counter() - t0) / psteps
    barrier()
    # ---- the host -> device copy of one step alone (all ranks at the same time): what the end-to-end leg cannot go below, and what
    # shows whether ranks slow each other down on the host side (shared memory controllers / PCIe root complexes)
    batch.write(pinned)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        batch.write(pinned)
    h2d_only_s = (time.perf_counter() - t0) / args.steps
    barrier()

    # ---- max over ranks
    if dist is not None:
        import torch

        t = torch.tensor([total_ms, e2e_s * 1e3, e2e_page_s * 1e3, h2d_only_s * 1e3], dtype=torch.float64)
        tmin = t.clone()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        total_ms, e2e_ms, e2e_page_ms, h2d_only_ms = (float(x) for x in t)
        h2d_only_min_ms = float(tmin[3])
    else:
        e2e_ms, e2e_page_ms, h2d_only_ms = e2e_s * 1e3, e2e_page_s * 1e3, h2d_only_s * 1e3
        h2d_only_min_ms = h2d_only_ms
    if rank != 0:
        dist.barrier()
        dist.destroy_process_group()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    H0, W0 = FRAME_SHAPE
    alg_bytes = n * H0 * W0 * 2                      # SURVEY.md 8(d): one read of every raw uint16 frame per step
    step_ms = total_ms / args.steps
    frames_total = world * n * args.steps
    # per-kernel table: the bytes a kernel has to touch once (pilot: every 32nd row; stream: the cropped view; window kernels: the
    # (leaf, picket) windows of PicketFence._get_mlc_window; tail / finalize: 1-D partial sums and window results)
    H, W = H0 - 2 * params.crop_px, W0 - 2 * params.crop_px
    m0 = int(res.summary["n_meas"][0])
    widths = {int(params.leaf_num[i]): params.leaf_width_mm[i] * DPMM for i in range(params.n_leaves)}
    spacing = int(float(res.summary["picket_spacing_px"][0]))
    win_px = sum(int(widths[int(l)]) * spacing for l in res.meas["leaf_num"][0, :m0])
    own = {"k_pf_init + k_pf_pilot": n * ((H + 31) // 32) * W * 2, "k_pf_stream": n * H * W * 2, "k_pf_windows_fast": n * win_px * 2,
           "k_pf_win_medians": n * win_px * 2}
    ktable = []
    for name, ms in stage_ms.items():
        if ms <= 0:
            continue
        ab = own.get(name)
        ktable.append({"kernel": name, "ms": ms, "share": ms / step_ms, "own_bytes": ab, "own_GBps": (ab / (ms * 1e-3) / 1e9) if ab else None,
                       "own_frac": (ab / (ms * 1e-3) / 1e9 / peak) if ab else None,
                       "frac_on_one_read_bytes": alg_bytes / (ms * 1e-3) / 1e9 / peak})
    dom = max(ktable, key=lambda k: k["ms"])
    dom_gbs = alg_bytes / (dom["ms"] * 1e-3) / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "dominant_traffic.json")))
        if tj.get("kernel") == dom["kernel"]:   # ncu dram__bytes_read + dram__bytes_write of one launch, scaled from the captured batch size
            traffic = tj["dram_bytes_per_launch"] * n / tj["frames"]
    except Exception:
        pass
    pipe_gbs = alg_bytes / (step_ms * 1e-3) / 1e9
    out = {
        "metric": METRIC, "value": frames_total / (total_ms * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u16 pixels / int exact sums / f64 profiles", "data": "synthetic",
        "config": {"workload": f"PicketFence.analyze() on a batch of {n} synthetic 1024x1024 MLC picket frames per GPU "
                               "(BASELINE.json configs[1]); 10 pickets x 50 leaf pairs = 500 kisses per frame",
                   "frames_per_gpu": n, "parallelism": f"frames sharded over {world} GPU(s), no data-path collective",
                   "host_numa": numa,
                   "l2": f"batch = {n * H0 * W0 * 2 / 1e6:.0f} MB per GPU, larger than the 126 MB L2; no flush needed"},
        "e2e": {"value": frames_total / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": int(n * H0 * W0 * 2),
                "d2h_bytes_per_step": int(summ_bytes + meas_bytes), "ms_per_step": e2e_ms / args.steps,
                "api": "pylinac_b200.picketfence.analyze_batch(host uint16 frames in page-locked memory) -> per-frame results"
                       + (" + ncclAllGather of the summaries" if world > 1 else ""),
                "h2d_only_ms_per_step": {"max_over_ranks": h2d_only_ms, "min_over_ranks": h2d_only_min_ms,
                                         "GBps_per_rank_at_max": n * H0 * W0 * 2 / (h2d_only_ms * 1e-3) / 1e9,
                                         "note": "the step's host->device copy alone, all ranks copying at the same time: the floor of "
                                                 "the end-to-end step; growth with the rank count = host-side contention, not NVLink"}},
        "e2e_pageable": {"value": world * n / (e2e_page_ms * 1e-3), "unit": "frames/s", "ms_per_step": e2e_page_ms, "steps": psteps,
                         "frac_of_pinned": (world * n / (e2e_page_ms * 1e-3)) / (frames_total / (e2e_ms * 1e-3)),
                         "api": "the same call on an ordinary (pageable) numpy array allocated on the GPU's NUMA node: chunks are staged through a page-locked "
                                "ring by a pool of copy threads (non-temporal stores)"},
        "gpu_launches": int(launches_timed),
        "roofline": {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom_gbs, "peak": peak, "unit": "GB/s", "frac": dom_gbs / peak,
                     "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms_per_launch": dom["ms"],
                     "kernel_share_of_step": dom["ms"] / step_ms,
                     "note": "dominant kernel by share of the step (CUDA events between the kernels inside the timed region), on SURVEY.md "
                             "8(d)'s bytes: one read of every raw 1024x1024 uint16 frame per step; kernels[] lists every stage with the "
                             "bytes it has to touch itself (own_*)",
                     "pipeline": {"achieved": pipe_gbs, "frac": pipe_gbs / peak,
                                  "what": "whole step: device-resident frames/s per GPU x 2 097 152 B (SURVEY.md 8(d)) / peak"},
                     "kernels": ktable},
        "clocks": clk,
    }
    if cpu_base is not None:
        out["cpu_baseline"] = cpu_base
    if world == 1:
        # ---- the per-frame fallback workload: 5 % of the frames carry hot pixels (the reference median-filters them)
        try:
            rng = np.random.default_rng(1)
            mixed = np.array(pageable, copy=True)
            for i in rng.choice(n, max(1, n // 20), replace=False):
                f = mixed[i] // 2
                f.ravel()[rng.integers(0, f.size, 40)] = 65535
                mixed[i] = f
            mb = nat.Batch.upload(ctx, mixed)
            nat.pf_bench_timed(ctx, mb, params, 2)
            msteps = args.steps
            # every step of this workload has a host round trip (deferred count -> re-run): three repetitions, the fastest one is
            # reported (all three are listed: the spread is host scheduling, not the device)
            ex0 = ctx.counter(nat.CTR_PF_EXACT_FRAMES)
            reps = [nat.pf_bench_timed(ctx, mb, params, msteps) for _ in range(3)]
            exact = (ctx.counter(nat.CTR_PF_EXACT_FRAMES) - ex0) / (3 * msteps)
            mt, _, mlaunch, redone = min(reps, key=lambda r: r[0])
            mb.free()
            out["config"]["mixed_noisy_5pct"] = {
                "workload": f"the same batch with {max(1, n // 20)} of {n} frames carrying 40 hot pixels (noise filter: certified-noise "
                            "re-run by the fast pipeline on a second stream while the batch's window stages run; exact pipeline only "
                            "for frames that cannot be certified)",
                "ms_per_step": mt / msteps, "value": n * msteps / (mt * 1e-3), "ratio_to_clean_step": (mt / msteps) / step_ms,
                "frames_rerun_per_step": redone / msteps, "frames_exact_pipeline_per_step": exact,
                "gpu_launches_per_step": mlaunch / msteps, "ms_per_step_all_repetitions": [r[0] / msteps for r in reps]}
            del mixed
        except Exception as e:  # pragma: no cover
            out["config"]["mixed_noisy_5pct"] = {"error": repr(e)}
        if not args.no_modules:
            batch.free()
            del pinned
            try:
                out["modules"] = bench_modules(ctx, nat, peak, cores)
            except Exception as e:  # pragma: no cover
                out["modules"] = {"error": repr(e)}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res.summary, res.meas)
    print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
