#!/usr/bin/env python
"""Per-stage device times of the PicketFence pipeline on the bench workload (512 synthetic frames), for the window-path variants.
usage: python tools/r2_stages.py [--frames 512] [--win2 0|1] [--iters 5] [--mixed PCT]"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--win2", type=int, default=1)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--mixed", type=float, default=0.0, help="percent of frames with hot pixels (noise filter -> per-frame exact re-run)")
    ap.add_argument("--unique", type=int, default=32)
    a = ap.parse_args()
    from oracle import synth
    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    base = np.stack([synth.bench_pf_frame(i) for i in range(a.unique)])
    frames = np.ascontiguousarray(base[np.arange(a.frames) % a.unique])
    if a.mixed > 0:
        rng = np.random.default_rng(1)
        k = max(1, int(round(a.frames * a.mixed / 100.0)))
        for i in rng.choice(a.frames, k, replace=False):
            f = frames[i] // 2
            f.ravel()[rng.integers(0, f.size, 40)] = 65535
            frames[i] = f
    ctx = nat.Context.default()
    ctx.set_option(nat.OPT_PF_WIN2, a.win2)
    params = pf.make_params(2.56, frames.shape[1:])
    b = nat.Batch.upload(ctx, frames)
    nat.pf_bench(ctx, b, params, 3)
    total, stream_ms, launches = nat.pf_bench(ctx, b, params, a.iters)
    st = nat.pf_bench_stages(ctx, b, params, a.iters)
    out = {"frames": a.frames, "win2": a.win2, "mixed_pct": a.mixed, "ms_per_step": total / a.iters,
           "fps": a.frames * a.iters / (total * 1e-3), "launches_per_step": launches / a.iters,
           "redone": ctx.counter(nat.CTR_PF_REDONE_FRAMES), "stages_ms": {k: round(v, 4) for k, v in st.items() if v > 0}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
