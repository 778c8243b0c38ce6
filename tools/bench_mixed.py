"""The per-frame fallback workload of bench.py (`mixed_noisy_5pct`) on its own: 512 frames, 25 of them with hot pixels; clean step,
mixed step and the per-stage event times of both."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from pylinac_b200 import _native as nat
from pylinac_b200 import picketfence as pf
from oracle import synth

n = 512
uniq = np.stack([synth.bench_pf_frame(i) for i in range(16)])
frames = np.concatenate([uniq] * (n // 16))
ctx = nat.Context.default(0)
params = pf.make_params(2.56, (1024, 1024))
b = nat.Batch.upload(ctx, frames)
nat.pf_bench_timed(ctx, b, params, 3)
t, st, l, r = nat.pf_bench_timed(ctx, b, params, 10)
print(f"clean: {t / 10:.3f} ms/step, launches {l / 10:.0f}, redone {r}")
rng = np.random.default_rng(1)
mixed = frames.copy()
for i in rng.choice(n, n // 20, replace=False):
    f = mixed[i] // 2
    f.ravel()[rng.integers(0, f.size, 40)] = 65535
    mixed[i] = f
mb = nat.Batch.upload(ctx, mixed)
for fast_redo in (0, 1):
    ctx.set_option(nat.OPT_PF_FAST_REDO, fast_redo)
    nat.pf_bench_timed(ctx, mb, params, 2)
    for rep in range(3):
        e0 = ctx.counter(nat.CTR_PF_EXACT_FRAMES)
        t, st, l, r = nat.pf_bench_timed(ctx, mb, params, 10)
        print(f"mixed fast_redo={fast_redo}: {t / 10:.3f} ms/step, launches {l / 10:.0f}, redone/step {r / 10:.0f}, "
              f"exact/step {(ctx.counter(nat.CTR_PF_EXACT_FRAMES) - e0) / 10:.0f}; stages(us): " +
              ", ".join(f"{k.split(' ')[0]} {v * 1e3:.0f}" for k, v in st.items() if v > 0))
