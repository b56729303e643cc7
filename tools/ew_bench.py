"""Times the HBM-bound kernels at the bench shape with CUDA events: python tools/ew_bench.py [B]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import json
import torch
from musediffusion_b200 import _lib, ops
from musediffusion_b200.diffusion import SpacedDiffusion, get_named_beta_schedule, space_timesteps

B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
L, D, V, H = 2096, 128, 729, 768
M = B * L
dev = torch.device("cuda")
pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
peak = json.load(open(pk))["hbm_gbs"] if os.path.exists(pk) else 6548.2
d = SpacedDiffusion(use_timesteps=space_timesteps(2000, [2000]), betas=get_named_beta_schedule("sqrt", 2000), rescale_timesteps=True, predict_xstart=True)
d._upload_schedule()
x = torch.randn(B, L, D, device=dev); xs = torch.randn(B, L, D, device=dev); out = torch.empty_like(x)
xb = torch.empty(B, L, D, device=dev, dtype=torch.bfloat16)
E = torch.randn(V, D, device=dev); idx = torch.randint(0, V, (M,), device=dev, dtype=torch.int32)
t = torch.tensor([1500], device=dev, dtype=torch.int32)
mask = (torch.rand(B, L, device=dev) > 0.02).to(torch.int32).unsqueeze(-1).expand(B, L, D)
noise = torch.randn(B, L, D, device=dev)
h = torch.randn(M, H, device=dev).to(torch.bfloat16); r = torch.randn(M, H, device=dev).to(torch.bfloat16); ho = torch.empty_like(h)
g = torch.ones(H, device=dev); bt = torch.zeros(H, device=dev)


def timeit(fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def rep(name, ms, nbytes):
    print("%-42s %8.3f ms  %7.1f GB/s  %.1f%% of measured HBM peak (%.0f GB/s)" % (name, ms, nbytes / ms / 1e6, 100 * nbytes / ms / 1e6 / peak, peak))


ms = timeit(lambda: ops.posterior_step(x, t, _lib.STEP_DDPM, idx=idx, E=E, seed=1, step_counter=3, mask=mask, x_start=xs, top_p=1.0, out=out, out_bf16=xb))
rep("posterior DDPM philox top_p=1 (+bf16 copy)", ms, M * (512 + 4 + 512 + 256))
Ec = ops.SplitEmbedding(E).E_clamped
ms = timeit(lambda: ops.posterior_step(x, t, _lib.STEP_DDPM, idx=idx, E=Ec, seed=1, step_counter=3, mask=mask, x_start=xs, top_p=1.0, clip=2, out=out, out_bf16=xb))
rep("  ... gathering pre-clamped rows (the loop's path)", ms, M * (512 + 4 + 512 + 256))
ms = timeit(lambda: ops.posterior_step(x, t, _lib.STEP_DDPM, idx=idx, E=E, noise=noise, mask=mask, x_start=xs, out=out, out_bf16=xb))
rep("posterior DDPM external noise", ms, M * (512 + 4 + 512 + 512 + 256))
ms = timeit(lambda: ops.posterior_step(x, t, _lib.STEP_DDIM, idx=idx, E=E, seed=1, step_counter=3, mask=mask, x_start=xs, out=out, out_bf16=xb))
rep("posterior DDIM eta=0 (sigma 0: no draws)", ms, M * (512 + 4 + 512 + 256))
# the general quantile (top_p = 0 or > 1): DDPM with top_p > 1, DDIM with eta > 0, the generation-mode initial noise
ms = timeit(lambda: ops.posterior_step(x, t, _lib.STEP_DDPM, idx=idx, E=E, seed=1, step_counter=3, mask=mask, x_start=xs, top_p=2.0, out=out, out_bf16=xb))
rep("posterior DDPM philox top_p=2 (general)", ms, M * (512 + 4 + 512 + 256))
ms = timeit(lambda: ops.posterior_step(x, t, _lib.STEP_DDIM, idx=idx, E=E, seed=1, step_counter=3, mask=mask, x_start=xs, eta=0.5, out=out, out_bf16=xb))
rep("posterior DDIM philox eta=0.5 (general)", ms, M * (512 + 4 + 512 + 256))
ms = timeit(lambda: ops.fill_normal((B, L, D), dev, seed=1, step_counter=3))
rep("fill_normal untruncated (general)", ms, M * D * 4)
ms = timeit(lambda: ops.layernorm(h, g, bt, 1e-12, resid=r, out=ho))
rep("layernorm(x + resid) bf16", ms, M * H * 2 * 3)
ms = timeit(lambda: ops.round_argmin(x, E))
print("%-42s %8.3f ms  %.1f TFLOP/s fp32" % ("round_argmin", ms, 2.0 * M * V * D / ms / 1e9))
se = ops.SplitEmbedding(E)
ms = timeit(lambda: ops.round_argmin_tc(x, se))
print("%-42s %8.3f ms  %.1f TFLOP/s (4 x 2MVD split-bf16)  %.1f%% of HBM peak on %d algorithmic bytes/token" % ("round_argmin_tc", ms, 8.0 * M * 768 * D / ms / 1e9, 100 * M * 516 / ms / 1e6 / peak, 516))

# ---- SURVEY section 8(f) row 1: batched token-level decode (one warp per row) against the CPU port of the reference's
# per-row Python (the checker under oracle/, timed on a bounded sample of the same rows)
import time
import numpy as np
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import decode_oracle as DO
from musediffusion_b200.synthetic import make_synthetic_batch
cond = make_synthetic_batch("modification", B, L, seed=7)
rows = cond["input_ids"].copy()
for b in range(B):                      # keep roughly as many BARs as chord bars so that most rows take the full path
    n0 = int((cond["input_mask"][b] == 0).sum())
    n_cb = int((rows[b, 11:n0 - 1] == 432).sum())
    bars = np.nonzero(rows[b, n0:] == 2)[0] + n0
    rows[b, bars[n_cb:]] = 3
tok_d = torch.from_numpy(rows).to(dev).to(torch.int32)
msk_d = torch.from_numpy(cond["input_mask"]).to(dev).to(torch.int32)
ms = timeit(lambda: ops.decode_prepare(tok_d, msk_d, True))
st = ops.decode_prepare(tok_d, msk_d, True)[0].cpu().numpy()
n_cpu = min(B, 32)
t0 = time.perf_counter()
want = DO.decode_prepare_batch(rows[:n_cpu], cond["input_mask"][:n_cpu], True)
cpu_ms = (time.perf_counter() - t0) * 1e3 / n_cpu
print("%-42s %8.3f ms for %d rows (%.2f us/row; %d OK)   CPU port %.2f ms/row on 1 core   status parity on the sample: %s"
      % ("decode_prepare strict (L=%d)" % L, ms, B, ms * 1e3 / B, int((st == 0).sum()), cpu_ms, bool((want[0] == st[:n_cpu]).all())))
