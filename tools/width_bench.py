"""Fused reverse-step time at several embedding widths D (hidden_dim), at the bench's token count.

    python tools/width_bench.py [--widths 128,500,512] [--seq-len 256] [--tokens 536576] [--steps 8] [--rounds 3]

Workload: the base encoder (bert-base sizes) with random weights, modification mode, DDPM with rounding every step, the
CUDA-graph loop the samplers use; B = tokens / L sequences of length L (default 2096 x 256 = 256 x 2096 tokens, one encoder
pass).  A width that is not a multiple of 64 runs its tensor-core operands padded to Dp = round_up(D, 64), so D = 500 and
D = 512 run the same GEMM and rounding shapes; what differs is the elementwise work on the D-wide fp32 state (D = 128 has
a warp-per-row posterior kernel, other widths the generic one).

Per width and round: a chain of `warmup` steps and one of `warmup + steps` steps from the same state, timed with CUDA
events; the difference over `steps` is the steady-state step time (it excludes the eager first step and the capture).
The widths alternate inside every round.  Then one eager step per width under `ops.profile_step` gives the per-kernel
breakdown (CUDA events around every launch; a separate pass, the profiler slows the host).  Prints the card name and power
limit, then one JSON line per width.  Writes nothing."""
import argparse
import json
import os
import subprocess
import sys
from functools import partial
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from musediffusion_b200 import _lib, ops  # noqa: E402
from musediffusion_b200.initialization import create_model_and_diffusion  # noqa: E402
from musediffusion_b200.rounding import denoised_fn_round  # noqa: E402
from musediffusion_b200.sample import build_model_emb  # noqa: E402
from musediffusion_b200.synthetic import make_synthetic_batch  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--widths", default="128,500,512")
ap.add_argument("--seq-len", type=int, default=256)
ap.add_argument("--tokens", type=int, default=256 * 2096)
ap.add_argument("--steps", type=int, default=8)
ap.add_argument("--warmup", type=int, default=4)
ap.add_argument("--rounds", type=int, default=3)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("width_bench.py measures on a CUDA device; none is visible")
dev = torch.device("cuda:0")
T, L = 2000, a.seq_len
B = a.tokens // L
widths = [int(w) for w in a.widths.split(",")]


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


print(json.dumps({"card": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": power_limit(),
                  "seq_len": L, "sequences": B, "tokens": B * L}), flush=True)

cond = make_synthetic_batch("modification", B, L, seed=105)
setups = {}
for D in widths:
    targs = SimpleNamespace(hidden_dim=D, hidden_t_dim=128, vocab_size=729, seq_len=L, dropout=0.1, noise_schedule="sqrt",
                            diffusion_steps=T, timestep_respacing="", rescale_timesteps=True, predict_xstart=True)
    torch.manual_seed(D)
    model, diffusion = create_model_and_diffusion(targs)
    model.eval().requires_grad_(False).to(dev)
    emb = build_model_emb(model, dev)
    ids = torch.from_numpy(cond["input_ids"]).to(dev)
    x_start = model.get_embeds(ids)
    mask = torch.broadcast_to(torch.from_numpy(cond["input_mask"]).to(dev).unsqueeze(-1), x_start.shape)
    x0 = diffusion.q_sample(x_start.unsqueeze(-1), torch.full((B, 1), T - 1, device=dev), mask=mask).squeeze(-1)
    setups[D] = (model, diffusion, partial(denoised_fn_round, emb, dist=None), x_start, mask, x0)


def chain(D, n):
    model, diffusion, fn, x_start, mask, x0 = setups[D]
    return diffusion.p_sample_loop(model, tuple(x0.shape), noise=x0, denoised_fn=fn, model_kwargs={}, top_p=1, clamp_step=0,
                                   clamp_first=True, mask=mask, x_start=x_start, t_enc=n, only_last=True)


def timed_chain(D, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    chain(D, n)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


for D in widths:                    # warm every shape: module loads, tensor maps, graph pools
    timed_chain(D, a.warmup)
step_ms = {D: [] for D in widths}
for _ in range(a.rounds):
    for D in widths:
        short, long_ = timed_chain(D, a.warmup), timed_chain(D, a.warmup + a.steps)
        step_ms[D].append((long_ - short) / a.steps)

for D in widths:
    model, diffusion, fn, x_start, mask, x0 = setups[D]
    diffusion.use_cuda_graph = False
    gen = diffusion._loop(_lib.STEP_DDPM, model, tuple(x0.shape), x0, True, fn, None, dev, False, 1, 0, True, mask, x_start,
                          0.0, list(range(T))[::-1][:4], want_aux=False)
    next(gen)                                                       # one-time set-up outside the profile
    kernels = {}
    for _ in range(3):
        for name, detail, ms in ops.profile_step(lambda: next(gen)):
            key = name + (" " + detail if detail else "")
            kernels[key] = kernels.get(key, 0.0) + ms / 3
    diffusion.use_cuda_graph = True
    print(json.dumps({"D": D, "Dp": ops.padded_width(D), "step_ms_median": float(np.median(step_ms[D])),
                      "step_ms_rounds": [round(v, 3) for v in step_ms[D]],
                      "kernels_ms_per_step": {k: round(v, 4) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1])}}),
          flush=True)
