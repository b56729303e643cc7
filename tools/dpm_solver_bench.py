"""DPM-Solver++(2M) at the base config (B = 256, L = 2096, D = 128, 2000-step sqrt table), in one process:

  kernel   md_dpm_solver_step alone as the fused loop calls it (ids gathered from clamp(E, -1, 1), token mask, bf16 copy,
           a second-order row selected by the cursor, x_out = x_t), CUDA events around --launches back-to-back launches,
           eager and as replays of a captured graph of 20 launches (no host overhead), and md_posterior_step (DDIM) the same
           way for comparison;
           GB/s from the bytes the step must move per token: x_t, history read and write, x_out (4 x 512 B), bf16 copy
           256 B, id and mask 4 B each = 2312 B, 1.24 GB per launch.  The state, history and bf16 copy (0.69 GB) are far
           larger than the 126 MB L2, so every launch streams from HBM.
  step     ms per evaluation of the graph-replayed DPM body and DDIM body (ddim_sample_loop, gap 1) in this process,
           alternating, --rounds times: the time of a 12-evaluation chain minus a 4-evaluation chain over 8, so set-up and
           capture cancel.
  e2e      sequences/s of sample_batch(sampler="dpm_solver++") in modification mode at strength 1 (the whole chain) for
           N = 10, 20, 50 evaluations, every call ending in a device synchronise.

Weights are the model's own random initialisation: the timing does not depend on them, and sample quality is not
measured here.  Card name and power limit are read in the same call.
python tools/dpm_solver_bench.py [--batch 256] [--rounds 3] [--launches 200] [--out profiles/dpm_solver_bench.json]"""
import argparse
import json
import os
import subprocess
import sys
import time
from functools import partial
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from musediffusion_b200 import ops  # noqa: E402
from musediffusion_b200.diffusion import dpm_solver_coefficients, dpm_solver_indices  # noqa: E402
from musediffusion_b200.initialization import create_model_and_diffusion  # noqa: E402
from musediffusion_b200.rounding import denoised_fn_round  # noqa: E402
from musediffusion_b200.sample import build_model_emb, sample_batch  # noqa: E402
from musediffusion_b200.synthetic import make_synthetic_batch  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--launches", type=int, default=200)
ap.add_argument("--evals", default="10,20,50")
ap.add_argument("--out", default=None, help="also write the records to this JSON file")
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("dpm_solver_bench.py measures on a CUDA device; none is visible")
dev = torch.device("cuda:0")
T, L, D, B = 2000, 2096, 128, a.batch
records = []


def emit(rec):
    records.append(rec)
    print(json.dumps(rec), flush=True)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


emit({"card": torch.cuda.get_device_name(dev), "name_power_limit_max_sm_clock": card(), "batch": B, "seq_len": L, "D": D,
      "diffusion_steps": T})
targs = SimpleNamespace(hidden_dim=D, hidden_t_dim=128, vocab_size=729, seq_len=L, dropout=0.1, noise_schedule="sqrt",
                        diffusion_steps=T, timestep_respacing="", rescale_timesteps=True, predict_xstart=True)
torch.manual_seed(0)
model, diffusion = create_model_and_diffusion(targs)
model.eval().requires_grad_(False).to(dev)
model_emb = build_model_emb(model, dev)
fn = partial(denoised_fn_round, model_emb, dist=None)
cond = make_synthetic_batch("modification", B, L, seed=105)
tcond = {k: torch.from_numpy(v) for k, v in cond.items()}
x_start = model.get_embeds(tcond["input_ids"].to(dev))
mask = torch.broadcast_to(tcond["input_mask"].to(dev).unsqueeze(-1), x_start.shape)

# ---- kernel alone
M = B * L
x = torch.randn((B, L, D), device=dev)
hist = torch.randn((B, L, D), device=dev)
xb = torch.empty((B, L, D), dtype=torch.bfloat16, device=dev)
se = ops.split_embedding(model_emb.weight)
ids = torch.randint(0, se.V, (M,), dtype=torch.int32, device=dev)
m32 = tcond["input_mask"].to(dev).to(torch.int32).contiguous().unsqueeze(-1).expand(B, L, D)
ab = diffusion.alphas_cumprod
coef = torch.from_numpy(dpm_solver_coefficients(ab, dpm_solver_indices(ab, T - 1, 20), 2).astype(np.float32)).to(dev)
cursor = torch.tensor([6], dtype=torch.int32, device=dev)          # row 5: second order, the history is read


def kernel():
    ops.dpm_solver_step(x, coef, hist, idx=ids, E=se.E_clamped, clip=2, cursor=cursor, mask=m32, x_start=x_start, out=x,
                        out_bf16=xb)


t_cur = torch.tensor([1500], dtype=torch.int32, device=dev)


def posterior():
    """md_posterior_step as the DDIM loop calls it (same gather, mask and bf16 copy; no history): the point of comparison"""
    ops.posterior_step(x, t_cur, 1, idx=ids, E=se.E_clamped, clip=2, seed=1, step_counter=3, mask=m32, x_start=x_start, out=x,
                       out_bf16=xb)


def events(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


bytes_per_token = 4 * 4 * D + 2 * D + 4 + 4
diffusion._upload_schedule()
for name, launch, nbytes in (("md_dpm_solver_step", kernel, bytes_per_token), ("md_posterior_step DDIM", posterior, 2 * 512 + 256 + 8)):
    for _ in range(10):
        launch()
    torch.cuda.synchronize()
    eager = events(launch, a.launches)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        g.capture_begin()
        for _ in range(20):
            launch()
        g.capture_end()
    torch.cuda.current_stream().wait_stream(side)
    replay = events(g.replay, max(1, a.launches // 20)) / 20
    emit({"what": name + " alone", "launches": a.launches, "ms_per_launch_eager": eager, "ms_per_launch_graph": replay,
          "bytes_per_token": nbytes, "GB": M * nbytes / 1e9, "GB_per_s_graph": M * nbytes / (replay * 1e-3) / 1e9})
    del g
del x, hist, xb, ids
torch.cuda.empty_cache()

# ---- ms per evaluation: DPM body against DDIM body, alternating
x0 = diffusion.q_sample(x_start.unsqueeze(-1), torch.full((B, 1), T - 1, device=dev), mask=mask).squeeze(-1).clone()
common = dict(noise=x0, denoised_fn=fn, model_kwargs={}, mask=mask, x_start=x_start, only_last=True)


def chain(kind, n):
    torch.cuda.synchronize()
    tic = time.perf_counter()
    if kind == "dpm":
        diffusion.dpm_solver_sample_loop(model, tuple(x0.shape), steps=n, t_start=T - 1, **common)
    else:
        diffusion.ddim_sample_loop(model, tuple(x0.shape), gap=1, eta=0.0, t_enc=n, **common)
    torch.cuda.synchronize()
    return (time.perf_counter() - tic) * 1e3


for kind in ("dpm", "ddim"):
    chain(kind, 4)                                           # warm-up of every shape and the capture path
per_eval = {"dpm": [], "ddim": []}
for _ in range(a.rounds):
    for kind in ("dpm", "ddim"):
        short, long_ = chain(kind, 4), chain(kind, 12)
        per_eval[kind].append((long_ - short) / 8)
med = {k: float(np.median(v)) for k, v in per_eval.items()}
emit({"what": "ms per evaluation, graph-replayed body, (t(12) - t(4)) / 8", "median": med, "all": per_eval,
      "dpm_over_ddim": med["dpm"] / med["ddim"]})

# ---- sequences/s end to end through sample_batch
sample_batch(model, diffusion, model_emb, tcond, "modification", 4, T, strength=1.0, sampler="dpm_solver++")
for n in (int(v) for v in a.evals.split(",")):
    torch.cuda.synchronize()
    tic = time.perf_counter()
    tok = sample_batch(model, diffusion, model_emb, tcond, "modification", n, T, strength=1.0, sampler="dpm_solver++")
    torch.cuda.synchronize()
    sec = time.perf_counter() - tic
    emit({"what": "sample_batch(sampler='dpm_solver++'), modification, strength 1", "evaluations": n, "seconds": sec,
          "sequences_per_s": B / sec, "tokens_shape": list(tok.shape)})
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(records, f, indent=1)
