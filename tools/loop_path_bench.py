"""ms per reverse step of the per-step path (`GaussianDiffusion._step`: eager launches, fresh outputs, the fp32 model output
and a separate split pass) against the fused loop (`_fused_loop`, graph-replayed) on the chains that took the per-step path
before the fused loop learned clamp gating and progressive loops:

  clamp256  clamp-gated DDPM, B = 256, L = 2096: 6 rounding steps from the top of the 2000-step table, then 6 plain ones
  clamp4    the same chain at B = 4
  prog4     p_sample_loop_progressive at B = 4 (every step yields sample, pred_xstart, greedy_mean and the variances)

The two paths are timed in the same process, alternating, `--rounds` times each; every timed chain ends in a device
synchronise.  The per-step driver below is the per-step branch of `_loop`.
python tools/loop_path_bench.py [--rounds 5] [--only clamp4,prog4]"""
import argparse, json, os, subprocess, sys, time
from functools import partial
from types import SimpleNamespace
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from musediffusion_b200 import _lib
from musediffusion_b200.initialization import create_model_and_diffusion
from musediffusion_b200.rounding import denoised_fn_round
from musediffusion_b200.sample import build_model_emb
from musediffusion_b200.synthetic import make_synthetic_batch

ap = argparse.ArgumentParser()
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--only", default="clamp256,clamp4,prog4")
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("loop_path_bench.py measures on a CUDA device; none is visible")
dev = torch.device("cuda:0")
T, L, STEPS, CLAMP = 2000, 2096, 12, 1994            # indices 1999..1988; rounding at i >= 1994, plain below


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


print(json.dumps({"card": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": power_limit(), "seq_len": L}),
      flush=True)
targs = SimpleNamespace(hidden_dim=128, hidden_t_dim=128, vocab_size=729, seq_len=L, dropout=0.1, noise_schedule="sqrt",
                        diffusion_steps=T, timestep_respacing="", rescale_timesteps=True, predict_xstart=True)
torch.manual_seed(0)
model, diffusion = create_model_and_diffusion(targs)
model.eval().requires_grad_(False).to(dev)
fn = partial(denoised_fn_round, build_model_emb(model, dev), dist=None)


def setup(B):
    c = make_synthetic_batch("modification", B, L, seed=105)
    x_start = model.get_embeds(torch.from_numpy(c["input_ids"]).to(dev))
    mask = torch.broadcast_to(torch.from_numpy(c["input_mask"]).to(dev).unsqueeze(-1), x_start.shape)
    x = diffusion.q_sample(x_start.unsqueeze(-1), torch.full((B, 1), T - 1, device=dev), mask=mask).squeeze(-1)
    return SimpleNamespace(x=x, x_start=x_start, mask=mask)


def per_step(s, clamp_step, progressive):
    """the per-step branch of `_loop` for our denoiser (D = 128: the bf16 copy needs no pad columns)."""
    indices = list(range(T))[::-1][:STEPS]
    t_idx = torch.tensor(indices, dtype=torch.int32, device=dev)
    t_model = diffusion._model_timesteps(t_idx.long()).float()
    x, x_bf16 = s.x, None
    diffusion._noise_calls = 0
    for k, i in enumerate(indices):
        mo = model.denoise(x, t_model[k:k + 1], x_bf16=x_bf16, uniform_t=True)
        x_bf16 = torch.empty_like(x, dtype=torch.bfloat16)
        x, pred, mean = diffusion._step(_lib.STEP_DDPM, model, x, t_idx[k:k + 1], True, fn if i >= clamp_step else None, None,
                                        1, s.mask, s.x_start, 0.0, want_aux=progressive, model_output=mo, out_bf16=x_bf16)
        if progressive:                                   # what p_sample_loop_progressive yields for the step
            step_out = {"sample": x, "pred_xstart": pred, "greedy_mean": mean,
                        "out": diffusion._mean_variance(mean, pred, t_idx[k:k + 1], x.shape)}
    return x


def fused(s, clamp_step, progressive):
    diffusion._noise_calls = 0
    kw = dict(noise=s.x, denoised_fn=fn, top_p=1, clamp_step=clamp_step, clamp_first=True, mask=s.mask, x_start=s.x_start,
              t_enc=STEPS)
    if progressive:
        for out in diffusion.p_sample_loop_progressive(model, tuple(s.x.shape), **kw):
            pass
        return out["sample"]
    return diffusion.p_sample_loop(model, tuple(s.x.shape), only_last=True, **kw)[-1]


def timed(f, *args):
    torch.cuda.synchronize()
    tic = time.perf_counter()
    f(*args)
    torch.cuda.synchronize()
    return (time.perf_counter() - tic) / STEPS * 1e3


WORKLOADS = {"clamp256": (256, CLAMP, False), "clamp4": (4, CLAMP, False), "prog4": (4, 0, True)}
for name in a.only.split(","):
    B, clamp_step, progressive = WORKLOADS[name]
    s = setup(B)
    same = torch.equal(per_step(s, clamp_step, progressive), fused(s, clamp_step, progressive))   # warm-up of both
    times = {"per_step": [], "fused_graph": []}
    for _ in range(a.rounds):
        times["per_step"].append(timed(per_step, s, clamp_step, progressive))
        times["fused_graph"].append(timed(fused, s, clamp_step, progressive))
    med = {k: float(np.median(v)) for k, v in times.items()}
    print(json.dumps({"workload": name, "batch": B, "steps": STEPS, "clamp_step": clamp_step, "progressive": progressive,
                      "ms_per_step_median": med, "ms_per_step_all": times,
                      "per_step_over_fused": med["per_step"] / med["fused_graph"], "warmup_outputs_equal": same}), flush=True)
    del s
    torch.cuda.empty_cache()
