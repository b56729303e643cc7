#!/usr/bin/env python
"""Benchmark of the B200-native MuseDiffusion sampling path (BASELINE.json metric: sequences/sec of full
reverse-diffusion sampling; ms per denoiser step).

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU under torchrun for N > 1)
  python bench.py --impl reference --steps K --warmup W    the UNMODIFIED reference's CPU path (oracle/_ref via oracle/ref_harness.py)
                                                            on the host cores; the numpy port if that tree is absent
  python bench.py --mode generation --batch 128            BASELINE.json configs[2] (unconditional generation path)
  python bench.py --steps K --dump-outputs DIR             also writes what the last timed step computed (dump_outputs)

Workload (config 2 of BASELINE.json): base TransformerNetModel (bert-base encoder, seq_len 2096, hidden_dim 128,
vocab 729), random-init weights, synthetic ComMU-shaped modification batch, 256 sequences per GPU, DDPM chain of
2000 steps with rounding every step (top_p = 1 truncated noise), bf16 denoiser, fp32 state.
A bench "step" = ONE reverse-diffusion step of the chain over the whole batch (denoiser forward + nearest-embedding
rounding + fused posterior update) — every step of the chain launches the same kernels on the same shapes, so
`value` = sequences / (ms_per_step * 2000 + decode) is the full-chain throughput extrapolated from K consecutive
chain steps starting at t = 1999 (`--full-chain` runs all 2000 instead).  `e2e` is measured through the public API
(`sample_batch`: pinned host token ids in, decoded token ids out to host) running K chain steps via the reference's
own `t_enc` argument, host<->device copies inside the timed region, scaled the same way."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DIFFUSION_STEPS = 2000
L, D, V, H, F, NL, NH = 2096, 128, 729, 768, 3072, 12, 12


def set_model_shape(args):
    """--scaled switches to BASELINE.json config 5 (bert-large-shaped denoiser, 2x seq_len); individual flags override."""
    global L, H, F, NL, NH
    if args.scaled:
        L, H, F, NL, NH = 4192, 1024, 4096, 24, 16
    L = args.seq_len or L
    H = args.hidden or H
    F = args.ffn or F
    NL = args.layers or NL
    NH = args.heads or NH


def flops_per_sequence_step():
    """SURVEY.md section 8(d): L * [2(2DH + 2H^2) + NL(8H^2 + 4HF + 4LH) + 2VD]."""
    return L * (2 * (2 * D * H + 2 * H * H) + NL * (8 * H * H + 4 * H * F + 4 * L * H) + 2 * V * D)


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_burst": float(p["bf16_tflops"]),
                "bf16_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "source": "fallback"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw,power.limit")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [s.strip() for s in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(float(s[0])) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons,
               "samples": len(sm)}
        try:                                                    # board power next to its limit: the step runs AT the cap
            watts = sorted(float(s[6]) for s in self.samples if len(s) >= 8)
            out["power_w"], out["power_limit_w"] = watts[len(watts) // 2], float(self.samples[0][7])
        except (ValueError, IndexError):
            pass
        return out


# ------------------------------------------------------------------------------------------------ reference arm
def _reference_sampler():
    """The UNMODIFIED reference (oracle/_ref copy on the GPU box, /root/reference in the build container) on the host CPU,
    or None when neither tree is present (then the numpy port of oracle/ is the CPU arm)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import ref_harness
        if not ref_harness.available():
            return None
        return ref_harness.ReferenceSampler(seq_len=L, diffusion_steps=DIFFUSION_STEPS, seed=0)
    except Exception as exc:                                    # noqa: BLE001 - fall back to the port, but say why
        print("bench: reference import failed (%s: %s); using the numpy port" % (type(exc).__name__, exc), file=sys.stderr)
        return None


def time_reference_cpu(mode, B, warmup, steps):
    """BASELINE.md section 3: the reference's own `sample_fn(...)` + `get_logits` + `argmax` (run/sample.py:200-220), fp32,
    all host threads, on B synthetic sequences of the workload; the chain is cut to `steps` reverse steps through the
    reference's own t_enc argument (every step of the chain costs the same) and extrapolated to 2000.
    Returns (seconds per reverse step, kind, threads, description)."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import musediff_oracle as O
    cond = O.make_synthetic_batch(mode, B, L, seed=105)
    ref = _reference_sampler() if (L, H, F, NL, NH) == (2096, 768, 3072, 12, 12) else None
    if ref is not None:
        import torch
        tcond = {k: torch.from_numpy(np.asarray(v)) for k, v in cond.items()}
        torch.manual_seed(105)
        if warmup > 0:
            ref.sample(tcond, mode, DIFFUSION_STEPS, strength=1.0, top_p=1, n_steps=warmup)
        tic = time.perf_counter()
        ref.sample(tcond, mode, DIFFUSION_STEPS, strength=1.0, top_p=1, n_steps=steps)
        per_step = (time.perf_counter() - tic) / steps
        return per_step, "reference", ref.threads, (
            "unmodified MuseDiffusion p_sample_loop + denoised_fn_round + get_logits/argmax (run/sample.py:177-220) via "
            "oracle/ref_harness.py, fp32 torch CPU, %d threads: %d sequences x %d chain steps (t_enc), %.2f s/step, "
            "extrapolated to the 2000-step chain" % (ref.threads, B, steps, per_step))
    p = O.make_random_params(seed=0, seq_len=L)
    s = O.make_schedule("sqrt", DIFFUSION_STEPS)
    x_start = O.get_embeds(p, cond["input_ids"])
    mask = np.broadcast_to(cond["input_mask"][..., None], x_start.shape)
    noise = O.NoiseStream(105)
    x = O.q_sample(s, x_start, np.full((B,), DIFFUSION_STEPS - 1), noise.randn(x_start.shape), mask)
    E = p["word_embedding.weight"]
    times = []
    for k in range(warmup + steps):
        t = np.full((B,), DIFFUSION_STEPS - 1 - k, dtype=np.int64)
        tic = time.perf_counter()
        mo = O.denoiser_forward(p, x, s.model_timestep(t))
        x = O.p_sample_step(s, x, t, mo, noise.truncated(x.shape, 1), E, True, mask, x_start)["sample"]
        times.append(time.perf_counter() - tic)
    per_step = sum(times[warmup:]) / steps
    return per_step, "port", os.cpu_count(), (
        "numpy port of the reference algorithm (oracle/musediff_oracle.py; reference tree not present): %d sequences x %d "
        "chain steps, %.2f s/step, extrapolated to the 2000-step chain" % (B, steps, per_step))


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores, on our arm's config /
    metric / unit; each step = one reverse step of the chain on a bounded sample (args.ref_batch sequences, BASELINE.md
    section 3 uses 4).  Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = args.ref_batch
    per_step, kind, threads, sample = time_reference_cpu(args.mode, B, args.warmup, args.steps)
    ms = 1e3 * per_step
    value = B / (per_step * DIFFUSION_STEPS)
    line = {"impl": "reference", "metric": "sequences/sec full reverse-diffusion sampling", "value": value,
            "unit": "sequences/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": workload_config(args.batch, args.gpus, mode=args.mode),
            "cpu_baseline": {"value": value, "unit": "sequences/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(batch_per_gpu, n_gpus, note=None, mode="modification"):
    base = (L, H, F, NL, NH) == (2096, 768, 3072, 12, 12)
    which = ("configs[1]" if mode == "modification" else "configs[2]") if base else "configs[4] family"
    c = {"workload": ("BASELINE.json %s: base TransformerNetModel (bert-base encoder 12x768, seq_len 2096, "
                      "hidden_dim 128, vocab 729)" % which if base else
                      "BASELINE.json configs[4] family: scaled denoiser (encoder %dx%d, %d heads, FFN %d, seq_len %d, "
                      "hidden_dim 128, vocab 729)" % (NL, H, NH, F, L)) +
                     " random-init; %s sampling, DDPM 2000 steps, "
                     "rounding every step, top_p=1; batch %d sequences per GPU"
                     % ("modification (seq2seq)" if mode == "modification" else "unconditional generation (sample_generation path)",
                        batch_per_gpu),
         "global_batch": batch_per_gpu * n_gpus, "seq_len": L, "chain_steps": DIFFUSION_STEPS,
         "parallelism": "dp%d (batch sharded by sequence, replicated weights, no collective in the loop)" % n_gpus,
         "step_definition": "one reverse-diffusion step over the whole batch; value extrapolated to the full chain",
         "l2_policy": "per-step working set (>10 GB of activations) far exceeds the 126 MB L2; no explicit flush"}
    if note:
        c["note"] = note
    return c


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import numpy as np
    import torch
    from types import SimpleNamespace
    from musediffusion_b200 import _lib, dist, ops
    from musediffusion_b200.initialization import create_model_and_diffusion, seed_all
    from musediffusion_b200.rounding import denoised_fn_round
    from musediffusion_b200.sample import build_model_emb, sample_batch
    from musediffusion_b200.synthetic import make_synthetic_batch
    from functools import partial

    rank, world, dev = dist.setup()
    B = args.batch
    targs = SimpleNamespace(hidden_dim=D, hidden_t_dim=128, vocab_size=V, seq_len=L, dropout=0.1, noise_schedule="sqrt",
                            diffusion_steps=DIFFUSION_STEPS, timestep_respacing="", rescale_timesteps=True,
                            predict_xstart=True,
                            encoder_config=dict(hidden_size=H, num_hidden_layers=NL, num_attention_heads=NH,
                                                intermediate_size=F))
    torch.manual_seed(0)
    model, diffusion = create_model_and_diffusion(targs)
    model.eval().requires_grad_(False).to(dev)
    dist.broadcast_model(model)                                   # NCCL: replicated weights (one-time)
    model_emb = build_model_emb(model, dev)
    seed_all(105, deterministic=True)
    diffusion.seq_offset = rank * B
    cond_np = make_synthetic_batch(args.mode, B, L, seed=105 + rank)
    cond_host = {k: torch.from_numpy(v).pin_memory() for k, v in cond_np.items() if k != "length"}
    fn = partial(denoised_fn_round, model_emb, dist=None)

    # ---- device-resident timed region: K consecutive chain steps through the loop generator
    ids = cond_host["input_ids"].to(dev)
    mask_ori = cond_host["input_mask"].to(dev)
    x_start = model.get_embeds(ids)
    mask = torch.broadcast_to(mask_ori.unsqueeze(-1), x_start.shape)
    if args.mode == "generation":                              # run/sample.py:190-193
        x_noised = ops.q_sample(x_start, None, seed=diffusion._seed(), step_counter=diffusion._next_counter(),
                                seq_offset=diffusion.seq_offset, mask=mask_ori)
    else:                                                      # run/sample.py:195-197
        x_noised = diffusion.q_sample(x_start.unsqueeze(-1), torch.full((B, 1), DIFFUSION_STEPS - 1, device=dev),
                                      mask=mask).squeeze(-1)
    model.decode_tokens(x_noised)                              # one-time set-up of the decode kernel (split embedding, attributes)
    n_total = DIFFUSION_STEPS if args.full_chain else args.warmup + args.steps
    gen = diffusion._loop(_lib.STEP_DDPM, model, tuple(x_start.shape), x_noised, True, fn, None, dev, False, 1, 0, True,
                          mask, x_start, 0.0, list(range(DIFFUSION_STEPS))[::-1][:n_total + 1], want_aux=False)
    sampler = ClockSampler(dev.index or 0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    last = None
    launches0 = 0
    timed_steps = n_total - args.warmup
    for k in range(n_total):
        if k == args.warmup:
            dist.barrier()
            torch.cuda.synchronize()
            sampler.start()
            launches0 = ops.launch_count()
            ev0.record()
        last = next(gen)
    ev1.record()
    torch.cuda.synchronize()
    dist.barrier()
    launches = ops.launch_count() - launches0
    ms_total = ev0.elapsed_time(ev1)
    # final decode (get_logits + argmax fused), once per batch
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record()
    tokens = model.decode_tokens(last[0])
    d1.record()
    torch.cuda.synchronize()
    sampler.stop_flag = True
    ms_decode = d0.elapsed_time(d1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last[0], tokens)
    t = torch.tensor([ms_total, ms_decode], device=dev, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms_total, ms_decode = float(t[0]), float(t[1])
    ms_step = ms_total / timed_steps
    value = (B * world) / ((ms_step * DIFFUSION_STEPS + ms_decode) * 1e-3)

    # ---- per-kernel breakdown of one step (CUDA events around every launch), dominant-kernel roofline
    peaks = load_peaks()
    prof = None
    if not args.full_chain and not args.no_breakdown and n_total + 4 <= DIFFUSION_STEPS:
        # CUDA events around every launch need the eager loop (the timed region above replays the captured step graph):
        # three more steps of the same chain, averaged, so that one step's clock wobble does not pick the dominant kernel
        saved, diffusion.use_cuda_graph = diffusion.use_cuda_graph, False
        gen_e = diffusion._loop(_lib.STEP_DDPM, model, tuple(x_start.shape), last[0], True, fn, None, dev, False, 1, 0, True,
                                mask, x_start, 0.0, list(range(DIFFUSION_STEPS))[::-1][n_total:n_total + 5], want_aux=False)
        next(gen_e)
        prof = ops.profile_step(lambda: [next(gen_e) for _ in range(3)])
        prof = [(n, d, ms / 3.0) for n, d, ms in prof]
        diffusion.use_cuda_graph = saved
    roofline, breakdown = None, None
    if prof:
        breakdown = summarize_profile(prof, B)
        top = max((v for v in breakdown.values() if v["flops"] > 0), key=lambda v: v["ms"])
        ach = top["flops"] / (top["ms"] * 1e-3) / 1e12
        roofline = {"kernel": top["name"], "bound": "tensor", "achieved": ach, "peak": peaks["bf16_sustained"],
                    "unit": "TFLOP/s", "frac": ach / peaks["bf16_sustained"], "traffic": ncu_traffic(top["name"], B),
                    "peak_source": peaks["source"] + " (sustained bf16, kernel timed inside a long step)",
                    "launches_per_step": top["launches"], "ms_per_step": top["ms"]}
        if top["name"] == "md_attention_bf16":
            # the same kernel timed ALONE (its clock is then not the step's): against the burst peak, as the recipe says
            NHh = NH
            Ba = max(1, min(B, (256 * 2096) // L))          # at most the base config's token count (memory at the scaled config)
            qkv = (torch.randn(Ba * L, 3 * NHh * 64, device=dev) * 0.7).to(torch.bfloat16)
            o = torch.empty(Ba * L, NHh * 64, device=dev, dtype=torch.bfloat16)
            for _ in range(3):
                ops.attention(qkv, Ba, L, NHh, out=o)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(10):
                ops.attention(qkv, Ba, L, NHh, out=o)
            a1.record()
            torch.cuda.synchronize()
            alone = 4.0 * Ba * NHh * L * L * 64 / (a0.elapsed_time(a1) / 10 * 1e-3) / 1e12
            roofline["alone"] = {"achieved": alone, "peak": peaks["bf16_burst"], "frac": alone / peaks["bf16_burst"],
                                 "ms_per_launch": a0.elapsed_time(a1) / 10,
                                 "sequences": Ba, "note": "10 back-to-back launches outside the step; burst bf16 peak"}
            del qkv, o
    step_tflops = flops_per_sequence_step() * B / (ms_step * 1e-3) / 1e12

    # ---- end to end through the public API: pinned host ids -> tokens on host, K chain steps via t_enc
    e2e = None
    if not args.full_chain and not args.no_e2e:
        k_e2e = args.steps
        strength = (k_e2e + 0.5) / DIFFUSION_STEPS                # int(2000 * strength) == k_e2e (k / 2000 can round below)
        for it in range(2):                                        # first pass = warm-up
            dist.barrier()
            torch.cuda.synchronize()
            tic = time.perf_counter()
            if args.mode == "generation":
                tok = sample_generation_steps(model, diffusion, model_emb, cond_host, k_e2e, dev)
            else:
                tok = sample_batch(model, diffusion, model_emb, cond_host, "modification", DIFFUSION_STEPS, DIFFUSION_STEPS,
                                   strength=strength, top_p=1, clamp_step=0, device=dev)
            tok = dist.all_gather_tokens(tok)                      # NCCL all-gather of the decoded ids (no-op at N = 1)
            tok_host = tok.to("cpu", non_blocking=False) if rank == 0 else None
            torch.cuda.synchronize()
            t_e2e = time.perf_counter() - tic
        te = torch.tensor([t_e2e], device=dev, dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(te, op=torch.distributed.ReduceOp.MAX)
        t_e2e = float(te[0])
        e2e = {"value": (B * world) / (t_e2e * DIFFUSION_STEPS / k_e2e), "unit": "sequences/s",
               "h2d_bytes_per_step": int(sum(v.numel() * v.element_size() for v in cond_host.values())),
               "d2h_bytes_per_step": int(B * world * L * 8),
               "gathered": "decoded ids of all ranks all-gathered over NCCL inside the timed region, rank 0 copies [%d, %d] int64 to the host" % (B * world, L),
               "note": "sample_batch() public API, %d chain steps via t_enc incl. H2D ids/mask, embedding gather, "
                       "q_sample, decode and D2H tokens; whole call scaled by 2000/%d" % (k_e2e, k_e2e),
               "seconds_per_call": t_e2e}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_sample(args.mode)

    if rank == 0:
        line = {"metric": "sequences/sec full reverse-diffusion sampling", "value": value, "unit": "sequences/s",
                "n_gpus": world, "steps": timed_steps, "warmup": args.warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": workload_config(B, world, mode=args.mode), "ms_per_denoiser_step": ms_step, "ms_decode": ms_decode,
                "step_tflops": step_tflops, "step_frac_of_bf16_sustained": step_tflops / peaks["bf16_sustained"],
                "clocks": sampler.summary(), "gpu_launches": launches,
                "launch_mode": ("one captured CUDA graph of the reverse step replayed per step (device-resident step index / "
                                "Philox counter)" if diffusion.use_cuda_graph else "eager launches"),
                "e2e": e2e, "roofline": roofline,
                "cpu_baseline": cpu_baseline, "kernels": breakdown}
        print(json.dumps(line))
    dist.barrier()


DUMP_BYTES = 56 << 20                                          # --dump-outputs stays below 64 MB in all


def dump_outputs(out_dir, sample, tokens):
    """`--dump-outputs DIR`: what the timed chain hands its caller after its last step, `sample.npy` (x_t, fp32 [n, L, 128]),
    and the final decode of it, `tokens.npy` (token ids as fp32 [n, L]), for n sequences drawn with a fixed seed from the
    batch (all of them when they fit DUMP_BYTES; rank 0's batch under torchrun), so that two builds can be compared output
    for output."""
    import numpy as np
    import torch
    B, Ls, Ds = sample.shape
    n = min(B, DUMP_BYTES // (Ls * (Ds + 1) * 4))
    rows = torch.from_numpy(np.sort(np.random.default_rng(0).choice(B, n, replace=False))).to(sample.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "sample.npy"), sample.index_select(0, rows).float().cpu().numpy())
    np.save(os.path.join(out_dir, "tokens.npy"), tokens.index_select(0, rows).cpu().numpy().astype(np.float32))


def sample_generation_steps(model, diffusion, model_emb, cond, k_steps, dev):
    """sample_batch()'s generation branch (run/sample.py:177-220) cut to the first k_steps chain indices through the
    reference's own t_enc argument (generation mode has no strength flag to shorten the chain with)."""
    import torch
    from functools import partial
    from musediffusion_b200 import ops
    from musediffusion_b200.rounding import denoised_fn_round
    ids = torch.as_tensor(cond["input_ids"]).to(dev, non_blocking=True)
    mask_ori = torch.as_tensor(cond["input_mask"]).to(dev, non_blocking=True)
    x_start = model.get_embeds(ids)
    mask = torch.broadcast_to(mask_ori.unsqueeze(-1), x_start.shape)
    x_noised = ops.q_sample(x_start, None, seed=diffusion._seed(), step_counter=diffusion._next_counter(),
                            seq_offset=diffusion.seq_offset, mask=mask_ori)
    samples = diffusion.p_sample_loop(model=model, shape=tuple(x_start.shape), noise=x_noised, clip_denoised=True,
                                      denoised_fn=partial(denoised_fn_round, model_emb, dist=None), model_kwargs=cond,
                                      top_p=1, clamp_step=0, clamp_first=True, mask=mask, x_start=x_start, gap=1,
                                      t_enc=k_steps, only_last=True)
    return model.decode_tokens(samples[-1])


def ncu_traffic(kernel, B):
    """dram bytes (read + write) per launch from the committed `ncu --set full` capture of this kernel
    (profiles/r2_traffic.json, written by tools/summarize_profiles.py from tools/ncu_round.sh's reports: bytes of ONE launch at
    the captured batch, scaled linearly to B); null when no capture exists for this kernel."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            t = json.load(f)
        ent = t.get(kernel) or t.get(kernel.split(":")[0])
        if ent is None and ":" in kernel:                      # same GEMM shape captured at another batch: match on N x K + epilogue
            tail = kernel.split("x", 1)[1]
            ent = next((v for k, v in t.items() if ":" in k and k.split("x", 1)[1] == tail), None)
        return float(ent["dram_bytes_per_launch"]) * B / float(ent["batch"]) if ent else None
    except Exception:
        return None


def summarize_profile(prof, B):
    """prof: list of (kernel name, detail, ms).  FLOPs: linear 2MNK, attention 4 B NH L^2 64."""
    out = {}
    for name, detail, ms in prof:
        key = name + (":" + detail if detail else "")
        e = out.setdefault(key, {"name": key, "ms": 0.0, "launches": 0, "flops": 0.0})
        e["ms"] += ms
        e["launches"] += 1.0 / 3.0                                  # three profiled steps, per-step figures
        if name == "md_linear_bf16":
            M, N, K = [int(v) for v in detail.split(" ")[0].split("x")]
            e["flops"] += 2.0 * M * N * K / 3.0
        elif name == "md_attention_bf16":
            e["flops"] += 4.0 * B * NH * L * L * 64 / 3.0
    for e in out.values():
        e["launches"] = int(round(e["launches"]))
        if e["flops"]:
            e["tflops"] = e["flops"] / (e["ms"] * 1e-3) / 1e12
    return out


def cpu_baseline_sample(mode):
    """bounded CPU sample of the same workload (10-30 s of host work): the unmodified reference at batch 4 (BASELINE.md
    section 3) for 1 warm-up + 3 timed chain steps; the numpy port (1 sequence) if the reference tree is absent."""
    have_ref = os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "MuseDiffusion")) or os.path.isdir("/root/reference/MuseDiffusion")
    Bc = 4 if have_ref else 1
    per_step, kind, threads, sample = time_reference_cpu(mode, Bc, 1, 3)
    return {"value": Bc / (per_step * DIFFUSION_STEPS), "unit": "sequences/s", "cores": threads, "kind": kind, "sample": sample}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed chain steps (default 10; not with --full-chain)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="sequences per GPU")
    ap.add_argument("--ref-batch", type=int, default=4, help="sequences per step for --impl reference (BASELINE.md section 3: 4)")
    ap.add_argument("--mode", default="modification", choices=["modification", "generation"],
                    help="modification = BASELINE.json configs[1] (default); generation = configs[2] (sample_generation path)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="label of the run: weak = --batch sequences per GPU whatever N (default); strong = the caller divides a "
                         "fixed total by N itself (BASELINE.json configs[4]: 2048 sequences over 2/4/8 GPUs)")
    ap.add_argument("--full-chain", action="store_true", help="run all 2000 chain steps instead of extrapolating")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-breakdown", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaled", action="store_true", help="BASELINE.json config 5: hidden 1024, 24 layers, 16 heads, FFN 4096, seq_len 4192")
    ap.add_argument("--seq-len", type=int, default=0)
    ap.add_argument("--hidden", type=int, default=0)
    ap.add_argument("--ffn", type=int, default=0)
    ap.add_argument("--layers", type=int, default=0)
    ap.add_argument("--heads", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the chain state x_t and its decoded token ids as DIR/<name>.npy "
                         "(a fixed seeded sample of the sequences, < 64 MB; rank 0's shard under torchrun)")
    args = ap.parse_args()
    set_model_shape(args)
    if (L, H, F, NL, NH) != (2096, 768, 3072, 12, 12):
        args.no_cpu_baseline = True      # the CPU port sample is sized for the base config only
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.full_chain and args.steps is not None:
        ap.error("--full-chain times the %d - warmup steps left after the warm-up; leave --steps out" % DIFFUSION_STEPS)
    if args.steps is None:
        args.steps = 10
    if args.steps < 1 or (not args.full_chain and args.warmup + args.steps > DIFFUSION_STEPS):
        ap.error("--steps takes 1 to %d - warmup (%d) chain steps" % (DIFFUSION_STEPS, args.warmup))
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours computes")
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    finally:
        import torch.distributed as torch_dist
        if torch_dist.is_available() and torch_dist.is_initialized():
            torch_dist.destroy_process_group()


if __name__ == "__main__":
    main()
