"""The hot slice of MuseDiffusion/run/sample.py (:84-114 set-up, :177-220 per-batch sampling) as a library call plus a
small command line with the reference's sub-commands and flag names (`generation` / `modification`;
MuseDiffusion/config/sample.py:93-112,137-209).  MIDI decoding, metrics and the dataset pipeline stay with the
reference (out of scope, SURVEY.md section 8f): this entry point reads token batches (.npz) or synthesises
ComMU-shaped ones and writes decoded token ids."""
import argparse
import json
import os
import time
from functools import partial
from types import SimpleNamespace

import numpy as np
import torch

from . import ops
from .initialization import create_model_and_diffusion, seed_all
from .rounding import denoised_fn_round


def build_model_emb(model, device):
    """run/sample.py:92-101: frozen copy of the word embedding used by the rounding callback.  Its split-bf16 form for the
    tensor-core rounding is built here, once, so the first sampling call launches the same kernels as every later one."""
    w = model.word_embedding.weight
    emb = torch.nn.Embedding(num_embeddings=w.shape[0], embedding_dim=w.shape[1], padding_idx=0,
                             _weight=w.detach().clone())
    emb = emb.eval().requires_grad_(False).to(device)
    ops.split_embedding(emb.weight)
    return emb


SAMPLERS = ("reference", "dpm_solver++")


@torch.no_grad()
def sample_batch(model, diffusion, model_emb, cond, mode, step, diffusion_steps, strength=0.75, top_p=1, clamp_step=0,
                 clip_denoised=True, device=None, fused_decode=True, return_sample=False, sampler="reference"):
    """run/sample.py:177-220 for one batch: cond = {'input_ids', 'input_mask'} (host or device int tensors) ->
    int64 token ids [B, L] on the device.  `fused_decode=False` keeps the reference's get_logits + argmax pair;
    `return_sample=True` also returns the final x_0 estimate `samples[-1]` (fp32 [B, L, D]).
    `sampler="dpm_solver++"` (not in the reference) samples with `diffusion.dpm_solver_sample_loop` in `step` model
    evaluations instead of the reference's DDPM / DDIM choice; top_p and clamp_step do not apply to it.  Its modification
    mode starts at index t_start = int(strength * T) - 1 of the diffusion's T indices, so `strength` is the fraction of the
    chain whatever `step` is (the reference's DDIM starts at int(step * strength) - 1 and reads the table with gap
    T // step)."""
    if sampler not in SAMPLERS:
        raise ValueError("sampler must be one of %s, got %r" % (SAMPLERS, sampler))
    dpm = sampler == "dpm_solver++"
    device = device or next(model.parameters()).device
    input_ids = torch.as_tensor(cond["input_ids"]).to(device, non_blocking=True)
    mask_ori = torch.as_tensor(cond["input_mask"]).to(device, non_blocking=True)
    x_start = model.get_embeds(input_ids)                                               # :185
    input_ids_mask = torch.broadcast_to(mask_ori.unsqueeze(dim=-1), x_start.shape)      # :186
    if mode == "generation":                                                            # :190-193
        noising_t = None
        t_start = diffusion.num_timesteps - 1
        if diffusion.noise_source is not None:
            noise = diffusion._external_noise(x_start.shape, "randn", device)
        else:
            noise = None
        x_noised = ops.q_sample(x_start, None, noise=noise, seed=diffusion._seed(),
                                step_counter=diffusion._next_counter(), seq_offset=diffusion.seq_offset, mask=mask_ori)
    else:                                                                               # :195-197
        noising_t = int(step * strength)
        t_start = int(strength * diffusion.num_timesteps) - 1 if dpm else noising_t - 1
        if dpm and t_start < 0:
            raise ValueError("strength=%r leaves no diffusion index to start from (T=%d)" % (strength, diffusion.num_timesteps))
        timestep = torch.full((x_start.shape[0], 1), t_start, device=device)
        x_noised = diffusion.q_sample(x_start.unsqueeze(-1), timestep, mask=input_ids_mask).squeeze(-1)
    denoised_fn = partial(denoised_fn_round, model_emb, dist=None)
    if dpm:
        samples = diffusion.dpm_solver_sample_loop(model=model, shape=tuple(x_start.shape), noise=x_noised,
                                                   clip_denoised=clip_denoised, denoised_fn=denoised_fn, model_kwargs=cond,
                                                   mask=input_ids_mask, x_start=x_start, steps=step, t_start=t_start,
                                                   only_last=True)
    else:
        if step == diffusion_steps:                                                     # :109-114
            gap, sample_fn = 1, diffusion.p_sample_loop
        else:
            gap, sample_fn = diffusion_steps // step, diffusion.ddim_sample_loop
        samples = sample_fn(model=model, shape=tuple(x_start.shape), noise=x_noised, clip_denoised=clip_denoised,
                            denoised_fn=denoised_fn, model_kwargs=cond, top_p=top_p, clamp_step=clamp_step, clamp_first=True,
                            mask=input_ids_mask, x_start=x_start, gap=gap, t_enc=noising_t, only_last=True)   # :200-215
    sample = samples[-1]
    if fused_decode:
        tokens = model.decode_tokens(sample)
    else:
        tokens = torch.argmax(model.get_logits(sample), dim=-1)                         # :219-220
    return (tokens, sample) if return_sample else tokens


def load_training_args(model_path):
    """config/sample.py:114-134: `training_args.json` (the reference's `TrainSettings(...).json()`) sits next to the checkpoint."""
    from .checkpoint import load_training_args as _load
    return _load(model_path)


def load_model(model_path, device):
    """run/sample.py:76-88: model + diffusion from a model directory.  `model_path` is either the reference's `model_*.pt`
    (state dict; `training_args.json` next to it) or a packed weight file `*.mdpack` written by `python -m
    musediffusion_b200 pack` (its header carries the model configuration, so training_args.json is optional)."""
    from . import checkpoint
    if model_path.endswith(".mdpack"):
        header, _ = checkpoint.read_pack_header(model_path)
        cfg = header["config"]
        targs_path = checkpoint.training_args_path(model_path)
        targs = checkpoint.load_training_args(targs_path) if os.path.isfile(targs_path) else SimpleNamespace(**checkpoint.MODEL_FIELDS)
        for k in checkpoint.MODEL_FIELDS:
            if k in cfg:
                setattr(targs, k, cfg[k])
        targs.encoder_config = {k: cfg[k] for k in ("hidden_size", "num_hidden_layers", "num_attention_heads", "intermediate_size",
                                                     "layer_norm_eps") if k in cfg}
        model, diffusion = create_model_and_diffusion(targs)
        model.eval().requires_grad_(False)
        model.load_weight_pack(model_path, device)
    else:
        targs = load_training_args(model_path)
        model, diffusion = create_model_and_diffusion(targs)
        model.load_state_dict(checkpoint.load_state_dict(model_path, map_location="cpu"))
        model.eval().requires_grad_(False).to(device)
    return model, diffusion, targs


def create_parser():
    p = argparse.ArgumentParser(prog="python -m musediffusion_b200")
    sub = p.add_subparsers(dest="mode", required=True)
    pk = sub.add_parser("pack", help="write a packed bf16 weight file (*.mdpack) from a reference checkpoint")
    pk.add_argument("--model_path", required=True, help="model_*.pt written by the reference's trainer")
    pk.add_argument("--out", default=None, help="output path (default: <model_path minus .pt>.mdpack)")
    for name in ("generation", "modification"):
        sp = sub.add_parser(name)
        sp.add_argument("--model_path", required=True)
        sp.add_argument("--step", type=int, default=100)
        sp.add_argument("--out_dir", default="./out")
        sp.add_argument("--batch_size", type=int, default=50)
        sp.add_argument("--top_p", type=int, default=1)
        sp.add_argument("--clamp_step", type=int, default=0)
        sp.add_argument("--sample_seed", type=int, default=105)
        sp.add_argument("--clip_denoised", type=lambda s: s.lower() in ("1", "true", "yes"), default=True)
        sp.add_argument("--sampler", choices=SAMPLERS, default="reference",
                        help="reference: the reference's DDPM (--step = diffusion_steps) or DDIM; dpm_solver++: DPM-Solver++(2M) "
                             "with --step model evaluations (not in the reference; --strength is then the fraction of the chain)")
        sp.add_argument("--input_npz", default=None, help="npz with input_ids/input_mask [N, L] (else synthetic)")
        sp.add_argument("--strict_validation", action="store_true",
                        help="also run validate_rigidly (the reference does when it computes metrics, run/sample.py:240)")
        if name == "modification":
            sp.add_argument("--strength", type=float, default=0.75)
            sp.add_argument("--num_batches", type=int, default=1)
            boolean = lambda s: s.lower() in ("1", "true", "yes")                     # noqa: E731
            # config/sample.py:139-153: each defaults to the value in training_args.json
            sp.add_argument("--use_corruption", type=boolean, default=None)
            sp.add_argument("--corr_available", type=str, default=None)
            sp.add_argument("--corr_max", type=int, default=None)
            sp.add_argument("--corr_p", type=float, default=None)
            sp.add_argument("--corr_kwargs", type=str, default=None)
        else:
            sp.add_argument("--num_samples", type=int, default=1000)
            from .meta import add_meta_arguments
            add_meta_arguments(sp)                       # config/sample.py:223-230: --bpm ... --chord_progression / --meta_json
    return p


def corruption_from_args(args, targs):
    """run/sample.py:125-135 + config/sample.py:150-153: corruption flags left unset take the training run's values; returns
    the `Corruptions` callable or None when corruption is off."""
    from .corruption import Corruptions
    pick = lambda k: getattr(args, k, None) if getattr(args, k, None) is not None else getattr(targs, k, None)   # noqa: E731
    if not pick("use_corruption"):
        return None
    return Corruptions.from_config(pick("corr_available"), pick("corr_max"), pick("corr_p"), pick("corr_kwargs"))


def batch_metrics(total, prep, correct_ids, mask, batch_index):
    """run/sample.py:244-280: ONNC over (ground truth + generated) note sequences of the batch's VALID rows, pitch / velocity
    controllability of the generated ones; sums kept the way the reference weights them."""
    from . import decode_util, metric
    keep = [k for k in range(len(prep.status)) if prep.status[k] == decode_util.OK]
    truth = decode_util.prepare_batch(torch.as_tensor(correct_ids).to(mask.device)[keep], mask[keep])
    if any(ns is None for ns in truth.note_seqs):
        raise decode_util.SequenceToMidiError("ground-truth row cannot be split into meta and notes")
    generated, metas = [prep.note_seqs[k] for k in keep], [prep.metas[k] for k in keep]
    onnc = float(metric.ONNC(tuple(truth.note_seqs) + tuple(generated), device=mask.device))
    total_p, wrong_p = metric.Controllability_Pitch(metas, generated, device=mask.device)
    total_v, wrong_v = metric.Controllability_Velocity(metas, generated, device=mask.device)
    total["onnc_sum"] += len(keep) * onnc
    total["onnc_count"] += len(keep)
    total["total_total_p"] += total_p
    total["total_wrong_p"] += wrong_p
    total["total_total_v"] += total_v
    total["total_wrong_v"] += wrong_v
    print((" Metric of Batch %d " % batch_index).center(60, "="))
    print((" ONNC: %.6f " % onnc).center(60))
    print((" CP: %.6f " % (wrong_p / total_p)).center(60))
    print((" CV: %.6f " % (wrong_v / total_v)).center(60))
    print("=" * 60 + "\n")


def pack_main(args):
    """`python -m musediffusion_b200 pack --model_path model_000000.pt`: checkpoint -> packed weight file (host only)."""
    from . import checkpoint
    targs = load_training_args(args.model_path)
    model, _ = create_model_and_diffusion(targs)
    sd = checkpoint.load_state_dict(args.model_path, map_location="cpu")
    missing = set(model.state_dict()) - set(sd)
    if missing:
        raise KeyError("checkpoint lacks %d keys, e.g. %s" % (len(missing), sorted(missing)[:3]))
    out = args.out or (args.model_path[:-3] if args.model_path.endswith(".pt") else args.model_path) + ".mdpack"
    checkpoint.write_pack(out, sd, checkpoint.model_config_of(targs, model))
    print("### wrote %s (%.1f MB)" % (out, os.path.getsize(out) / 1e6))
    return out


def main(argv=None):
    args = create_parser().parse_args(argv)
    if args.mode == "pack":
        return pack_main(args)
    from . import decode_util, dist
    rank, world, dev = dist.setup()
    model, diffusion, targs = load_model(args.model_path, dev)
    model_emb = build_model_emb(model, dev)
    seed_all(args.sample_seed, deterministic=True)
    midi_meta = None
    if args.mode == "generation":
        from .meta import meta_from_args, meta_to_batch
        midi_meta = meta_from_args(args)
    correct_all = None
    if args.input_npz:
        data = np.load(args.input_npz)
        ids_all, mask_all = data["input_ids"], data["input_mask"]
        if args.mode == "modification" and "correct_ids" in data.files:      # data/wrapper.py:118-124: what the loader keeps
            correct_all = data["correct_ids"]                                # beside the (possibly corrupted) input_ids
        elif args.mode == "modification":
            corruption = corruption_from_args(args, targs)
            if corruption is not None:                                        # data/wrapper.py:73-86: row by row, in order
                correct_all, ids_all = ids_all, np.array(ids_all)
                lengths = data["length"] if "length" in data.files else (ids_all != 0).cumsum(1).argmax(1) + 1
                for row, n in zip(ids_all, lengths):
                    row[:n] = corruption(row[:n])
    elif midi_meta is not None:                                   # run/sample.py:117-121: every sample from the one meta
        b = meta_to_batch(midi_meta, args.num_samples, targs.seq_len)
        ids_all, mask_all = b["input_ids"].numpy(), b["input_mask"].numpy()
    else:
        from .synthetic import make_synthetic_batch
        n = args.num_samples if args.mode == "generation" else args.batch_size * args.num_batches
        b = make_synthetic_batch(args.mode, n, targs.seq_len, seed=args.sample_seed)
        ids_all, mask_all = b["input_ids"], b["input_mask"]
        # the synthetic prefixes draw every meta token from its whole range, "unknown" included; a MIDI file cannot carry an
        # unknown tempo / key / time signature (the reference's writer raises on them), so the stand-in input takes the first
        # known class instead
        for col, unknown in ((0, 560), (1, 601), (2, 626)):
            ids_all[:, col] = np.where(ids_all[:, col] == unknown, unknown + 1, ids_all[:, col])
    out_dir = os.path.join(args.out_dir, os.path.basename(os.path.dirname(os.path.abspath(args.model_path))),
                           os.path.basename(args.model_path) + "." + args.mode + ".samples")
    os.makedirs(out_dir, exist_ok=True)
    tic = time.time()
    n_batches = (len(ids_all) + args.batch_size - 1) // args.batch_size
    L = ids_all.shape[1]
    rows = []                                                     # rank 0: (batch index, tokens, mask) in batch order
    for base in range(0, n_batches, world):                       # one round = `world` consecutive batches, one per rank
        bi = base + rank                                          # run/sample.py:169-172: batch bi belongs to rank bi % world
        tok_pad = torch.zeros((args.batch_size, L), dtype=torch.int32, device=dev)
        if bi < n_batches:
            sl = slice(bi * args.batch_size, (bi + 1) * args.batch_size)
            diffusion.seq_offset = sl.start
            cond = {"input_ids": torch.from_numpy(ids_all[sl]), "input_mask": torch.from_numpy(mask_all[sl])}
            tok = sample_batch(model, diffusion, model_emb, cond, args.mode, args.step, targs.diffusion_steps,
                               strength=getattr(args, "strength", 0.75), top_p=args.top_p, clamp_step=args.clamp_step,
                               clip_denoised=args.clip_denoised, device=dev, sampler=args.sampler)
            tok_pad[:tok.shape[0]] = tok.to(torch.int32)
        # decoded ids of the round to every rank with ONE NCCL all-gather ([world, batch, L] int32), instead of the reference's
        # rank-after-rank decode with a broadcast + barrier per rank (run/sample.py:222-294)
        gathered = dist.all_gather_tokens(tok_pad).view(world, args.batch_size, L)
        if rank == 0:
            for k in range(min(world, n_batches - base)):
                n = min(args.batch_size, len(ids_all) - (base + k) * args.batch_size)
                rows.append((base + k, gathered[k, :n]))
    if rank == 0:
        # decode_batch (utils/decode_util.py:233-384) on the gathered ids: one launch per batch for the token-level half, then one
        # MIDI file per valid row, named and numbered like the reference's
        flat, statuses, valid = [], [], 0
        metric_total = dict(onnc_sum=0.0, onnc_count=0, total_total_p=0, total_wrong_p=0, total_total_v=0, total_wrong_v=0)
        for bi, tok in rows:
            mask = torch.from_numpy(mask_all[bi * args.batch_size: bi * args.batch_size + tok.shape[0]]).to(dev)
            prep = decode_util.prepare_batch(tok, mask, strict_validation=args.strict_validation)
            flat.append(tok.cpu().numpy().astype(np.int64))
            statuses.append(prep.status)
            n_valid = decode_util.decode_batch(args.mode, tok, mask, batch_index=bi, output_dir=out_dir,
                                               previous_count=valid if args.mode == "generation" else bi * args.batch_size,
                                               strict_validation=args.strict_validation, prepared=prep)
            valid += n_valid
            if correct_all is not None and n_valid:
                batch_metrics(metric_total, prep, correct_all[bi * args.batch_size: bi * args.batch_size + tok.shape[0]], mask, bi)
        np.save(os.path.join(out_dir, "tokens.npy"), np.concatenate(flat, axis=0))
        np.save(os.path.join(out_dir, "decode_status.npy"), np.concatenate(statuses))
        if correct_all is not None and metric_total["onnc_count"]:                # run/sample.py:303-311
            print(" Total Metric ".center(60, "="))
            print((" ONNC: %.6f " % (metric_total["onnc_sum"] / metric_total["onnc_count"])).center(60))
            print((" CP: %.6f " % (metric_total["total_wrong_p"] / metric_total["total_total_p"])).center(60))
            print((" CV: %.6f " % (metric_total["total_wrong_v"] / metric_total["total_total_v"])).center(60))
            print("=" * 60 + "\n")
        print("### Total takes %.2fs; %d sequences (%d valid) -> %s"
              % (time.time() - tic, sum(len(t) for t in flat), valid, out_dir))
    dist.barrier()
