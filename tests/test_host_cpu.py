"""CPU tests of the host side: the C-ABI library loads and exports every symbol of include/musediff_b200.h (no
compute calls), the host mirror reproduces the reference's schedule tables and state-dict layout, product code never
imports the oracle, and the world_size-2 sharding logic works over gloo."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "musediff_b200.h")).read()
    declared = set(re.findall(r"\b(md_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 15
    from musediffusion_b200 import _lib
    for name in declared:
        assert hasattr(_lib.lib, name), name
    assert declared - {"md_last_error", "md_abi_version"} == set(_lib.SIGNATURES)
    assert _lib.lib.md_abi_version() == 2
    assert _lib.lib.md_last_error() is not None


def test_ops_refuse_cpu_tensors():
    from musediffusion_b200 import _lib, ops
    with pytest.raises(_lib.MuseDiffLibraryError):
        ops.round_argmin(torch.zeros(4, 128), torch.zeros(729, 128))
    with pytest.raises(_lib.MuseDiffLibraryError):
        ops.cast_bf16(torch.zeros(8, 128))


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "musediffusion_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "musediff_oracle" not in src and "decode_oracle" not in src and "oracle/" not in src, f


TABLES = ["betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod",
          "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_variance",
          "posterior_log_variance_clipped", "posterior_mean_coef1", "posterior_mean_coef2"]


@pytest.mark.parametrize("sched,T,resp", [("sqrt", 2000, ""), ("linear", 1000, ""), ("cosine", 500, ""),
                                          ("trunc_cos", 400, ""), ("trunc_lin", 300, ""), ("pw_lin", 200, ""),
                                          ("sqrt", 2000, "ddim50"), ("sqrt", 300, "10,15,20")])
def test_host_schedules_bit_exact_vs_reference(golden_dir, sched, T, resp):
    from musediffusion_b200.diffusion import SpacedDiffusion, get_named_beta_schedule, space_timesteps
    g = np.load(os.path.join(golden_dir, "schedules.npz"))
    key = "%s_%d_%s" % (sched, T, resp.replace(",", "-") or "full")
    betas = get_named_beta_schedule(sched, T)
    assert np.array_equal(betas, g[key + "/raw_betas"])
    d = SpacedDiffusion(use_timesteps=space_timesteps(T, resp if resp else [T]), betas=betas, rescale_timesteps=True,
                        predict_xstart=True)
    assert np.array_equal(np.asarray(d.timestep_map), g[key + "/timestep_map"])
    for n in TABLES:
        assert np.array_equal(getattr(d, n), g[key + "/" + n]), n


def test_state_dict_layout_and_factory():
    import musediff_oracle as O
    from types import SimpleNamespace
    from musediffusion_b200.initialization import create_model_and_diffusion, seed_all
    args = SimpleNamespace(hidden_dim=128, hidden_t_dim=128, vocab_size=729, seq_len=2096, dropout=0.1,
                           noise_schedule="sqrt", diffusion_steps=2000, timestep_respacing="", rescale_timesteps=True,
                           predict_xstart=True)
    model, diffusion = create_model_and_diffusion(args)
    sd = model.state_dict()
    assert len(sd) == 211 and sum(p.numel() for p in model.parameters()) == 88598489      # SURVEY.md Appendix B
    p = O.make_random_params(seed=0, seq_len=64)
    small, _ = create_model_and_diffusion(SimpleNamespace(**{**vars(args), "seq_len": 64}))
    assert set(small.state_dict()) == set(p)
    assert all(tuple(small.state_dict()[k].shape) == p[k].shape for k in p)
    assert small.lm_head.weight is small.word_embedding.weight
    assert diffusion.num_timesteps == 2000 and diffusion.timestep_map[-1] == 1999
    t = diffusion._model_timesteps(torch.tensor([1999, 0]))
    assert t.tolist() == [999.5, 0.0]
    with pytest.raises(Exception):
        model(torch.zeros(1, 8, 128), torch.zeros(1))                  # CPU tensors: no fallback path
    seed_all(105, deterministic=True)
    assert torch.initial_seed() == 105


def test_synthetic_batches_match_oracle_generator():
    import musediff_oracle as O
    from musediffusion_b200.synthetic import make_synthetic_batch
    for mode in ("generation", "modification"):
        a, b = make_synthetic_batch(mode, 5, 96, seed=9), O.make_synthetic_batch(mode, 5, 96, seed=9)
        assert all(np.array_equal(a[k], b[k]) and a[k].dtype == b[k].dtype for k in b)


def test_world_size_2_sharding_gloo(tmp_path):
    """two CPU ranks over gloo: contiguous shards cover the batch, all_gather_tokens restores global order."""
    script = tmp_path / "w.py"
    script.write_text(
        "import os, sys, torch\n"
        "sys.path.insert(0, %r)\n"
        "from musediffusion_b200 import dist\n"
        "rank, world, dev = dist.setup(backend='gloo')\n"
        "lo, hi = dist.shard_range(10, rank, world)\n"
        "tok = torch.arange(lo, hi).view(-1, 1).repeat(1, 4)\n"
        "full = dist.all_gather_tokens(tok)\n"
        "assert full[:, 0].tolist() == list(range(10)), full\n"
        "lin = torch.nn.Linear(3, 3)\n"
        "dist.broadcast_model(lin)\n"
        "ws = dist.gather_objects(lin.weight.sum().item())\n"
        "assert abs(ws[0] - ws[1]) < 1e-7\n"
        "dist.barrier()\n"
        "print('rank', rank, 'ok')\n" % ROOT)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29611", str(script)],
                       capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))       # CPU ranks even where a GPU is present
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("ok") == 2


def test_custom_ops_are_registered_for_cuda_only():
    """BASELINE.json north star: the kernels are exposed as PyTorch custom ops (`torch.ops.musediff.*`) — registered for the
    CUDA dispatch key and nothing else, so a CPU tensor can never take a fallback path."""
    import torch
    from musediffusion_b200 import _lib, custom_ops
    for name in custom_ops.OP_NAMES:
        op = getattr(torch.ops.musediff, name)
        assert "musediff::" + name in str(op.default._schema)
    # every kernel entry of the header has its op (md_set_schedule is a host->device table copy, the padded-vocab helper is host only)
    entries = set(_lib.SIGNATURES) - {"md_set_schedule", "md_round_tc_padded_vocab"}
    assert {"md_" + n for n in custom_ops.OP_NAMES} == entries
    with pytest.raises(NotImplementedError):
        torch.ops.musediff.cast_f32_bf16(torch.ones(4), torch.empty(4, dtype=torch.bfloat16))
    with pytest.raises(_lib.MuseDiffLibraryError):
        from musediffusion_b200 import ops
        ops.cast_bf16(torch.ones(4))
