"""Embedding widths that are not a multiple of 64 (`--hidden_dim` is a free parameter of the reference's TrainSettings).
The bf16 tensor-core operands are zero-padded to Dp = round_up(D, 64); every tensor of the public API stays D wide.
Forward, rounding, padding neutrality, the paper configuration (D = 500, L = 256), eps-prediction, graph replay,
sharding, weight packs and the command line, against the numpy oracle."""
import json
import os
from functools import partial
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import musediff_oracle as O

pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

from musediffusion_b200 import ops  # noqa: E402
from musediffusion_b200.initialization import create_model_and_diffusion  # noqa: E402
from musediffusion_b200.rounding import denoised_fn_round, get_efficient_knn  # noqa: E402
from musediffusion_b200.sample import build_model_emb  # noqa: E402
from test_sampling_gpu import DEV, assert_chain_parity, oracle_trace, rel, run_with_trace  # noqa: E402

WIDTHS = [16, 100, 200, 500]          # 200 is a multiple of 8 but not of 64


def make(D, L, seed, pxs=True, T=2000, params=None):
    p = params if params is not None else O.make_random_params(seed=seed, seq_len=L, hidden_dim=D)
    args = SimpleNamespace(hidden_dim=D, hidden_t_dim=128, vocab_size=729, seq_len=L, dropout=0.1, noise_schedule="sqrt",
                           diffusion_steps=T, timestep_respacing="", rescale_timesteps=True, predict_xstart=pxs)
    model, diffusion = create_model_and_diffusion(args)
    model.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in p.items()}, strict=True)
    model.eval().requires_grad_(False).to(DEV)
    return model, diffusion, p


@pytest.mark.parametrize("D", WIDTHS)
def test_forward_decode_and_logits(D):
    L = 80
    model, _, p = make(D, L, seed=D)
    rng = np.random.default_rng(D)
    x = rng.standard_normal((3, L, D)).astype(np.float32)
    t = np.array([1999.0, 250.0, 0.0], dtype=np.float32)
    xt = torch.from_numpy(x).to(DEV)
    out = model(xt, torch.from_numpy(t).to(DEV))
    assert out.shape == (3, L, D) and out.dtype == torch.float32
    r = rel(out.cpu().numpy(), O.denoiser_forward(p, x, t))
    print("hidden_dim %d: max-norm relative error of the denoiser output vs the oracle %.4f" % (D, r))
    assert r < 2e-2, r
    t_same = torch.full((3,), 250.0, device=DEV)
    a = model.denoise(xt, t_same, uniform_t=True).clone()
    assert torch.equal(a, model.denoise(xt, t_same, uniform_t=False))
    assert np.array_equal(model.decode_tokens(xt).cpu().numpy(), O.logits_argmax(p, x))
    assert rel(model.get_logits(xt).cpu().numpy(), O.get_logits(p, x)) < 2e-5
    ids = torch.from_numpy(rng.integers(0, 729, size=(3, L))).to(DEV)
    assert torch.equal(model.get_embeds(ids), model.word_embedding.weight[ids])


def _f64_best(x, E, bias=None):
    """float64 ids (lowest on ties) and top-2 margins of argmin |x - E_v|^2 (bias None) or argmax x.E_v + bias_v."""
    x64, E64 = x.astype(np.float64), E.astype(np.float64)
    dot = x64 @ E64.T
    score = (E64 ** 2).sum(1)[None] + (x64 ** 2).sum(1)[:, None] - 2 * dot if bias is None else -(dot + bias.astype(np.float64))
    order = np.argsort(score, axis=1, kind="stable")
    rows = np.arange(len(x))
    return order[:, 0], score[rows, order[:, 1]] - score[rows, order[:, 0]]


@pytest.mark.parametrize("D", [16, 64, 100, 500, 768])
def test_rounding_paths_vs_float64(D):
    """Every rounding entry at width D: the tensor-core contraction (argmin and argmax modes), the fp32 kernels behind
    ops.round_argmin / ops.logits_argmax, denoised_fn_round and get_efficient_knn.  Ids equal the float64 ones wherever the
    top-2 margin exceeds 1e-3; duplicated rows tie and the lowest id wins; rows equal to an embedding find it."""
    V, M = 729, 1000
    rng = np.random.default_rng(D)
    E = (0.1 * rng.standard_normal((V, D))).astype(np.float32)
    E[3] *= 3                                                       # a long row: x = E_3 is its own best logit too
    E[700] = E[3]                                                   # exact duplicate of row 3 (higher id)
    bias = (0.01 * rng.standard_normal(V)).astype(np.float32)
    bias[700] = bias[3]
    near = rng.integers(0, V, size=M)
    x = (E[near] + 0.05 * rng.standard_normal((M, D))).astype(np.float32)
    hits = np.arange(0, M, 7)
    x[hits] = E[near[hits]]                                         # exact hits
    x[5] = E[700]                                                   # exact hit on a tied pair: id 3
    Et, xt, bt = (torch.from_numpy(a).to(DEV) for a in (E, x, bias))
    ref_d, m_d = _f64_best(x, E)
    ref_l, m_l = _f64_best(x, E, bias)
    se = ops.SplitEmbedding(Et)
    got = {
        "tc argmin": (ops.round_argmin_tc(xt, se), ref_d, m_d),
        "tc argmax": (ops.round_argmin_tc(xt, se, cst=se.logit_cst(bt), mode=1), ref_l, m_l),
        "fp32 argmin": (ops.round_argmin(xt, Et), ref_d, m_d),
        "fp32 argmax": (ops.logits_argmax(xt, Et, bt), ref_l, m_l),
        "get_efficient_knn": (get_efficient_knn(Et, xt)[1][0], ref_d, m_d),
    }
    emb = torch.nn.Embedding(V, D, _weight=Et.clone())
    rows = denoised_fn_round(emb, xt.view(10, M // 10, D), None).view(M, D)
    for tag, (ids, ref, margin) in got.items():
        ids = ids.long().cpu().numpy()
        clear = margin > 1e-3
        assert clear.mean() > 0.5, (tag, clear.mean())           # the comparison is not vacuous
        assert np.array_equal(ids[clear], ref[clear]), tag
        assert ids[5] == 3, tag                                     # tie -> lowest id
        if ref is ref_d:
            assert np.array_equal(ids[hits], np.where(near[hits] == 700, 3, near[hits])), tag
    assert torch.equal(rows, Et[got["fp32 argmin"][0].long()])
    clear = m_d > 1e-3
    assert np.array_equal(rows.cpu().numpy()[clear], E[ref_d[clear]])


def _zero_extend(p, D, Dn):
    """the same model at width Dn > D: zero embedding columns, zero input_up_proj.0 columns, zero output_down_proj.2 rows."""
    q = dict(p)
    pad = lambda a, axis: np.concatenate([a, np.zeros(a.shape[:axis] + (Dn - D,) + a.shape[axis + 1:], a.dtype)], axis)
    q["word_embedding.weight"] = q["lm_head.weight"] = pad(p["word_embedding.weight"], 1)       # tied
    q["input_up_proj.0.weight"] = pad(p["input_up_proj.0.weight"], 1)
    q["output_down_proj.2.weight"] = pad(p["output_down_proj.2.weight"], 0)
    q["output_down_proj.2.bias"] = pad(p["output_down_proj.2.bias"], 0)
    return q


def test_padding_is_neutral():
    """D = 500 and the same parameters zero-extended to D = 512, fed the same noise (zeros in the 12 extra columns): the ids
    of every rounding call, the decoded tokens and sample[..., :500] are bit-identical."""
    D, Dn, L = 500, 512, 64
    m500, d500, p = make(D, L, seed=50)
    m512, d512, _ = make(Dn, L, seed=0, params=_zero_extend(p, D, Dn))
    cond = {k: torch.from_numpy(np.asarray(v)) for k, v in O.make_synthetic_batch("modification", 2, L, seed=6).items()}
    res = []
    for model, diffusion, width in ((m500, d500, D), (m512, d512, Dn)):
        stream = O.NoiseStream(17)

        def source(shape, kind, width=width):
            logical = tuple(shape[:2]) + (D,) + tuple(shape[3:])          # [B, L, D] or q_sample's [B, L, D, 1]
            n = stream.truncated(logical, 1) if kind == "truncated" else stream.randn(logical)
            return np.concatenate([n, np.zeros(tuple(shape[:2]) + (width - D,) + tuple(shape[3:]), np.float32)], 2)

        diffusion.noise_source = source
        diffusion.rounding_trace = []
        try:
            from musediffusion_b200.sample import sample_batch
            tok, sample = sample_batch(model, diffusion, build_model_emb(model, DEV), cond, "modification", 2000, 2000,
                                       strength=6.2 / 2000, top_p=1, return_sample=True)
            res.append((tok, sample, [ids for ids, _ in diffusion.rounding_trace]))
        finally:
            diffusion.noise_source = diffusion.rounding_trace = None
    (tok_a, s_a, ids_a), (tok_b, s_b, ids_b) = res
    assert len(ids_a) == len(ids_b) == 6
    assert all(torch.equal(a, b) for a, b in zip(ids_a, ids_b))
    assert torch.equal(tok_a, tok_b)
    assert torch.equal(s_a, s_b[..., :D]) and not s_b[..., D:].any()


@pytest.mark.parametrize("sampler", ["ddpm", "ddim"])
def test_paper_configuration_vs_oracle(sampler):
    """The reference's documented model: embedding dimension 500, max length 256, modification mode."""
    D, L = 500, 256
    model, diffusion, p = make(D, L, seed=500)
    model_emb = build_model_emb(model, DEV)
    s = O.make_schedule("sqrt", 2000)
    cond = O.make_synthetic_batch("modification", 2, L, seed=12)
    step, strength = (2000, 10.2 / 2000) if sampler == "ddpm" else (100, 0.1)    # 10 DDPM steps / DDIM gap 20, 10 steps
    record = []
    want = O.sample_batch(s, p, cond, "modification", step, O.NoiseStream(21), strength=strength, top_p=1, record=record)
    ref_ids, ref_margin = oracle_trace(s, p, record)
    tcond = {k: torch.from_numpy(np.asarray(v)) for k, v in cond.items()}
    tok, ids, _, _ = run_with_trace(model, diffusion, model_emb, tcond, "modification", step, 2000, strength, 1, 21)
    assert len(ids) == 10
    # distances between 500-wide embeddings are D/128 times those at width 128
    assert_chain_parity("hidden_dim 500, L 256, %s vs oracle" % sampler, ref_ids, ref_margin, want, ids, tok,
                        cond["input_mask"], tol_scale=D / 128)


def test_eps_prediction_ragged_length_vs_oracle():
    """predict_xstart = False at D = 100 and a ragged length: the last Linear stores its 100 real fp32 columns of Dp = 128."""
    D, L, T = 100, 75, 40
    model, diffusion, p = make(D, L, seed=100, pxs=False, T=T)
    model_emb = build_model_emb(model, DEV)
    s = O.make_schedule("sqrt", T, "", rescale_timesteps=True, predict_xstart=False)
    cond = O.make_synthetic_batch("modification", 2, L, seed=3)
    record = []
    want = O.sample_batch(s, p, cond, "modification", T, O.NoiseStream(33), strength=1.0, top_p=1, record=record)
    ref_ids, ref_margin = oracle_trace(s, p, record)
    tcond = {k: torch.from_numpy(np.asarray(v)) for k, v in cond.items()}
    tok, ids, _, _ = run_with_trace(model, diffusion, model_emb, tcond, "modification", T, T, 1.0, 1, 33)
    scale = np.maximum(1.0, np.asarray(s.sqrt_recipm1_alphas_cumprod)[[r["t"] for r in record]])
    assert_chain_parity("hidden_dim 100, L 75, predict_eps vs oracle", ref_ids, ref_margin, want, ids, tok, cond["input_mask"],
                        tol_scale=scale)


@pytest.mark.parametrize("D,pxs", [(500, True), (100, False)])
def test_graph_replay_and_shards_bit_identical(D, pxs):
    """The captured-graph loop replays the padded buffers: it equals eager launches, and two shards with `seq_offset` set
    reproduce the whole batch bit for bit."""
    L, B, steps = 64, 4, 6
    model, diffusion, _ = make(D, L, seed=7, pxs=pxs)
    fn = partial(denoised_fn_round, build_model_emb(model, DEV), dist=None)
    b = O.make_synthetic_batch("modification", B, L, seed=8)
    torch.manual_seed(5)

    def run(rows, offset, use_graph):
        diffusion._noise_calls = 0
        diffusion.seq_offset = offset
        diffusion.use_cuda_graph = use_graph
        ids = torch.from_numpy(b["input_ids"][rows]).to(DEV)
        x_start = model.get_embeds(ids)
        mask = torch.broadcast_to(torch.from_numpy(b["input_mask"][rows]).to(DEV).unsqueeze(-1), x_start.shape)
        x0 = diffusion.q_sample(x_start.unsqueeze(-1), torch.full((ids.shape[0], 1), 1999, device=DEV), mask=mask).squeeze(-1)
        out = diffusion.p_sample_loop(model, tuple(x_start.shape), noise=x0, denoised_fn=fn, model_kwargs={}, top_p=1,
                                      clamp_step=0, clamp_first=True, mask=mask, x_start=x_start, t_enc=steps, only_last=True)[-1]
        return out.clone(), x_start, mask

    try:
        eager, x_start, mask = run(slice(0, B), 0, False)
        graph = run(slice(0, B), 0, True)[0]
        assert torch.equal(eager, graph)
        assert torch.isfinite(graph).all() and torch.equal(graph[mask == 0], x_start[mask == 0])
        lo, hi = run(slice(0, 2), 0, True)[0], run(slice(2, 4), 2, True)[0]
        assert torch.equal(torch.cat([lo, hi]), graph)
    finally:
        diffusion.seq_offset = 0
        diffusion.use_cuda_graph = True


def test_weight_pack_round_trip(tmp_path):
    """A D = 500 .mdpack keeps the reference's tensor shapes (padding happens at load) and serves the same forward pass and
    decoded tokens as the state-dict path, bit for bit."""
    from musediffusion_b200 import checkpoint
    D, L = 500, 64
    model, _, p = make(D, L, seed=9)
    path = checkpoint.write_pack(str(tmp_path / "w500.mdpack"), model.state_dict(), checkpoint.model_config_of(None, model))
    header, _ = checkpoint.read_pack_header(path)
    shapes = {t["name"]: t["shape"] for t in header["tensors"]}
    assert shapes["up1_w"] == [768, D] and shapes["dn2_w"] == [D, 768] and shapes["E"] == [729, D]
    model2, _, _ = make(D, L, seed=10)                             # other weights, replaced by the pack's
    model2.load_weight_pack(path, DEV)
    x = torch.from_numpy(np.random.default_rng(4).standard_normal((2, L, D)).astype(np.float32)).to(DEV)
    t = torch.tensor([600.0, 20.0], device=DEV)
    assert torch.equal(model(x, t), model2(x, t))
    assert torch.equal(model.decode_tokens(x), model2.decode_tokens(x))


@pytest.mark.parametrize("mode", ["generation", "modification"])
def test_command_line_on_a_500_wide_checkpoint(golden_dir, tmp_path, mode):
    from musediffusion_b200.sample import main
    L = 64
    d = tmp_path / "diffusion_models"
    d.mkdir()
    raw = json.load(open(os.path.join(golden_dir, "training_args_default.json")))
    raw.update(seq_len=L, hidden_dim=500, use_corruption=False)
    (d / "training_args.json").write_text(json.dumps(raw))
    p = O.make_random_params(seed=5, seq_len=L, hidden_dim=500)
    torch.save({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in p.items()}, str(d / "model_000000.pt"))
    argv = ["--step", "20", "--batch_size", "2"]
    if mode == "generation":
        argv += ["--num_samples", "2"]                               # no meta flags: synthetic prefixes
    else:
        argv += ["--num_batches", "1", "--strength", "0.5"]
    main([mode, "--model_path", str(d / "model_000000.pt"), "--out_dir", str(tmp_path / "out")] + argv)
    out = tmp_path / "out" / "diffusion_models" / ("model_000000.pt.%s.samples" % mode)
    tokens, status = np.load(out / "tokens.npy"), np.load(out / "decode_status.npy")
    assert tokens.shape == (2, L) and status.shape == (2,)
    assert ((tokens >= 0) & (tokens < 729)).all()
