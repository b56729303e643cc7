"""DPM-Solver++(2M) on the GPU: md_dpm_solver_step against a float32 emulation of its operation order, the graph-replayed
fused loop against the eager loop and the per-step path, the per-step path against the numpy oracle under the parity
rule, first order at every index against the reference-pinned DDIM loop, and shard invariance."""
from functools import partial
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import dpm_solver_oracle as DO
import musediff_oracle as O
import parity_rule as R

pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

from musediffusion_b200 import ops  # noqa: E402
from musediffusion_b200.diffusion import dpm_solver_coefficients, dpm_solver_indices  # noqa: E402
from musediffusion_b200.initialization import create_model_and_diffusion  # noqa: E402
from musediffusion_b200.rounding import denoised_fn_round  # noqa: E402
from musediffusion_b200.sample import build_model_emb, sample_batch  # noqa: E402
from test_fused_loop_options_gpu import _Spy, _walk  # noqa: E402
from test_reverse_step_gpu import DOWNSTREAM_TOL, LOGIT_TOL, MARGIN_TOL, PhiloxStream, _oracle_ids  # noqa: E402

DEV = torch.device("cuda:0")
F32 = np.float32
SENTINEL = 0x7FC1                      # a bf16 NaN pattern no kernel writes


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


# ------------------------------------------------------------------------------------------------ 1. the kernel
def _emulate(x, p, q, row, clip, keep, x_start):
    """numpy float32 replay of dpm_solver_step_kernel: every product and sum rounded, no fused multiply-add.
    -> (x_out, history after the step)."""
    a, b, c0, c1 = (F32(v) for v in row)
    if clip == 1:
        p = np.minimum(np.maximum(p, F32(-1.0)), F32(1.0))
    d = (c0 * p + c1 * q) if c1 != 0 else c0 * p
    o = (a * x + b * d) if a != 0 else b * d
    if keep is not None:
        o = np.where(keep, x_start, o)
    assert o.dtype == F32 and p.dtype == F32
    return o, p


@pytest.mark.parametrize("D", [16, 100, 128, 500])
def test_dpm_solver_step_matches_float32_emulation(D):
    """First-order rows on a NaN-filled history (finite output, history overwritten with p), second-order rows, the final
    row (x_out == p bit for bit), each selected by the cursor (rows *cursor - 1, clamped) and as a one-row table; idx
    gather vs pred_in at clip 0 / 1 / 2; no mask, token mask, element mask; unpadded and padded bf16 copy whose pad
    columns keep a sentinel; x_out aliasing x_t."""
    B, L = 3, 37
    rng = np.random.default_rng(D)
    x = rng.standard_normal((B, L, D)).astype(F32)
    pred = (2.0 * rng.standard_normal((B, L, D))).astype(F32)
    q = rng.standard_normal((B, L, D)).astype(F32)
    x_start = rng.standard_normal((B, L, D)).astype(F32)
    E = (1.5 * rng.standard_normal((729, D))).astype(F32)
    idx = rng.integers(0, 729, (B * L,)).astype(np.int32)
    mask_tok = (rng.random((B, L)) > 0.3).astype(np.int32)
    mask_elem = (rng.random((B, L, D)) > 0.5).astype(np.int32)
    se = ops.SplitEmbedding(_dev(E))
    gathered = E[idx].reshape(B, L, D)
    ab = O.make_schedule("sqrt", 2000).alphas_cumprod
    table = dpm_solver_coefficients(ab, dpm_solver_indices(ab, 1999, 10), 2).astype(F32)
    coef = _dev(table)
    rows = {"first order": 0, "second order": 5, "final": 9}
    assert table[0, 3] == 0 and table[5, 3] != 0 and tuple(table[9]) == (0, 1, 1, 0)
    masks = {"no mask": (None, None),
             "token mask": (torch.broadcast_to(_dev(mask_tok).unsqueeze(-1), (B, L, D)), np.broadcast_to(mask_tok[..., None] == 0, (B, L, D))),
             "element mask": (_dev(mask_elem), mask_elem == 0)}
    for rname, r in rows.items():
        for select in ("cursor", "one row"):
            for clip in (0, 1, 2):
                kw = dict(pred=_dev(pred)) if clip == 0 else dict(idx=_dev(idx), E=se.E_clamped if clip == 2 else _dev(E))
                p_in = pred if clip == 0 else gathered
                for mname, (mask, keep) in masks.items():
                    for ld in (D, ops.padded_width(D) if D % 64 else D + 64):
                        tag = (D, rname, select, clip, mname, ld)
                        if select == "cursor":
                            cursor = torch.tensor([r + 1], dtype=torch.int32, device=DEV)
                            tab = coef
                        else:
                            cursor, tab = None, coef[r:r + 1].clone()
                        first = table[r, 3] == 0
                        hist = torch.full((B, L, D), float("nan"), device=DEV) if first else _dev(q)
                        ob = torch.empty((B, L, ld), dtype=torch.bfloat16, device=DEV)
                        ob.view(torch.int16).fill_(SENTINEL)
                        xt = _dev(x)
                        out = ops.dpm_solver_step(xt, tab, hist, cursor=cursor, mask=mask,
                                                  x_start=_dev(x_start) if mask is not None else None, clip=clip,
                                                  out=xt if clip == 1 else None, out_bf16=ob, **kw)
                        want, want_hist = _emulate(x, p_in, q, table[r], min(clip, 1), keep, x_start)
                        got = out.cpu().numpy()
                        assert np.array_equal(got, want), (tag, int((got != want).sum()))
                        assert np.array_equal(hist.cpu().numpy(), want_hist), tag
                        assert torch.isfinite(out).all(), tag
                        assert torch.equal(ob[..., :D].view(torch.int16), out.to(torch.bfloat16).view(torch.int16)), tag
                        assert (ob[..., D:].view(torch.int16) == SENTINEL).all(), tag
                        if rname == "final":
                            free = np.ones((B, L, D), bool) if keep is None else ~keep
                            assert np.array_equal(got[free].view(np.int32), want_hist[free].view(np.int32)), tag
    # the cursor is clamped to the table: 0 selects the first row, past the end the last
    for cur, r in ((0, 0), (99, 9)):
        hist = _dev(q)
        out = ops.dpm_solver_step(_dev(x), coef, hist, pred=_dev(pred), clip=0,
                                  cursor=torch.tensor([cur], dtype=torch.int32, device=DEV))
        assert np.array_equal(out.cpu().numpy(), _emulate(x, pred, q, table[r], 0, None, None)[0]), cur


def test_dpm_solver_step_argument_checks():
    x = torch.zeros((1, 4, 8), device=DEV)
    one, two = torch.zeros((1, 4), device=DEV), torch.zeros((2, 4), device=DEV)
    with pytest.raises(Exception):
        ops.dpm_solver_step(x, two, torch.zeros_like(x), pred=x)                    # several rows need a cursor
    with pytest.raises(Exception):
        ops.dpm_solver_step(x, one, torch.zeros_like(x), pred=x, idx=torch.zeros(4, dtype=torch.int32, device=DEV))
    with pytest.raises(Exception):
        ops.dpm_solver_step(x, one, torch.zeros_like(x), pred=x, clip=2)            # clip 2 needs gathered rows
    with pytest.raises(Exception):
        ops.dpm_solver_step(x, one, torch.zeros((1, 4, 4), device=DEV), pred=x)     # history shaped like x_t


# ------------------------------------------------------------------------------------------------ set-up
def _setup(D, L, B, T, pxs=True, seed=11, schedule="sqrt"):
    torch.manual_seed(seed)
    p = O.make_random_params(seed=seed, seq_len=L, hidden_dim=D)
    args = SimpleNamespace(hidden_dim=D, hidden_t_dim=128, vocab_size=729, seq_len=L, dropout=0.1, noise_schedule=schedule,
                           diffusion_steps=T, timestep_respacing="", rescale_timesteps=True, predict_xstart=pxs)
    model, diffusion = create_model_and_diffusion(args)
    model.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in p.items()}, strict=True)
    model.eval().requires_grad_(False).to(DEV)
    model_emb = build_model_emb(model, DEV)
    return SimpleNamespace(p=p, model=model, diffusion=diffusion, model_emb=model_emb,
                           fn=partial(denoised_fn_round, model_emb, dist=None), D=D, L=L, B=B, T=T, pxs=pxs, schedule=schedule)


def _inputs(s, mode, seed):
    cond = O.make_synthetic_batch(mode, s.B, s.L, seed=seed)
    ids = torch.from_numpy(cond["input_ids"]).to(DEV)
    x_start = s.model.get_embeds(ids)
    mask = torch.broadcast_to(torch.from_numpy(cond["input_mask"]).to(DEV).unsqueeze(-1), x_start.shape)
    return cond, x_start, mask


def _no_noise(shape, kind):
    raise AssertionError("the DPM-Solver++ loop draws no noise")


# ------------------------------------------------------------------------------------------------ 2. the fused loop
LOOPS = {
    # name: mode, width D, length L, batch B, table size T, evaluations, strength, predict_xstart, clip_denoised
    "gen-d128": dict(mode="generation", D=128, L=64, B=2, T=2000, steps=12),
    "mod-d128": dict(mode="modification", D=128, L=64, B=3, T=2000, steps=10, strength=0.6),
    "mod-d100": dict(mode="modification", D=100, L=64, B=2, T=2000, steps=8, strength=1.0),
    "gen-d500": dict(mode="generation", D=500, L=64, B=2, T=2000, steps=6),
    "mod-d128-eps": dict(mode="modification", D=128, L=64, B=2, T=40, steps=10, strength=0.5, pxs=False),
    "gen-d100-eps-noclip": dict(mode="generation", D=100, L=64, B=2, T=40, steps=8, pxs=False, clip=False),
    "mod-d128-noclip": dict(mode="modification", D=128, L=64, B=2, T=2000, steps=10, strength=0.3, clip=False),
    "base-mod-d128": dict(mode="modification", D=128, L=2096, B=1, T=2000, steps=5, strength=1.0),
}


def _loop_config(c):
    out = dict(strength=1.0, pxs=True, clip=True)
    out.update(c)
    return SimpleNamespace(**out)


@pytest.mark.parametrize("name", list(LOOPS))
def test_fused_loop_matches_eager_and_per_step_path(name):
    """dpm_solver_sample_loop on one fixed starting state, graph-replayed, eager and through the per-step path
    (noise_source set, which it never calls): every yielded state bit for bit.  Then sample_batch(sampler="dpm_solver++")
    the three ways (the per-step path fed the loop's Philox draw): final sample, decoded tokens and noise-call count."""
    c = _loop_config(LOOPS[name])
    s = _setup(c.D, c.L, c.B, c.T, pxs=c.pxs, seed=30 + sum(map(ord, name)) % 50)
    dif = s.diffusion
    cond, x_start, mask = _inputs(s, c.mode, seed=len(name))
    T = dif.num_timesteps
    t_start = T - 1 if c.mode == "generation" else int(c.strength * T) - 1
    x0 = (1.3 * torch.randn(x_start.shape, device=DEV)).contiguous()
    kw = dict(noise=x0, clip_denoised=c.clip, denoised_fn=s.fn, model_kwargs={}, mask=mask, x_start=x_start, steps=c.steps,
              t_start=t_start)
    try:
        dif.noise_source = _no_noise
        ref = dif.dpm_solver_sample_loop(s.model, tuple(x0.shape), **kw)
        dif.noise_source = None
        assert len(ref) == c.steps
        for use_graph in (True, False):
            dif.use_cuda_graph = use_graph
            got = dif.dpm_solver_sample_loop(s.model, tuple(x0.shape), **kw)
            for k, (a, b) in enumerate(zip(ref, got)):
                assert torch.equal(a, b), (name, use_graph, k, int((a != b).sum()))
        assert torch.equal(ref[-1][mask == 0], x_start[mask == 0])
        assert torch.isfinite(ref[-1]).all()
        # through sample_batch
        tcond = {k: torch.from_numpy(v) for k, v in cond.items()}
        stream = PhiloxStream()
        dif.noise_source = lambda shape, kind: stream.randn(shape)
        dif._noise_calls = 0
        tok_ref, sample_ref = sample_batch(s.model, dif, s.model_emb, tcond, c.mode, c.steps, c.T, strength=c.strength,
                                           clip_denoised=c.clip, return_sample=True, sampler="dpm_solver++")
        sample_ref = sample_ref.clone()
        calls_ref = dif._noise_calls
        assert calls_ref == stream.calls == 1
        dif.noise_source = None
        for use_graph in (True, False):
            dif.use_cuda_graph = use_graph
            dif._noise_calls = 0
            tok, sample = sample_batch(s.model, dif, s.model_emb, tcond, c.mode, c.steps, c.T, strength=c.strength,
                                       clip_denoised=c.clip, return_sample=True, sampler="dpm_solver++")
            tag = (name, use_graph)
            assert dif._noise_calls == calls_ref, tag
            assert torch.equal(sample, sample_ref), (tag, int((sample != sample_ref).sum()))
            assert torch.equal(tok, tok_ref), tag
    finally:
        dif.noise_source = None
        dif.use_cuda_graph = True
        dif._noise_calls = 0


@pytest.mark.parametrize("D,pxs", [(128, True), (100, True), (128, False)])
def test_one_captured_body_replays_every_evaluation(D, pxs, monkeypatch):
    """One graph per chain; its recorded launches equal one eager evaluation's; a replayed evaluation launches as many
    kernels as an eager one and allocates nothing."""
    s = _setup(D, 64, 2, 2000, pxs=pxs, seed=7)
    dif = s.diffusion
    _, x_start, mask = _inputs(s, "modification", seed=4)
    x0 = torch.randn(x_start.shape, device=DEV)
    n = 9
    idx = dpm_solver_indices(dif.alphas_cumprod, 1999, n)
    coef = dpm_solver_coefficients(dif.alphas_cumprod, idx, 2).astype(F32)
    spy = _Spy(dif, monkeypatch)
    per_mode = {}
    for use_graph in (False, True):
        dif.use_cuda_graph = use_graph
        spy.steps, spy.nodes = 0, []
        gen = dif._dpm_loop(s.model, tuple(x0.shape), x0, True, s.fn, {}, None, False, mask, x_start, idx, coef)
        out, deltas = _walk(gen)
        assert len(out) == n
        per_mode[use_graph] = [d[0] for d in deltas]
        if use_graph:
            assert len(spy.nodes) == 1 and spy.nodes[0] == per_mode[False][1] > 0, (spy.nodes, per_mode)
            assert all(d[1] == 0 for d in deltas[2:]), deltas
    dif.use_cuda_graph = True
    assert per_mode[True][1:] == per_mode[False][1:], per_mode


# ------------------------------------------------------------------------------------------------ 3. against the oracle
ORACLE = {
    "gen": dict(mode="generation", L=64, B=2, steps=10),
    "mod": dict(mode="modification", L=96, B=2, steps=20, strength=0.5),
    "mod-order1": dict(mode="modification", L=80, B=2, steps=12, strength=0.8, order=1),
}


@pytest.mark.parametrize("name", list(ORACLE))
def test_per_step_path_matches_oracle(name):
    """DO.dpm_solver_sample_loop from the same Philox starting draw against the per-step path (noise_source set, every
    rounding call traced): 0 parity-rule violations over the rounding calls, and decoded tokens equal wherever the ids
    never differed."""
    c = SimpleNamespace(**{**dict(strength=1.0, order=2), **ORACLE[name]})
    T, D = 2000, 128
    s = _setup(D, c.L, c.B, T, seed=60 + len(name))
    so = O.make_schedule("sqrt", T)
    cond = O.make_synthetic_batch(c.mode, c.B, c.L, seed=9 + len(name))
    x_start = O.get_embeds(s.p, cond["input_ids"])
    mask = np.broadcast_to(cond["input_mask"][..., None], x_start.shape)
    ostream = PhiloxStream()
    if c.mode == "generation":
        t_start = T - 1
        x_noised = np.where(mask == 0, x_start, ostream.randn(x_start.shape))
    else:
        t_start = int(c.strength * T) - 1
        t = np.full((c.B, 1), t_start, dtype=np.int64)
        x_noised = O.q_sample(so, x_start[..., None], t, ostream.randn(x_start.shape + (1,)), mask=mask[..., None])[..., 0]
    record = []
    out = DO.dpm_solver_sample_loop(so, s.p, x_noised, c.steps, t_start, c.order, True, True, mask, x_start, record)
    want = O.logits_argmax(s.p, out)
    assert [r["t"] for r in record] == dpm_solver_indices(so.alphas_cumprod, t_start, c.steps)
    ref_ids, ref_margin = _oracle_ids(so, s.p, record)
    dif = s.diffusion
    stream = PhiloxStream()
    dif.noise_source = lambda shape, kind: stream.randn(shape)
    dif.rounding_trace = []
    try:
        tcond = {k: torch.from_numpy(v) for k, v in cond.items()}
        if c.order == 2:
            tok = sample_batch(s.model, dif, s.model_emb, tcond, c.mode, c.steps, T, strength=c.strength, sampler="dpm_solver++")
        else:
            xs = s.model.get_embeds(tcond["input_ids"].to(DEV))
            m = torch.broadcast_to(tcond["input_mask"].to(DEV).unsqueeze(-1), xs.shape)
            xn = dif.q_sample(xs.unsqueeze(-1), torch.full((c.B, 1), t_start, device=DEV), mask=m).squeeze(-1)
            sample = dif.dpm_solver_sample_loop(s.model, tuple(xs.shape), noise=xn, denoised_fn=s.fn, mask=m, x_start=xs,
                                                steps=c.steps, t_start=t_start, order=1, only_last=True)[-1]
            tok = s.model.decode_tokens(sample)
        ids, _ = R.trace_to_numpy(dif.rounding_trace, c.B, c.L)
    finally:
        dif.noise_source = None
        dif.rounding_trace = None
    assert stream.calls == 1
    free = cond["input_mask"] != 0
    rep = R.chain_report(ref_ids, ref_margin, ids, free, MARGIN_TOL, DOWNSTREAM_TOL)
    tk = R.token_report(want, tok.cpu().numpy(), free, rep["never_divergent"], None, LOGIT_TOL)
    print("%s: %d rounding calls, id agreement %.5f, %d positions ever divergent, token agreement %.5f, violations %d + %d"
          % (name, rep["calls"], rep["id_agreement_all_calls"], rep["positions_ever_divergent"], tk["token_agreement"],
             rep["violations"], tk["token_violations"]))
    assert rep["calls"] == c.steps
    assert rep["violations"] == 0, rep
    assert tk["token_violations"] == 0, tk


# ------------------------------------------------------------------------------------------------ 4. tie to the DDIM loop
@pytest.mark.parametrize("mode", ["generation", "modification"])
def test_order1_every_index_matches_ddim_loop(mode):
    """cosine T = 30: order 1 with N = t_start + 1 evaluations is algebraically ddim_sample_loop(gap=1, eta=0), the
    reference-pinned loop.  Both on the GPU from one starting state, both traced: the DPM ids agree with the DDIM ids under
    the parity rule (the DDIM trace's margins as the reference side) and the decoded tokens are equal wherever the ids
    never differed."""
    T, L, B = 30, 64, 3
    s = _setup(128, L, B, T, seed=13, schedule="cosine")
    dif = s.diffusion
    cond, x_start, mask = _inputs(s, mode, seed=5)
    t_start = T - 1                  # the DDIM loop always starts from the top (t_enc only cuts its end)
    x0 = torch.where(mask == 0, x_start, torch.randn(x_start.shape, device=DEV)).contiguous()
    if mode == "modification":
        x0 = dif.q_sample(x_start.unsqueeze(-1), torch.full((B, 1), t_start, device=DEV), mask=mask).squeeze(-1).clone()
    common = dict(noise=x0, denoised_fn=s.fn, model_kwargs={}, mask=mask, x_start=x_start, only_last=True)
    try:
        dif.rounding_trace = []
        ddim = dif.ddim_sample_loop(s.model, tuple(x0.shape), gap=1, eta=0.0, t_enc=t_start + 1, **common)[-1].clone()
        ref_ids, ref_margin = R.trace_to_numpy(dif.rounding_trace, B, L)
        dif.rounding_trace = []
        dpm = dif.dpm_solver_sample_loop(s.model, tuple(x0.shape), steps=t_start + 1, t_start=t_start, order=1, **common)[-1]
        ids, _ = R.trace_to_numpy(dif.rounding_trace, B, L)
    finally:
        dif.rounding_trace = None
    free = cond["input_mask"] != 0
    rep = R.chain_report(ref_ids, ref_margin, ids, free, MARGIN_TOL, DOWNSTREAM_TOL)
    tok_ddim, tok_dpm = s.model.decode_tokens(ddim), s.model.decode_tokens(dpm)
    tk = R.token_report(tok_ddim.cpu().numpy(), tok_dpm.cpu().numpy(), free, rep["never_divergent"], None, LOGIT_TOL)
    err = float((dpm - ddim).abs().max() / ddim.abs().max())
    print("%s: %d calls, id agreement %.5f, %d positions ever divergent, token agreement %.5f, max-norm relative gap %.2e"
          % (mode, rep["calls"], rep["id_agreement_all_calls"], rep["positions_ever_divergent"], tk["token_agreement"], err))
    assert rep["calls"] == t_start + 1
    assert rep["violations"] == 0, rep
    assert tk["token_violations"] == 0, tk


# ------------------------------------------------------------------------------------------------ 5. sharding
def test_shard_invariance_and_determinism():
    """Generation, B = 4 in one call equals two calls of 2 at seq_offset 0 and 2 (the only draw is keyed by the global
    sequence index), bit for bit; the same call twice gives identical tokens."""
    s = _setup(128, 256, 4, 2000, seed=17)
    dif = s.diffusion
    b = O.make_synthetic_batch("generation", 4, 256, seed=2, per_row_prefix=True)
    torch.manual_seed(23)

    def run(rows, offset):
        dif._noise_calls = 0
        dif.seq_offset = offset
        cond = {k: torch.from_numpy(v[rows]) for k, v in b.items()}
        return sample_batch(s.model, dif, s.model_emb, cond, "generation", 10, 2000, return_sample=True, sampler="dpm_solver++")

    try:
        tok, full = run(slice(0, 4), 0)
        tok2, again = run(slice(0, 4), 0)
        assert torch.equal(tok, tok2) and torch.equal(full, again)
        tok_lo, lo = run(slice(0, 2), 0)
        tok_hi, hi = run(slice(2, 4), 2)
        assert torch.equal(torch.cat([lo, hi]), full)
        assert torch.equal(torch.cat([tok_lo, tok_hi]), tok)
    finally:
        dif.seq_offset = 0
