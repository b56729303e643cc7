"""Clamp gating, progressive loops and `rounding_trace` on the production loop, `GaussianDiffusion._fused_loop`.

Every chain that our denoiser can run with in-kernel noise takes the fused, graph-replayed loop; only arbitrary callables,
`noise_source` and other state shapes step through `_step`.  This file shows:

  1. which path each loop option takes, that the fused loop allocates nothing per replayed step beyond the tensors it
     hands to its caller, and that each captured body records exactly the launches of one eager step of that body;
  2. the fused loop (graph-replayed and eager) reproduces the per-step path, fed the same Philox draws, bit for bit: every
     yielded sample / pred_xstart / greedy_mean, every trace entry, the decoded tokens and the noise-call count;
  3. clamp-gated DDPM chains through the per-step path agree with the oracle's p_sample_loop under the parity rule, and
     x_{t-1} of the plain (non-rounding) steps within the north-star 1e-2."""
from functools import partial
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import musediff_oracle as O
import parity_rule as R

pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

import musediffusion_b200.diffusion as D  # noqa: E402
from musediffusion_b200 import ops  # noqa: E402
from musediffusion_b200.initialization import create_model_and_diffusion  # noqa: E402
from musediffusion_b200.rounding import denoised_fn_round  # noqa: E402
from musediffusion_b200.sample import build_model_emb  # noqa: E402
from test_reverse_step_gpu import DOWNSTREAM_TOL, MARGIN_TOL, PhiloxStream, _oracle_ids  # noqa: E402

DEV = torch.device("cuda:0")


# ------------------------------------------------------------------------------------------------ set-up
def _setup(D_, L, B, T, pxs=True, seed=11, mode="modification"):
    """model + diffusion from oracle-random weights, a synthetic batch and what the loops take for it."""
    torch.manual_seed(seed)
    p = O.make_random_params(seed=seed, seq_len=L, hidden_dim=D_)
    args = SimpleNamespace(hidden_dim=D_, hidden_t_dim=128, vocab_size=729, seq_len=L, dropout=0.1, noise_schedule="sqrt",
                           diffusion_steps=T, timestep_respacing="", rescale_timesteps=True, predict_xstart=pxs)
    model, diffusion = create_model_and_diffusion(args)
    model.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in p.items()}, strict=True)
    model.eval().requires_grad_(False).to(DEV)
    model_emb = build_model_emb(model, DEV)
    cond = O.make_synthetic_batch(mode, B, L, seed=seed % 89)
    ids = torch.from_numpy(cond["input_ids"]).to(DEV)
    x_start = model.get_embeds(ids)
    mask = torch.broadcast_to(torch.from_numpy(cond["input_mask"]).to(DEV).unsqueeze(-1), x_start.shape)
    return SimpleNamespace(p=p, model=model, diffusion=diffusion, fn=partial(denoised_fn_round, model_emb, dist=None),
                           cond=cond, x_start=x_start, mask=mask, T=T, pxs=pxs, D=D_)


def _x_init(s, t_enc):
    """the loop's starting state: x_start noised to index t_enc - 1 where the mask is set (drawn once, fixed here)."""
    t = torch.full((s.x_start.shape[0], 1), t_enc - 1, device=DEV)
    return s.diffusion.q_sample(s.x_start.unsqueeze(-1), t, mask=s.mask).squeeze(-1).clone()


class _Spy:
    """counts `_step` calls and records the launches every `_capture` records."""

    def __init__(self, diffusion, monkeypatch):
        self.steps, self.nodes = 0, []
        step = diffusion._step

        def counted(*a, **k):
            self.steps += 1
            return step(*a, **k)

        def capture(dev, fn, orig=D._capture):
            before = ops.launch_count()
            g = orig(dev, fn)
            self.nodes.append(ops.launch_count() - before)
            return g

        monkeypatch.setattr(diffusion, "_step", counted)
        monkeypatch.setattr(D, "_capture", capture)


def _ddpm(s, x0, n, clamp_step, clamp_first, progressive, **kw):
    common = dict(model=s.model, shape=tuple(x0.shape), noise=x0, denoised_fn=s.fn, model_kwargs={}, top_p=1,
                  clamp_step=clamp_step, clamp_first=clamp_first, mask=s.mask, x_start=s.x_start, t_enc=n, **kw)
    if progressive:
        return list(s.diffusion.p_sample_loop_progressive(**common))
    return [{"sample": x} for x in s.diffusion.p_sample_loop(only_last=False, **common)]


def _clamp_cases(n, T):
    return [(c, first) for c in (1, 3, n - 1, n, T + 5) for first in (True, False)]


def _rounds(indices, clamp_step, clamp_first):
    return [(i >= clamp_step) if clamp_first else not (i > clamp_step) for i in indices]


# ------------------------------------------------------------------------------------------------ 1. path selection
def _walk(gen):
    """drive a `_loop` generator: per step (launches, allocations) since the previous step, and what it yields"""
    out, deltas = [], []
    torch.cuda.synchronize()
    l0, a0 = ops.launch_count(), torch.cuda.memory_stats()["allocation.all.allocated"]
    for item in gen:
        l1, a1 = ops.launch_count(), torch.cuda.memory_stats()["allocation.all.allocated"]
        deltas.append((l1 - l0, a1 - a0))
        out.append(item)
        l0, a0 = ops.launch_count(), torch.cuda.memory_stats()["allocation.all.allocated"]
    return out, deltas


@pytest.mark.parametrize("pxs", [True, False])
def test_path_selection_launches_and_allocations(pxs, monkeypatch):
    """For clamp-gated DDPM chains (every clamp_step / clamp_first case), progressive and traced loops: `_step` never runs,
    one graph is captured per run of two or more steps, its recorded launches equal one eager step of that body, every
    step launches as many kernels graph-replayed as eager, and a replayed step allocates exactly the clones handed out
    (3 with want_aux, 2 per rounding step with a trace, none otherwise).  Arbitrary callables and noise_source step
    through `_step`; clamp_step None keeps the reference's TypeError."""
    n = 10
    s = _setup(128, 64, 2, n, pxs=pxs)
    dif = s.diffusion
    x0 = _x_init(s, n)
    idx_list = list(range(n))[::-1]
    spy = _Spy(dif, monkeypatch)
    cases = [(c, f, aux, tr) for c, f in _clamp_cases(n, n) for aux, tr in ((False, False), (True, True))]
    cases += [(0, True, True, False), (0, True, False, True)]
    for clamp_step, clamp_first, want_aux, traced in cases:
        rounds = _rounds(idx_list, clamp_step, clamp_first)
        runs = [k for k in range(n) if k == 0 or rounds[k] != rounds[k - 1]] + [n]
        per_mode = {}
        for use_graph in (False, True):
            dif.use_cuda_graph = use_graph
            dif.rounding_trace = [] if traced else None
            spy.steps, spy.nodes = 0, []
            gen = dif._loop(D._lib.STEP_DDPM, s.model, tuple(x0.shape), x0, True, s.fn, {}, None, False, 1, clamp_step,
                            clamp_first, s.mask, s.x_start, 0.0, idx_list, want_aux)
            out, deltas = _walk(gen)
            tag = (pxs, clamp_step, clamp_first, want_aux, traced, use_graph)
            assert spy.steps == 0 and len(out) == n, tag
            if traced:
                assert len(dif.rounding_trace) == sum(rounds), tag
            per_mode[use_graph] = [d[0] for d in deltas]
            if use_graph:
                long_runs = [(a, b) for a, b in zip(runs, runs[1:]) if b - a >= 2]
                assert len(spy.nodes) == len(long_runs), tag
                eager = per_mode[False]
                for (a, _), nodes in zip(long_runs, spy.nodes):
                    assert nodes == eager[a + 1] > 0, (tag, a, nodes, eager)          # step a + 1 is one eager step of the body
                for a, b in long_runs:
                    for k in range(a + 2, b):                                          # replayed steps
                        want = (3 if want_aux else 0) + (2 if traced and rounds[k] else 0)
                        assert deltas[k][1] == want, (tag, k, deltas[k])
        assert per_mode[True][1:] == per_mode[False][1:], (tag, per_mode)
    dif.rounding_trace = None
    dif.use_cuda_graph = True
    # progressive generators through the public API
    spy.steps = 0
    assert len(list(dif.p_sample_loop_progressive(s.model, tuple(x0.shape), noise=x0, denoised_fn=s.fn, top_p=1, clamp_step=3,
                                                  clamp_first=True, mask=s.mask, x_start=s.x_start))) == n
    assert len(list(dif.ddim_sample_loop_progressive(s.model, tuple(x0.shape), noise=x0, denoised_fn=s.fn, mask=s.mask,
                                                     x_start=s.x_start, gap=2))) == n // 2
    dif.p_sample_loop(s.model, tuple(x0.shape), noise=x0, denoised_fn=None, top_p=1, clamp_step=0, clamp_first=True,
                      mask=s.mask, x_start=s.x_start)
    assert spy.steps == 0
    # what cannot be captured steps through _step
    stream = PhiloxStream()
    dif.noise_source = lambda shape, kind: stream.randn(shape)
    try:
        _ddpm(s, x0, n, 0, True, False)
        assert spy.steps == n
    finally:
        dif.noise_source = None
    spy.steps = 0
    dif.p_sample_loop(s.model, tuple(x0.shape), noise=x0, denoised_fn=lambda x, t: x.clamp(-1, 1), top_p=1, clamp_step=0,
                      clamp_first=True, mask=s.mask, x_start=s.x_start)
    assert spy.steps == n
    spy.steps = 0
    dif.p_sample_loop(lambda x, ts, **kw: x * 0.5, tuple(x0.shape), noise=x0, denoised_fn=s.fn, top_p=1, clamp_step=0,
                      clamp_first=True, mask=s.mask, x_start=s.x_start, device=DEV)
    assert spy.steps == n
    with pytest.raises(TypeError):
        dif.p_sample_loop(s.model, tuple(x0.shape), noise=x0, denoised_fn=s.fn, top_p=1, mask=s.mask, x_start=s.x_start)


# ------------------------------------------------------------------------------------------------ 2. bit-identity
def _run(s, x0, n, clamp_step, clamp_first, stream=None, progressive=True, ddim=None):
    """one chain; `stream`: the per-step path fed those Philox draws.  -> (yielded dicts, trace, noise calls, tokens)"""
    dif = s.diffusion
    dif.noise_source = None if stream is None else (
        lambda shape, kind: stream.truncated(shape, 1) if kind == "truncated" else stream.randn(shape))
    dif.rounding_trace = []
    dif._noise_calls = 0
    try:
        if ddim is not None:
            gen = dif.ddim_sample_loop_progressive(s.model, tuple(x0.shape), noise=x0, denoised_fn=s.fn, mask=s.mask,
                                                   x_start=s.x_start, gap=ddim[0], eta=ddim[1], t_enc=n)
            out = list(gen)
        else:
            out = _ddpm(s, x0, n, clamp_step, clamp_first, progressive)
        return out, dif.rounding_trace, dif._noise_calls, s.model.decode_tokens(out[-1]["sample"])
    finally:
        dif.noise_source = None
        dif.rounding_trace = None


def _assert_same(tag, ref, got):
    out_r, tr_r, calls_r, tok_r = ref
    out_g, tr_g, calls_g, tok_g = got
    assert calls_g == calls_r, tag
    assert len(out_g) == len(out_r), tag
    for k, (a, b) in enumerate(zip(out_r, out_g)):
        for key in b:
            if key == "out":
                for v in ("mean", "variance", "log_variance", "pred_xstart"):
                    assert torch.equal(a["out"][v], b["out"][v]), (tag, k, v)
            else:
                assert torch.equal(a[key], b[key]), (tag, k, key, int((a[key] != b[key]).sum()))
    assert len(tr_g) == len(tr_r), tag
    for k, ((ia, ma), (ib, mb)) in enumerate(zip(tr_r, tr_g)):
        assert torch.equal(ia, ib) and torch.equal(ma, mb), (tag, "trace", k)
    assert torch.equal(tok_g, tok_r), tag


SHORT = {
    # name: width D, predict_xstart
    "d128-x0": (128, True),
    "d128-eps": (128, False),
    "d100-x0": (100, True),
    "d500-eps": (500, False),
}


@pytest.mark.parametrize("name", list(SHORT))
def test_clamp_gated_chains_match_per_step_path(name):
    """Modification chains (masked) over a 10-step table, every clamp_step / clamp_first case: the fused loop graph-replayed
    and eager (progressive, so every step's sample / pred_xstart / greedy_mean / variances are compared) and graph-replayed
    through p_sample_loop, against the per-step path fed the loop's Philox draws."""
    D_, pxs = SHORT[name]
    n = 10
    s = _setup(D_, 64, 2, n, pxs=pxs, seed=20 + D_)
    x0 = _x_init(s, n)
    for clamp_step, clamp_first in _clamp_cases(n, n):
        ref = _run(s, x0, n, clamp_step, clamp_first, stream=PhiloxStream())
        assert ref[2] == n and len(ref[1]) == sum(_rounds(range(n - 1, -1, -1), clamp_step, clamp_first))
        for use_graph in (True, False):
            s.diffusion.use_cuda_graph = use_graph
            _assert_same((name, clamp_step, clamp_first, use_graph), ref, _run(s, x0, n, clamp_step, clamp_first))
        s.diffusion.use_cuda_graph = True
        ref_plain = [{"sample": o["sample"]} for o in ref[0]]
        _assert_same((name, clamp_step, clamp_first, "p_sample_loop"), (ref_plain,) + ref[1:],
                     _run(s, x0, n, clamp_step, clamp_first, progressive=False))


@pytest.mark.parametrize("gap,eta", [(1, 0.0), (2, 0.3)])
def test_ddim_progressive_matches_per_step_path(gap, eta):
    """ddim_sample_loop_progressive (masked modification chain, D = 100): every yielded sample and pred_xstart, trace,
    tokens and noise calls, graph-replayed and eager."""
    s = _setup(100, 64, 3, 2000, seed=5)
    n = 8
    x0 = _x_init(s, n * gap)
    ref = _run(s, x0, n, None, None, stream=PhiloxStream(), ddim=(gap, eta))
    assert len(ref[0]) == n and len(ref[1]) == n
    for use_graph in (True, False):
        s.diffusion.use_cuda_graph = use_graph
        _assert_same(("ddim", gap, eta, use_graph), ref, _run(s, x0, n, None, None, ddim=(gap, eta)))
    s.diffusion.use_cuda_graph = True


@pytest.mark.parametrize("clamp_step,clamp_first", [(1997, True), (1996, False)])
def test_clamp_gated_base_shape_matches_per_step_path(clamp_step, clamp_first):
    """The base shape L = 2096 on the 2000-step table, 6 DDPM steps from the top, rounding and plain runs of 3 steps each."""
    s = _setup(128, 2096, 1, 2000, seed=3)
    n = 6
    x0 = _x_init(s, n)
    ref = _run(s, x0, n, clamp_step, clamp_first, stream=PhiloxStream())
    assert len(ref[1]) == 3
    for use_graph in (True, False):
        s.diffusion.use_cuda_graph = use_graph
        _assert_same(("base", clamp_step, clamp_first, use_graph), ref, _run(s, x0, n, clamp_step, clamp_first))
    s.diffusion.use_cuda_graph = True


# ------------------------------------------------------------------------------------------------ 3. against the oracle
@pytest.mark.parametrize("D_,clamp_step,clamp_first", [(128, 1995, True), (128, 1995, False), (100, 1996, False)])
def test_clamp_gated_per_step_path_matches_oracle(D_, clamp_step, clamp_first):
    """O.p_sample_loop with the same clamp_step / clamp_first on a PhiloxStream against the per-step path fed the same draws:
    0 parity-rule violations over the rounding calls, and on every plain step x_{t-1} within 1e-2 (max-norm relative) of
    the oracle wherever the rounding ids never differed."""
    n, T = 8, 2000
    s = _setup(D_, 64, 3, T, seed=40 + D_)
    so = O.make_schedule("sqrt", T, "", rescale_timesteps=True, predict_xstart=True)
    cond = s.cond
    x_start = O.get_embeds(s.p, cond["input_ids"])
    mask = np.broadcast_to(cond["input_mask"][..., None], x_start.shape)
    ostream = PhiloxStream()
    t = np.full((x_start.shape[0], 1), n - 1, dtype=np.int64)
    x_noised = O.q_sample(so, x_start[..., None], t, ostream.randn(x_start.shape + (1,)), mask=mask[..., None])[..., 0]
    record = []
    O.p_sample_loop(so, s.p, x_noised, ostream, True, True, 1, clamp_step, clamp_first, mask, x_start, n, record)
    rounds = _rounds([r["t"] for r in record], clamp_step, clamp_first)
    assert 0 < sum(rounds) < n
    ref_ids, ref_margin = _oracle_ids(so, s.p, [r for r, k in zip(record, rounds) if k])
    # the package: q_sample then the loop, every draw from the same stream
    stream = PhiloxStream()
    dif = s.diffusion
    dif.noise_source = lambda shape, kind: stream.truncated(shape, 1) if kind == "truncated" else stream.randn(shape)
    dif.rounding_trace = []
    dif._noise_calls = 0
    try:
        x0 = _x_init(s, n)
        samples = [o["sample"].cpu().numpy() for o in _ddpm(s, x0, n, clamp_step, clamp_first, False)]
        ids, _ = R.trace_to_numpy(dif.rounding_trace, *cond["input_mask"].shape)
    finally:
        dif.noise_source = None
        dif.rounding_trace = None
    assert stream.calls == 1 + n
    free = cond["input_mask"] != 0
    scale = D_ / 128
    rep = R.chain_report(ref_ids, ref_margin, ids, free, MARGIN_TOL * scale, DOWNSTREAM_TOL * scale)
    print("clamp_step %d clamp_first %s D %d: %d rounding calls, id agreement %.5f, %d positions ever divergent, violations %d"
          % (clamp_step, clamp_first, D_, rep["calls"], rep["id_agreement_all_calls"], rep["positions_ever_divergent"],
             rep["violations"]))
    assert rep["violations"] == 0, rep
    ok = np.broadcast_to((rep["never_divergent"] | ~free)[..., None], samples[0].shape)
    for k, r in enumerate(record):
        if rounds[k]:
            continue
        err = float(np.abs(samples[k] - r["sample"])[ok].max() / np.abs(r["sample"]).max())
        print("  plain step t = %d: x_{t-1} max-norm relative error %.2e" % (r["t"], err))
        assert err <= 1e-2, (r["t"], err)
