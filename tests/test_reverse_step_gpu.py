"""The production reverse step against independent references.

The sampling path users get (and bench.py times) is `GaussianDiffusion._fused_loop`: `md_step_advance` publishes the step's
schedule index, model timestep and Philox counter in device memory, the last Linear emits the [hi | lo] split the rounding
consumes, and `md_posterior_step` gathers rows of the pre-clamped embedding (clip = 2) and draws its noise in-kernel.  The
oracle chains elsewhere inject their noise, which sends `_loop` down the per-step `_step` path instead.  This file closes
the gap with a chain of bit-level links:

  A. the in-kernel noise of md_posterior_step (both kernels) and md_q_sample equals md_fill_normal bit for bit;
  B. both posterior kernels equal each other and a numpy float32 emulation of their operation order;
  C. md_step_advance publishes the tables and counter it documents;
  D. the per-step path fed the Philox draws as explicit noise agrees with the oracle under the parity rule, and the fused
     loop (graph-replayed and eager) reproduces that per-step path bit for bit."""
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

from musediffusion_b200 import _lib, ops  # noqa: E402
from musediffusion_b200.initialization import create_model_and_diffusion  # noqa: E402
from musediffusion_b200.rounding import denoised_fn_round  # noqa: E402
from musediffusion_b200.sample import build_model_emb, sample_batch  # noqa: E402

DEV = torch.device("cuda:0")
F32 = np.float32
LOGIT_TOL = 1e-3       # the parity rule's tolerances, as in test_sampling_gpu.py
DOWNSTREAM_TOL = 1.0
MARGIN_TOL = 0.5
SEED = 0xD1B54A32D192ED03          # a 64-bit Philox key: both key words are non-zero
MODES = {"ddpm": _lib.STEP_DDPM, "ddim": _lib.STEP_DDIM}


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _schedule(T=2000):
    s = O.make_schedule("sqrt", T)
    ops.set_schedule({n: getattr(s, n) for n in ops.TABLE_ORDER})
    return s


def _bf16_buffer(B, L, ld, sentinel=None):
    """bf16 [B, L, ld]; with `sentinel` every element holds that bit pattern (to see which columns a kernel writes)."""
    out = torch.empty((B, L, ld), dtype=torch.bfloat16, device=DEV)
    if sentinel is not None:
        out.view(torch.int16).fill_(sentinel)
    return out


# ------------------------------------------------------------------------------------------------ A. in-kernel noise
def _routes(D, mask_tok):
    """(name, mask, out_bf16 width) triples covering both posterior kernels at width D (elementwise.cu dispatch: D = 128 with a
    token-broadcast mask and an unpadded bf16 copy takes posterior_step_d128_kernel, everything else the generic kernel)."""
    B, L = mask_tok.shape
    tok = torch.broadcast_to(_dev(mask_tok).unsqueeze(-1), (B, L, D))                 # stride-0 expand: mask_d_stride 0
    elem = tok.contiguous()                                                           # same values, mask_d_stride 1
    if D == 128:
        return [("d128", tok, D), ("generic, element mask", elem, D), ("generic, padded bf16", tok, 192)]
    return [("generic", tok, D), ("generic, padded bf16", tok, ops.padded_width(D)), ("generic, element mask", elem, D)]


@pytest.mark.parametrize("D", [16, 100, 128, 500])
@pytest.mark.parametrize("mode", ["ddpm", "ddim"])
def test_posterior_in_kernel_noise_equals_fill_normal(mode, D):
    """md_posterior_step with noise = None draws, for element e of sequence b, the Philox value md_fill_normal writes at global
    element (seq_offset + b) L D + e: equal samples and bf16 copies for every quantile branch (top_p 0 and > 1: general,
    0 < top_p <= 1: central polynomial), sequence offset, per-sequence t with a t = 0 row (no noise there) and shared t, on
    both kernels; with `step_counter_dev` the counter comes from device memory and the argument counter is ignored."""
    _schedule()
    B, L = 3, 37
    rng = np.random.default_rng(D)
    x = rng.standard_normal((B, L, D)).astype(F32)
    pred = (1.5 * rng.standard_normal((B, L, D))).astype(F32)
    x_start = rng.standard_normal((B, L, D)).astype(F32)
    mask_tok = (rng.random((B, L)) > 0.25).astype(np.int32)
    eta = 0.0 if mode == "ddpm" else 0.5
    for top_p in (0.0, 0.5, 1.0, 2.0):
        for off in (0, 3):
            for t in (np.array([1999, 0, 700]), np.array([650])):
                c = 1000 + 17 * off + int(10 * top_p) + len(t)
                noise = ops.fill_normal((B, L, D), DEV, seed=SEED, step_counter=c, elem_offset=off * L * D, top_p=top_p)
                ctr = torch.tensor([c], dtype=torch.int64, device=DEV)
                for name, mask, ld in _routes(D, mask_tok):
                    kw = dict(pred=_dev(pred), seed=SEED, seq_offset=off, mask=mask, x_start=_dev(x_start), eta=eta, clip=True,
                              top_p=top_p)
                    tag = (mode, D, top_p, off, t.tolist(), name)
                    b_in, b_ex, b_dev = (_bf16_buffer(B, L, ld, 0) for _ in range(3))
                    got = ops.posterior_step(_dev(x), _dev(t), MODES[mode], noise=None, step_counter=c, out_bf16=b_in, **kw)
                    want = ops.posterior_step(_dev(x), _dev(t), MODES[mode], noise=noise, step_counter=c + 1, out_bf16=b_ex, **kw)
                    from_dev = ops.posterior_step(_dev(x), _dev(t), MODES[mode], noise=None, step_counter=c + 5, out_bf16=b_dev,
                                                  step_counter_dev=ctr, **kw)
                    assert torch.equal(got, want), tag
                    assert torch.equal(b_in, b_ex), tag
                    assert torch.equal(from_dev, want) and torch.equal(b_dev, b_ex), tag
                    # the noise is not vacuous: without it the free positions of a t != 0 row move
                    quiet = ops.posterior_step(_dev(x), _dev(t), MODES[mode], noise=torch.zeros_like(noise), **kw)
                    free = torch.broadcast_to(_dev(mask_tok).bool().unsqueeze(-1), (B, L, D))
                    assert not torch.equal(quiet[free], want[free]), tag


@pytest.mark.parametrize("D", [16, 100, 128, 500])
def test_q_sample_in_kernel_noise_equals_fill_normal(D):
    """md_q_sample / md_q_sample_ld with noise = None: the untruncated Philox draws of md_fill_normal, with t per sequence and
    with t = None (the generation-mode initialisation: noise wherever the mask is set)."""
    _schedule()
    B, L = 3, 29
    rng = np.random.default_rng(D + 1)
    x0 = rng.standard_normal((B, L, D)).astype(F32)
    mask_tok = (rng.random((B, L)) > 0.3).astype(np.int32)
    for t in (_dev(np.array([74, 1999, 0])), None):
        for off in (0, 3):
            for ld in sorted({D, ops.padded_width(D)}):
                c = 3 + off
                noise = ops.fill_normal((B, L, D), DEV, seed=SEED, step_counter=c, elem_offset=off * L * D, top_p=0.0)
                b_in, b_ex = _bf16_buffer(B, L, ld, 0), _bf16_buffer(B, L, ld, 0)
                got = ops.q_sample(_dev(x0), t, noise=None, seed=SEED, step_counter=c, seq_offset=off, mask=_dev(mask_tok),
                                   out_bf16=b_in)
                want = ops.q_sample(_dev(x0), t, noise=noise, seed=SEED, step_counter=c + 1, seq_offset=off, mask=_dev(mask_tok),
                                    out_bf16=b_ex)
                tag = (D, None if t is None else t.tolist(), off, ld)
                assert torch.equal(got, want), tag
                assert torch.equal(b_in, b_ex), tag
                if t is None:
                    keep = np.broadcast_to(mask_tok[..., None] == 0, x0.shape)
                    assert np.array_equal(got.cpu().numpy(), np.where(keep, x0, noise.cpu().numpy())), tag


# ------------------------------------------------------------------------------------------------ B. posterior-step precision
def _kernel_ddpm_sd(T):
    """the DDPM noise scale md_posterior_step uses at each schedule index 0..T-1: a step from x = pred = 0 with unit noise
    returns mean + sd * 1 = 0 + sd exactly."""
    z = torch.zeros((T, 1, 4), dtype=torch.float32, device=DEV)
    out = ops.posterior_step(z, torch.arange(T, device=DEV), _lib.STEP_DDPM, pred=z, noise=torch.ones_like(z), clip=False)
    return out[:, 0, 0].cpu().numpy()


def test_ddpm_noise_scale_is_expf_within_2ulp():
    """sd = (t != 0) * expf(0.5 * model_log_variance[t]): expf is the one operation of the posterior step that is not
    IEEE-rounded; CUDA bounds its error by 2 ulp.  Checked at every index of the 2000-step table against float64; t = 0 has
    no noise."""
    s = _schedule()
    sd = _kernel_ddpm_sd(2000)
    lv = np.asarray(s.model_log_variance, dtype=np.float64).astype(F32)
    exact = np.exp(0.5 * lv.astype(np.float64))
    assert sd[0] == 0.0
    ulps = np.abs(sd[1:].astype(np.float64) - exact[1:]) / np.spacing(exact[1:].astype(F32)).astype(np.float64)
    print("DDPM noise scale: max error %.3f ulp, %d of %d indices correctly rounded" % (ulps.max(), int((ulps <= 0.5).sum()),
                                                                                        len(ulps)))
    assert ulps.max() <= 2.0, ulps.max()


def _emulate(s, mode, x, p, n, t, eta, clip, keep=None, x_start=None):
    """numpy float32 replay of elementwise.cu step_coef / step_mean / the sample update: every operation IEEE-rounded in the
    kernel's order, no fused multiply-add.  `t` holds one schedule index per sequence.  The DDPM noise scale is the kernel's
    own expf value (checked to 2 ulp by test_ddpm_noise_scale_is_expf_within_2ulp), gated by t != 0 here.  Returns
    (pred, mean, sample)."""
    tab = lambda name: np.asarray(getattr(s, name), dtype=np.float64).astype(F32)[np.asarray(t)].reshape(-1, 1, 1)
    one = F32(1.0)
    nz = (np.asarray(t) != 0).astype(F32).reshape(-1, 1, 1)
    if clip == 1:
        p = np.minimum(np.maximum(p, F32(-1.0)), one)
    if mode == "ddpm":
        c1, c2 = tab("posterior_mean_coef1"), tab("posterior_mean_coef2")
        sd = nz * _kernel_ddpm_sd(s.num_timesteps)[np.asarray(t)].reshape(-1, 1, 1)
        mean = c1 * p + c2 * x
    else:
        sr, srm1 = tab("sqrt_recip_alphas_cumprod"), tab("sqrt_recipm1_alphas_cumprod")
        ab, abp = tab("alphas_cumprod"), tab("alphas_cumprod_prev")
        sigma = (F32(eta) * np.sqrt((one - abp) / (one - ab))) * np.sqrt(one - ab / abp)
        ca, cb = np.sqrt(abp), np.sqrt((one - abp) - sigma * sigma)
        sd = nz * sigma
        mean = p * ca + cb * ((sr * x - p) / srm1)
    sample = mean + sd * n
    if keep is not None:
        sample = np.where(keep, x_start, sample)
    for a in (p, mean, sample):
        assert a.dtype == F32
    return p, mean, sample


def _assert_matches_emulation(tag, got, ref):
    """pred_out, mean_out and the sample bit for bit."""
    for what, g, r in zip(("pred", "mean", "sample"), got, ref):
        g = g.cpu().numpy()
        assert np.array_equal(g, r), (tag, what, int((g != r).sum()), float(np.abs(g - r).max()))


def _run_step(x, t, mode, route_mask, x_start, ld, **kw):
    """one posterior step with pred_out / mean_out and a sentinel-filled bf16 copy of row stride ld; checks the bf16 copy
    (columns < D equal x_out rounded to bf16, columns >= D untouched) and returns (pred, mean, sample)."""
    B, L, D = x.shape
    pred_out, mean_out = torch.empty_like(x), torch.empty_like(x)
    sentinel = 0x7FC1                                                                 # a bf16 NaN pattern no kernel writes
    ob = _bf16_buffer(B, L, ld, sentinel)
    out = ops.posterior_step(x, t, mode, mask=route_mask, x_start=x_start, out_bf16=ob, pred_out=pred_out, mean_out=mean_out,
                             **kw)
    assert torch.equal(ob[..., :D].view(torch.int16), out.to(torch.bfloat16).view(torch.int16))
    assert (ob[..., D:].view(torch.int16) == sentinel).all()
    return pred_out, mean_out, out


def _step_inputs(D, seed, B=3, L=41):
    rng = np.random.default_rng(seed)
    return SimpleNamespace(
        x=rng.standard_normal((B, L, D)).astype(F32),
        pred=(2.0 * rng.standard_normal((B, L, D))).astype(F32),            # |pred| > 1 often: the clamp matters
        n=rng.standard_normal((B, L, D)).astype(F32),
        x_start=rng.standard_normal((B, L, D)).astype(F32),
        E=(1.5 * rng.standard_normal((729, D))).astype(F32),                # N(0, 1.5^2) rows: clip = 2 is not vacuous
        idx=rng.integers(0, 729, (B * L,)).astype(np.int32),
        mask_tok=(rng.random((B, L)) > 0.3).astype(np.int32),
        mask_elem=(rng.random((B, L, D)) > 0.5).astype(np.int32))


T_CASES = [np.array([1999, 0, 3]), np.array([0, 0, 1000]), np.array([700])]         # per sequence with t = 0 rows, shared


@pytest.mark.parametrize("mode,eta", [("ddpm", 0.0), ("ddim", 0.0), ("ddim", 0.5)])
@pytest.mark.parametrize("D", [16, 100, 128, 500])
def test_posterior_step_matches_float32_emulation(mode, eta, D):
    """The generic posterior kernel against `_emulate` at clip 0 (pred input), 1 (gathered E rows, clamped in the kernel) and
    2 (gathered rows of SplitEmbedding.E_clamped: equal to clip 1 bit for bit), token-broadcast / element / no mask,
    per-sequence and shared t.  The bf16 copy has a padded row stride (which routes D = 128 here too): its pad columns are
    never written."""
    s = _schedule()
    a = _step_inputs(D, seed=D)
    B, L = a.mask_tok.shape
    se = ops.SplitEmbedding(_dev(a.E))
    assert not torch.equal(se.E_clamped, _dev(a.E))
    gathered = a.E[a.idx].reshape(B, L, D)
    ld = ops.padded_width(D) if D % 64 else D + 64
    masks = {"token mask": (torch.broadcast_to(_dev(a.mask_tok).unsqueeze(-1), (B, L, D)),
                            np.broadcast_to(a.mask_tok[..., None] == 0, (B, L, D))),
             "element mask": (_dev(a.mask_elem), a.mask_elem == 0),
             "no mask": (None, None)}
    for t in T_CASES:
        t_rows = np.broadcast_to(t, (B,))
        for mname, (mask, keep) in masks.items():
            x_start = _dev(a.x_start) if mask is not None else None
            common = dict(noise=_dev(a.n), eta=eta)
            by_clip = {}
            for clip in (0, 1, 2):
                if clip == 0:
                    kw, p_in = dict(pred=_dev(a.pred)), a.pred
                else:
                    kw, p_in = dict(idx=_dev(a.idx), E=se.E_clamped if clip == 2 else _dev(a.E)), gathered
                tag = (mode, eta, D, t.tolist(), mname, clip)
                got = _run_step(_dev(a.x), _dev(t), MODES[mode], mask, x_start, ld, clip=clip, **kw, **common)
                ref = _emulate(s, mode, a.x, p_in, a.n, t_rows, eta, min(clip, 1), keep, a.x_start)
                _assert_matches_emulation(tag, got, ref)
                by_clip[clip] = got
            assert all(torch.equal(u, v) for u, v in zip(by_clip[1], by_clip[2]))


@pytest.mark.parametrize("mode,eta", [("ddpm", 0.0), ("ddim", 0.0), ("ddim", 0.3)])
def test_d128_and_generic_posterior_kernels_agree(mode, eta):
    """posterior_step_d128_kernel (token-broadcast or no mask, bf16 row stride 128) and posterior_step_kernel (the same mask
    laid out per element, or a bf16 copy of row stride 192) on identical D = 128 inputs: x_out, pred_out, mean_out and the
    bf16 copy bit for bit, clip 0 / 1 / 2, t shared or per sequence with t = 0 rows; both equal the float32 emulation."""
    s = _schedule()
    D = 128
    a = _step_inputs(D, seed=128 + int(10 * eta))
    B, L = a.mask_tok.shape
    se = ops.SplitEmbedding(_dev(a.E))
    gathered = a.E[a.idx].reshape(B, L, D)
    tok = torch.broadcast_to(_dev(a.mask_tok).unsqueeze(-1), (B, L, D))
    keep = np.broadcast_to(a.mask_tok[..., None] == 0, (B, L, D))
    for t in T_CASES:
        for clip in (0, 1, 2):
            kw = dict(pred=_dev(a.pred)) if clip == 0 else dict(idx=_dev(a.idx), E=se.E_clamped if clip == 2 else _dev(a.E))
            kw.update(noise=_dev(a.n), eta=eta, clip=clip)
            p_in = a.pred if clip == 0 else gathered
            for masked in (True, False):
                mask_fast, mask_gen = (tok, tok.contiguous()) if masked else (None, None)
                x_start = _dev(a.x_start) if masked else None
                fast = _run_step(_dev(a.x), _dev(t), MODES[mode], mask_fast, x_start, D, **kw)
                generic_elem = _run_step(_dev(a.x), _dev(t), MODES[mode], mask_gen, x_start, D, **kw) if masked else None
                generic_ld = _run_step(_dev(a.x), _dev(t), MODES[mode], mask_fast, x_start, 192, **kw)
                tag = (mode, eta, t.tolist(), clip, masked)
                for other in (generic_elem, generic_ld):
                    if other is not None:
                        assert all(torch.equal(u, v) for u, v in zip(fast, other)), tag
                ref = _emulate(s, mode, a.x, p_in, a.n, np.broadcast_to(t, (B,)), eta, min(clip, 1),
                               keep if masked else None, a.x_start)
                _assert_matches_emulation(tag, fast, ref)


# ------------------------------------------------------------------------------------------------ C. md_step_advance
def test_step_advance_publishes_the_step_tables():
    """k = cursor: t_cur = t_idx[min(k, n-1)], tm_cur = t_model[min(k, n-1)], ctr_cur = ctr_base + k, cursor = k + 1, over
    n + 2 calls (the last two clamp to the final entry; the counter keeps counting)."""
    t_idx = np.array([1999, 1500, 37, 1, 0], dtype=np.int32)
    t_model = np.array([999.5, 750.25, 18.5, 0.5, 0.125], dtype=np.float32)     # distinct from t_idx at every entry
    n = len(t_idx)
    base = (1 << 40) + 3                                                          # a counter past 32 bits
    cursor = torch.zeros(1, dtype=torch.int32, device=DEV)
    t_cur = torch.full((1,), -1, dtype=torch.int32, device=DEV)
    tm_cur = torch.full((1,), -1.0, dtype=torch.float32, device=DEV)
    ctr_cur = torch.zeros(1, dtype=torch.int64, device=DEV)
    for k in range(n + 2):
        ops.step_advance(cursor, _dev(t_idx), _dev(t_model), t_cur, tm_cur, ctr_cur, base)
        kk = min(k, n - 1)
        assert int(cursor.item()) == k + 1
        assert int(t_cur.item()) == t_idx[kk]
        assert tm_cur.cpu().numpy()[0] == t_model[kk]
        assert int(ctr_cur.item()) == base + k


# ------------------------------------------------------------------------------------------------ D. the loop vs the oracle
class PhiloxStream:
    """Duck-types O.NoiseStream with the package's own Philox draws: the k-th call returns md_fill_normal at counter k, keyed
    by torch.initial_seed() and the global index of the first sequence, the way GaussianDiffusion counts its noise calls
    (the q_sample / generation initialisation draws counter 1, reverse step j counter 1 + j)."""

    def __init__(self, seq_offset=0):
        self.seed = int(torch.initial_seed()) & (2 ** 64 - 1)
        self.seq_offset = seq_offset
        self.calls = 0

    def _draw(self, shape, top_p):
        self.calls += 1
        n = ops.fill_normal(tuple(shape), DEV, seed=self.seed, step_counter=self.calls,
                            elem_offset=self.seq_offset * int(np.prod(shape[1:])), top_p=top_p)
        return n.cpu().numpy()

    def randn(self, shape):
        return self._draw(shape, 0.0)

    def truncated(self, shape, top_p):
        return self._draw(shape, float(top_p) if top_p is not None and top_p > 0 else 0.0)


CHAINS = {
    # name: mode, width D, length L, batch B, table size T, --step, strength, top_p, eta, clip_denoised, predict_xstart
    "mod-ddpm-central": dict(mode="modification", D=128, L=64, B=3, T=2000, step=2000, strength=6.2 / 2000, top_p=1),
    "gen-ddpm-general": dict(mode="generation", D=128, L=96, B=2, T=10, step=10, top_p=2),
    "mod-ddim-eta": dict(mode="modification", D=128, L=64, B=2, T=2000, step=100, strength=6.2 / 100, eta=0.3),
    "mod-ddpm-eps": dict(mode="modification", D=128, L=64, B=2, T=40, step=40, strength=8.2 / 40, top_p=1, pxs=False),
    "mod-ddpm-noclip": dict(mode="modification", D=128, L=64, B=2, T=2000, step=2000, strength=5.2 / 2000, top_p=1, clip=False),
    "mod-ddpm-d100": dict(mode="modification", D=100, L=64, B=2, T=2000, step=2000, strength=5.2 / 2000, top_p=1, seq_offset=3),
    "mod-ddpm-d500": dict(mode="modification", D=500, L=64, B=2, T=2000, step=2000, strength=5.2 / 2000, top_p=1),
    "gen-ddpm-shard": dict(mode="generation", D=128, L=64, B=4, rows=slice(2, 4), T=6, step=6, top_p=1),
    "base-mod-ddpm": dict(mode="modification", D=128, L=2096, B=1, T=2000, step=2000, strength=4.2 / 2000, top_p=1),
}


def _chain_config(chain):
    c = dict(strength=1.0, top_p=0, eta=0.0, clip=True, pxs=True, rows=None, seq_offset=0)
    c.update(chain)
    if c["rows"] is not None:
        c["seq_offset"] = c["rows"].start
    return SimpleNamespace(**c)


def _oracle_chain(c, s, p, cond, stream, record):
    """O.sample_batch, or its modification branch with O.ddim_sample_loop at eta > 0 (sample_batch runs DDIM at eta 0)."""
    if c.eta == 0.0:
        return O.sample_batch(s, p, cond, c.mode, c.step, stream, strength=c.strength, top_p=c.top_p, clip_denoised=c.clip,
                              record=record)
    assert c.mode == "modification" and c.step != c.T
    x_start = O.get_embeds(p, cond["input_ids"])
    mask = np.broadcast_to(cond["input_mask"][..., None], x_start.shape)
    noising_t = int(c.step * c.strength)
    t = np.full((x_start.shape[0], 1), noising_t - 1, dtype=np.int64)
    x_noised = O.q_sample(s, x_start[..., None], t, stream.randn(x_start.shape + (1,)), mask=mask[..., None])[..., 0]
    out = O.ddim_sample_loop(s, p, x_noised, stream, c.clip, True, mask, x_start, c.T // c.step, c.eta, noising_t, record)
    return O.logits_argmax(p, out)


def _package_chain(c, model, diffusion, model_emb, cond):
    """sample_batch (run/sample.py:177-220), or its modification branch with ddim_sample_loop at eta > 0 -> (tokens, sample)."""
    if c.eta == 0.0:
        return sample_batch(model, diffusion, model_emb, cond, c.mode, c.step, c.T, strength=c.strength, top_p=c.top_p,
                            clip_denoised=c.clip, return_sample=True)
    ids = cond["input_ids"].to(DEV)
    x_start = model.get_embeds(ids)
    mask = torch.broadcast_to(cond["input_mask"].to(DEV).unsqueeze(-1), x_start.shape)
    noising_t = int(c.step * c.strength)
    x_noised = diffusion.q_sample(x_start.unsqueeze(-1), torch.full((ids.shape[0], 1), noising_t - 1, device=DEV),
                                  mask=mask).squeeze(-1)
    sample = diffusion.ddim_sample_loop(model=model, shape=tuple(x_start.shape), noise=x_noised, clip_denoised=c.clip,
                                        denoised_fn=partial(denoised_fn_round, model_emb, dist=None), model_kwargs={},
                                        mask=mask, x_start=x_start, gap=c.T // c.step, eta=c.eta, t_enc=noising_t,
                                        only_last=True)[-1]
    return model.decode_tokens(sample), sample


def _oracle_ids(s, p, record):
    """ids + top-2 margins of every rounding call of an oracle chain (x0 from eps first when the model predicts eps)."""
    fixed = []
    for r in record:
        mo = r["model_output"]
        if not s.predict_xstart:
            t = np.full((mo.shape[0],), r["t"], dtype=np.int64)
            mo = O.extract(s.sqrt_recip_alphas_cumprod, t, mo.ndim) * r["x_t"] - O.extract(s.sqrt_recipm1_alphas_cumprod, t, mo.ndim) * mo
        fixed.append({"model_output": mo.astype(F32)})
    return R.oracle_chain_trace(fixed, p["word_embedding.weight"])


@pytest.mark.parametrize("name", list(CHAINS))
def test_fused_loop_matches_oracle_through_per_step_path(name):
    """1. The oracle runs the chain on a PhiloxStream.  2. The per-step path (`noise_source` = another PhiloxStream, every
    rounding call traced) agrees with it under the parity rule.  3. The production loop (in-kernel noise, no trace), graph-
    replayed and eager, reproduces the per-step path's final sample and decoded tokens bit for bit and counts the same noise
    calls: step advance, counter base, pre-clamped embedding, split epilogue and in-kernel noise are those of step 2."""
    _check_chain(name, CHAINS[name])


def _check_chain(name, chain):
    """the three steps of test_fused_loop_matches_oracle_through_per_step_path for one CHAINS-style entry"""
    c = _chain_config(chain)
    seed = 1000 + sum(map(ord, name))
    torch.manual_seed(seed)
    p = O.make_random_params(seed=seed % 997, seq_len=c.L, hidden_dim=c.D)
    args = SimpleNamespace(hidden_dim=c.D, hidden_t_dim=128, vocab_size=729, seq_len=c.L, dropout=0.1, noise_schedule="sqrt",
                           diffusion_steps=c.T, timestep_respacing="", rescale_timesteps=True, predict_xstart=c.pxs)
    model, diffusion = create_model_and_diffusion(args)
    model.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in p.items()}, strict=True)
    model.eval().requires_grad_(False).to(DEV)
    model_emb = build_model_emb(model, DEV)
    s = O.make_schedule("sqrt", c.T, "", rescale_timesteps=True, predict_xstart=c.pxs)
    full = O.make_synthetic_batch(c.mode, c.B, c.L, seed=seed % 89)
    rows = c.rows if c.rows is not None else slice(None)
    cond = {k: np.asarray(v)[rows] for k, v in full.items()}
    tcond = {k: torch.from_numpy(v) for k, v in cond.items()}
    # 1. oracle
    record = []
    want = _oracle_chain(c, s, p, cond, PhiloxStream(c.seq_offset), record)
    steps = len(record)
    assert steps >= diffusion.GRAPH_MIN_STEPS
    ref_ids, ref_margin = _oracle_ids(s, p, record)
    fused = []                                                  # the `capture` flag of every _fused_loop call
    loop = diffusion._fused_loop
    diffusion._fused_loop = lambda *a: (fused.append(a[-1]), loop(*a))[1]
    try:
        diffusion.seq_offset = c.seq_offset
        # 2. per-step path, fed the same draws
        stream = PhiloxStream(c.seq_offset)
        diffusion.noise_source = lambda shape, kind: stream.truncated(shape, c.top_p) if kind == "truncated" else stream.randn(shape)
        diffusion.rounding_trace = []
        diffusion._noise_calls = 0
        tok_ref, sample_ref = _package_chain(c, model, diffusion, model_emb, tcond)
        calls_ref = diffusion._noise_calls
        assert calls_ref == stream.calls == 1 + steps
        assert fused == []
        ids, _ = R.trace_to_numpy(diffusion.rounding_trace, *cond["input_mask"].shape)
        free = cond["input_mask"] != 0
        scale = c.D / 128 if c.pxs else np.maximum(c.D / 128, np.asarray(s.sqrt_recipm1_alphas_cumprod)[[r["t"] for r in record]])
        rep = R.chain_report(ref_ids, ref_margin, ids, free, MARGIN_TOL * np.asarray(scale), DOWNSTREAM_TOL * np.asarray(scale))
        tk = R.token_report(want, tok_ref.cpu().numpy(), free, rep["never_divergent"], None, LOGIT_TOL)
        print("%s: %d rounding calls, id agreement %.5f, %d positions ever divergent, token agreement %.5f, violations %d + %d"
              % (name, rep["calls"], rep["id_agreement_all_calls"], rep["positions_ever_divergent"], tk["token_agreement"],
                 rep["violations"], tk["token_violations"]))
        assert rep["calls"] == steps
        assert rep["violations"] == 0, rep
        assert tk["token_violations"] == 0, tk
        sample_ref = sample_ref.clone()
        # 3. the production loop, graph-replayed and eager
        diffusion.noise_source = None
        diffusion.rounding_trace = None
        for use_graph in (True, False):
            diffusion.use_cuda_graph = use_graph
            diffusion._noise_calls = 0
            fused.clear()
            tok, sample = _package_chain(c, model, diffusion, model_emb, tcond)
            tag = (name, "graph" if use_graph else "eager")
            assert fused == [use_graph], tag                   # the fused loop ran, capturing a graph exactly when asked
            assert diffusion._noise_calls == calls_ref, tag
            assert torch.equal(sample, sample_ref), (tag, int((sample != sample_ref).sum()))
            assert torch.equal(tok, tok_ref), tag
    finally:
        del diffusion._fused_loop
        diffusion.noise_source = None
        diffusion.rounding_trace = None
        diffusion._noise_calls = 0
        diffusion.seq_offset = 0
        diffusion.use_cuda_graph = True
