"""The Philox noise against a host Philox and float64 quantiles, and the schedule tables past the __constant__ limit.

Every other noise test takes md_fill_normal as ground truth.  This file checks md_fill_normal itself:

  1. a numpy Philox4x32-R, pinned by known answers (R = 10: CUDA's curand_Philox4x32_10; R = 7), gives the 23 random bits
     of every element (`host_bits`): element 4g + j is word j of Philox4x32-7 at counter (g_lo, g_hi, step_lo, step_hi)
     and key (seed_lo, seed_hi), and the kernel keeps word >> 9;
  2. the kernel's output is a function N(b) of those bits alone.  Its table over all 2^23 patterns, scattered from 2^27
     draws by the host bits, must be single valued (which pins the whole stream), exactly odd, accurate against the float64
     quantile, monotone, and inside the truncation law, for the central polynomial (0 < top_p <= 1) and the general quantile;
  3. md_fill_normal at edge seeds, counters and offsets, and the in-kernel draws of md_posterior_step (both kernels) and
     md_q_sample at element indices past 2^34, equal table[host bits];
  4. with T > MD_MAX_CONST_T = 2048 the step kernels read the schedule from device memory (elementwise.cu `SchedRef`):
     md_posterior_step, md_xstart_from_eps and md_q_sample bit for bit against float32 replays at T = 2048, 2049 and 4000
     and across switches between the two routes on one device, and two short chains at diffusion_steps = 4000 through
     the fused loop.

Run with -s to see the MEASURED lines."""
import math

import numpy as np
import pytest
import torch
from scipy.special import erfinv

pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

from musediffusion_b200 import ops  # noqa: E402
from test_reverse_step_gpu import (MODES, SEED, _check_chain, _dev, _emulate, _kernel_ddpm_sd, _run_step,  # noqa: E402
                                   _schedule, _step_inputs)
from test_rounding_kernels_gpu import fma32  # noqa: E402

DEV = torch.device("cuda:0")
F32 = np.float32
U64 = 2 ** 64 - 1
NPAT = 1 << 23                          # random bits per normal


def _report(name, **kv):
    print("MEASURED %s %s" % (name, " ".join("%s=%s" % (k, ("%.4g" % v) if isinstance(v, float) else v) for k, v in kv.items())))


# ------------------------------------------------------------------------------------------------ 1. host Philox
M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85       # key schedule (Weyl constants)
LO32, SH32 = np.uint64(0xFFFFFFFF), np.uint64(32)


def philox4x32(ctr, key, rounds):
    """Philox4x32-R (Salmon et al., SC'11) in numpy uint64 on arrays of counter words (x, y, z, w) and a key (k0, k1):
    round r uses key + r (W0, W1), as NoiseGen::init precomputes it.  Returns the four output words."""
    x, y, z, w = (np.asarray(c, dtype=np.uint64) for c in ctr)
    for r in range(rounds):
        kx, ky = np.uint64((key[0] + r * W0) & 0xFFFFFFFF), np.uint64((key[1] + r * W1) & 0xFFFFFFFF)
        p0, p1 = M0 * x, M1 * z
        x, y, z, w = (p1 >> SH32) ^ y ^ kx, p1 & LO32, (p0 >> SH32) ^ w ^ ky, p0 & LO32
    return x, y, z, w


def host_bits(seed, step, g0, ngroups):
    """the 23 random bits of elements 4 g0 ... 4 (g0 + ngroups) - 1 of the stream (seed, step counter), int64"""
    g = np.arange(ngroups, dtype=np.uint64) + np.uint64(g0)
    words = philox4x32((g & LO32, g >> SH32, step & 0xFFFFFFFF, step >> 32), (seed & 0xFFFFFFFF, seed >> 32), 7)
    return (np.stack(words, axis=1) >> np.uint64(9)).astype(np.int64).reshape(-1)


KAT_IN = [((0, 0, 0, 0), (0, 0)),
          ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF)),
          ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0))]
KAT_OUT = {10: [(0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8),     # curand_Philox4x32_10 (curand_philox4x32_x.h)
                (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD),
                (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)],
           7: [(0x5F6FB709, 0x0D893F64, 0x4F121F81, 0x4F730A48),
               (0x5207DDC2, 0x45165E59, 0x4D8EE751, 0x8C52F662),
               (0x4DFCCABA, 0x190A87F0, 0xC47362BA, 0xB6B5242A)]}


@pytest.mark.parametrize("rounds", [7, 10])
def test_host_philox_known_answers(rounds):
    for (ctr, key), want in zip(KAT_IN, KAT_OUT[rounds]):
        assert tuple(int(v) for v in philox4x32(ctr, key, rounds)) == want, (rounds, ctr, key)


# ------------------------------------------------------------------------------------------------ the quantile's input
def noise_law(top_p):
    """NoiseGen::init for this top_p (a float on the C side): (q_scale, q_bias, span, central).  span is the exact
    probability of the band, erf(top_p / sqrt 2), for the truncation law; the kernel's float32 q_scale rounds it."""
    tp = float(F32(top_p))
    lo, span = 0.0, 1.0
    if tp > 0.0:
        lo = 0.5 * math.erfc(tp / math.sqrt(2.0))
        span = 1.0 - 2.0 * lo
    q_scale, q_bias = F32(span), F32((lo - 0.5 + 0.5 * span) + span * 2.0 ** -24)
    return q_scale, q_bias, math.erf(tp / math.sqrt(2.0)) if tp > 0.0 else 1.0, 0.0 < tp <= 1.0


def quantile64(q):
    """Phi^-1(0.5 + q) in float64 as sqrt(2) erfinv(2 q): 2 q is exact, where 0.5 + q would round away the low bits of a
    small q"""
    return math.sqrt(2.0) * erfinv(2.0 * np.asarray(q, dtype=np.float64))


def q_of_patterns(top_p):
    """q_b for every pattern b: the kernel's fmaf((1 + b 2^-23) - 1.5, q_scale, q_bias).  With q_bias = q_scale 2^-24 that is
    q_scale (b 2^-23 - 0.5 + 2^-24), exact in float64 (a 25-bit odd multiple of 2^-24 times a 24-bit q_scale), so one
    rounding to float32 gives the kernel's value bit for bit, and q is exactly odd: q(2^23 - 1 - b) = -q(b)."""
    q_scale, q_bias, *_ = noise_law(top_p)
    assert q_bias == F32(np.float64(q_scale) * 2.0 ** -24), (top_p, q_scale, q_bias)
    b = np.arange(NPAT, dtype=np.float64)
    return ((b * 2.0 ** -23 - 0.5 + 2.0 ** -24) * np.float64(q_scale)).astype(F32)


CENTRAL = [643.067138671875, -38.967872619628906, 21.74688720703125, 5.587021827697754, 2.6269679069519043, 2.506624698638916]


def central_emulation(q):
    """elementwise.cu norm_quantile_central(_x2) in float32 on the GPU: r = q q, five correctly rounded FMAs, p q"""
    q = torch.from_numpy(q).to(DEV)
    r = q * q
    p = torch.full_like(q, CENTRAL[0])
    for c in CENTRAL[1:]:
        p = fma32(p, r, torch.full_like(q, c))
    return (p * q).cpu().numpy()


def central_bound(q):
    """(P(q) in float64 with the kernel's coefficients, first-order bound on the kernel's rounding error): r = fl(q q) and
    every Horner step and the last product each add one float32 rounding, propagated through the remaining steps"""
    q = q.astype(np.float64)
    u = 2.0 ** -24
    r = q * q
    p, e = np.full_like(q, CENTRAL[0]), np.zeros_like(q)
    for c in CENTRAL[1:]:
        pn = p * r + c
        e = e * r + np.abs(p) * r * u + np.abs(pn) * u
        p = pn
    n = p * q
    return n, (np.abs(q) * e + np.abs(n) * u) * (1 + 2.0 ** -20)


# ------------------------------------------------------------------------------------------------ 2. exhaustive tables
TABLE_SEED, TABLE_CTR = 0x243F6A8885A308D3, 5
N_DRAWS = 1 << 27                       # 16 draws per pattern
CHUNK = 1 << 22                         # groups of 4 per host chunk
TOP_PS = [0.0, 1e-3, 0.5, 1.0, 1.5, 2.0, 3.0, 6.0]


@pytest.fixture(scope="module")
def tables():
    """top_p -> (amin, amax) over the draws of each of the 2^23 patterns, float32 numpy.  The 2^27 draws at TABLE_SEED /
    TABLE_CTR leave about one pattern uncovered; each such pattern is drawn again as the group of 4 past the 2^27 draws
    where the host stream first carries it."""
    idx = torch.empty(N_DRAWS, dtype=torch.int64, device=DEV)
    for g0 in range(0, N_DRAWS // 4, CHUNK):
        idx[4 * g0:4 * (g0 + CHUNK)] = torch.from_numpy(host_bits(TABLE_SEED, TABLE_CTR, g0, CHUNK)).to(DEV)
    seen = torch.zeros(NPAT, dtype=torch.bool, device=DEV)
    seen[idx] = True
    todo = set(torch.nonzero(~seen).flatten().tolist())
    extra_groups, g0 = [], N_DRAWS // 4
    while todo:
        bits = host_bits(TABLE_SEED, TABLE_CTR, g0, CHUNK)
        for k in np.nonzero(np.isin(bits, list(todo)))[0]:
            if int(bits[k]) in todo:
                todo.discard(int(bits[k]))
                extra_groups.append(g0 + int(k) // 4)
        g0 += CHUNK
    extra_idx = torch.from_numpy(np.concatenate([host_bits(TABLE_SEED, TABLE_CTR, g, 1) for g in extra_groups] or
                                                [np.zeros(0, np.int64)])).to(DEV)
    _report("table coverage", draws=N_DRAWS, patterns_missed=len(extra_groups))
    out = {}
    for top_p in TOP_PS:
        vals = [ops.fill_normal((N_DRAWS,), DEV, seed=TABLE_SEED, step_counter=TABLE_CTR, top_p=top_p)]
        vals += [ops.fill_normal((4,), DEV, seed=TABLE_SEED, step_counter=TABLE_CTR, elem_offset=4 * g, top_p=top_p)
                 for g in extra_groups]
        v, ix = torch.cat(vals), torch.cat([idx, extra_idx])
        lo = torch.full((NPAT,), float("nan"), device=DEV).scatter_reduce_(0, ix, v, "amin", include_self=False)
        hi = torch.full((NPAT,), float("nan"), device=DEV).scatter_reduce_(0, ix, v, "amax", include_self=False)
        out[top_p] = (lo.cpu().numpy(), hi.cpu().numpy())
        del vals, v, ix
    assert len(torch.unique(torch.cat([idx, extra_idx]))) == NPAT
    return out


def _table(tables, top_p):
    return torch.from_numpy(tables[top_p][0]).to(DEV)


@pytest.mark.parametrize("top_p", TOP_PS)
def test_quantile_table(top_p, tables):
    """N_top_p(b) over all 2^23 patterns b of the 23 random bits, against q_b and the float64 quantile:
    - a function of the bits: every draw of a pattern has the same float32 bits (min == max);
    - exactly odd: N(2^23 - 1 - b) == -N(b);
    - central polynomial (0 < top_p <= 1): bit-identical to a float32 emulation of its Horner scheme, and within the
      float64 error of the polynomial plus its derived rounding bound of Phi^-1(0.5 + q_b) (DESIGN: 1.2e-6 at most);
      general quantile: within 2^-21 |Phi^-1(0.5 + q_b)|;
    - non-decreasing in b;
    - the truncation law: |N| <= top_p, and |N - Phi^-1(0.5 + q_exact)|, q_exact = span (u_b - 0.5) with u_b = b 2^-23 +
      2^-24 (the band [Phi(-top_p), Phi(top_p)] sampled at u_b), within the accuracy bound plus |q_b - q_exact| / phi(n),
      the float32 error of q_b carried through the quantile."""
    amin, amax = tables[top_p]
    n = amin
    _, _, span, central = noise_law(top_p)
    q = q_of_patterns(top_p)
    assert np.array_equal(q[::-1], -q)
    diff = int((amin.view(np.int32) != amax.view(np.int32)).sum())
    odd = int((n[::-1].view(np.int32) != (-n).view(np.int32)).sum())
    ref = quantile64(q)
    n64 = n.astype(np.float64)
    err = np.abs(n64 - ref)
    if central:
        poly, rnd = central_bound(q)
        bound = np.abs(poly - ref) + rnd
        emul = int((central_emulation(q).view(np.int32) != n.view(np.int32)).sum())
    else:
        bound = 2.0 ** -21 * np.abs(ref)
        emul = 0
    over = err > bound
    step = np.diff(n64)
    dips = np.nonzero(step < 0)[0]
    q_exact = span * (np.arange(NPAT, dtype=np.float64) * 2.0 ** -23 + 2.0 ** -24 - 0.5)
    ideal = quantile64(q_exact)
    phi = np.exp(-0.5 * np.maximum(np.abs(ref), np.abs(ideal)) ** 2) / math.sqrt(2.0 * math.pi)
    law_err = np.abs(n64 - ideal)
    law_over = law_err > bound + np.abs(q.astype(np.float64) - q_exact) / phi
    trunc = int((np.abs(n) > F32(top_p)).sum()) if top_p > 0 else 0
    nz = np.abs(ref) > 0
    _report("quantile table", top_p=top_p, branch="central" if central else "general", max_abs_err=float(err.max()),
            at_q=float(q[np.argmax(err)]), max_rel_err=float((err[nz] / np.abs(ref[nz])).max()),
            worst_over_bound=float((err / bound).max()), over_bound=int(over.sum()), dips=len(dips),
            max_dip=float(-step[dips].min()) if len(dips) else 0.0, max_abs_n=float(np.abs(n).max()),
            law_max_err=float(law_err.max()), law_over=int(law_over.sum()), beyond_top_p=trunc, not_single_valued=diff,
            not_odd=odd, emulation_mismatches=emul)
    assert diff == 0, "%d patterns drew different values: the stream is not the host Philox" % diff
    assert odd == 0
    assert emul == 0
    assert not over.any(), (int(over.sum()), float(q[np.argmax(err / bound)]), float((err / bound).max()))
    assert len(dips) == 0, (len(dips), q[dips[:8]])
    assert trunc == 0
    assert not law_over.any(), int(law_over.sum())


# ------------------------------------------------------------------------------------------------ 3. the stream at its edges
def _expected(tables, top_p, seed, step, elem0, n):
    """table[host bits] for elements elem0 ... elem0 + n - 1 (elem0 a multiple of 4) of the stream (seed, step)"""
    bits = host_bits(seed, step, elem0 // 4, (n + 3) // 4)[:n]
    return _table(tables, top_p)[torch.from_numpy(bits).to(DEV)]


@pytest.mark.parametrize("seed", [0, SEED, U64])
def test_fill_normal_equals_host_stream(seed, tables):
    """md_fill_normal == table[host bits] at counters 0, 2^32 (step_hi only) and 2^64 - 1, element offsets 0 and 2^34 + 4
    (counter word g_hi non-zero), an odd element count (the last group of 4 is cut), every top_p of the tables; seed
    2^64 - 1 goes through the signed conversion of the op layer."""
    n = 1001
    for step in (0, 1 << 32, U64):
        for off in (0, (1 << 34) + 4):
            for top_p in TOP_PS:
                got = ops.fill_normal((n,), DEV, seed=seed, step_counter=step, elem_offset=off, top_p=top_p)
                want = _expected(tables, top_p, seed, step, off, n)
                assert torch.equal(got.view(torch.int32), want.view(torch.int32)), (seed, step, off, top_p)


@pytest.mark.parametrize("D", [100, 128])
@pytest.mark.parametrize("mode,eta", [("ddpm", 0.0), ("ddim", 0.5)])
def test_in_kernel_draws_equal_host_stream(mode, eta, D, tables):
    """md_posterior_step with noise = None (D = 128 with a token mask: posterior_step_d128_kernel; with an element mask and
    at D = 100: the generic kernel) and md_q_sample with noise = None (t per sequence, and t = None), at sequence offsets
    whose global element index (seq_offset + b) L D + e passes 2^34, equal the same calls fed table[host bits] as
    explicit noise, bit for bit."""
    _schedule()
    B, L = 3, 37
    rng = np.random.default_rng(D + int(10 * eta))
    x = _dev(rng.standard_normal((B, L, D)).astype(F32))
    pred = _dev((1.5 * rng.standard_normal((B, L, D))).astype(F32))
    x_start = _dev(rng.standard_normal((B, L, D)).astype(F32))
    mask_tok = _dev((rng.random((B, L)) > 0.25).astype(np.int32))
    tok = torch.broadcast_to(mask_tok.unsqueeze(-1), (B, L, D))
    t = _dev(np.array([1999, 1, 700]))
    for seed, step in ((SEED, 7), (U64, U64), (0, 1 << 32)):
        for off in ((1 << 34) // (L * D) + 1, (1 << 40) // (L * D) + 3):
            assert off * L * D >= 1 << 34
            for top_p in (0.0, 0.5, 1.0, 2.0):
                noise = _expected(tables, top_p, seed, step, off * L * D, B * L * D).reshape(B, L, D)
                for name, mask in (("token mask", tok), ("element mask", tok.contiguous())):
                    kw = dict(pred=pred, seed=seed, step_counter=step, seq_offset=off, mask=mask, x_start=x_start, eta=eta,
                              clip=True, top_p=top_p)
                    got = ops.posterior_step(x, t, MODES[mode], noise=None, **kw)
                    want = ops.posterior_step(x, t, MODES[mode], noise=noise, **kw)
                    assert torch.equal(got, want), (mode, D, seed, step, off, top_p, name)
            noise = _expected(tables, 0.0, seed, step, off * L * D, B * L * D).reshape(B, L, D)
            for tt in (t, None):
                got = ops.q_sample(x, tt, noise=None, seed=seed, step_counter=step, seq_offset=off, mask=mask_tok)
                want = ops.q_sample(x, tt, noise=noise, seed=seed, step_counter=step, seq_offset=off, mask=mask_tok)
                assert torch.equal(got, want), ("q_sample", D, seed, step, off, tt is None)


# ------------------------------------------------------------------------------------------------ 4. schedules past 2048
def _tab(s, name):
    return np.asarray(getattr(s, name), dtype=np.float64).astype(F32)


def _t_cases(T, B):
    """per sequence: 0, 1, 2047, 2048 and T - 1 where T allows them (B of them, the last repeated); shared: T - 1"""
    per = sorted({0, 1, min(2047, T - 1), T - 1} | ({2048} if T > 2048 else set()))
    return [np.array((per + per[-1:] * B)[:B]), np.array([T - 1])]


def _check_steps(s, T, seed, clips=(0, 1, 2)):
    """md_posterior_step on both kernels (D = 128 token mask / element mask / padded bf16 copy, and D = 100), DDPM and DDIM
    at eta 0 and 0.5, every clip, against _emulate bit for bit"""
    B = 5
    for D in (128, 100):
        a = _step_inputs(D, seed=seed + D, B=B, L=23)
        L = a.mask_tok.shape[1]
        se = ops.SplitEmbedding(_dev(a.E))
        gathered = a.E[a.idx].reshape(B, L, D)
        tok = torch.broadcast_to(_dev(a.mask_tok).unsqueeze(-1), (B, L, D))
        keep = np.broadcast_to(a.mask_tok[..., None] == 0, (B, L, D))
        routes = [("token mask", tok, D), ("element mask", tok.contiguous(), D), ("padded bf16", tok, ops.padded_width(D + 1))]
        for t in _t_cases(T, B):
            t_rows = np.broadcast_to(t, (B,))
            for mode, eta in (("ddpm", 0.0), ("ddim", 0.0), ("ddim", 0.5)):
                for clip in clips:
                    kw = dict(pred=_dev(a.pred)) if clip == 0 else dict(idx=_dev(a.idx), E=se.E_clamped if clip == 2 else _dev(a.E))
                    p_in = a.pred if clip == 0 else gathered
                    ref = _emulate(s, mode, a.x, p_in, a.n, t_rows, eta, min(clip, 1), keep, a.x_start)
                    for name, mask, ld in routes:
                        got = _run_step(_dev(a.x), _dev(t), MODES[mode], mask, _dev(a.x_start), ld, noise=_dev(a.n), eta=eta,
                                        clip=clip, **kw)
                        for what, g, r in zip(("pred", "mean", "sample"), got, ref):
                            g = g.cpu().numpy()
                            assert np.array_equal(g, r), (T, D, t.tolist(), mode, eta, clip, name, what, int((g != r).sum()))


def _check_xstart_and_q_sample(s, T, seed):
    """md_xstart_from_eps = fl(fl(sr x) - fl(srm1 eps)) and md_q_sample = fl(fl(sqrt_ab x) + fl(sqrt_1mab n)) (x where the
    mask is 0) in float32, bit for bit, t per sequence and shared"""
    B, L, D = 5, 19, 100
    rng = np.random.default_rng(seed)
    x, e, n = (rng.standard_normal((B, L, D)).astype(F32) for _ in range(3))
    mask_tok = (rng.random((B, L)) > 0.3).astype(np.int32)
    keep = np.broadcast_to(mask_tok[..., None] == 0, (B, L, D))
    for t in _t_cases(T, B):
        ti = np.broadcast_to(t, (B,))[:, None, None]
        got = ops.xstart_from_eps(_dev(x), _dev(e), _dev(t)).cpu().numpy()
        want = _tab(s, "sqrt_recip_alphas_cumprod")[ti] * x - _tab(s, "sqrt_recipm1_alphas_cumprod")[ti] * e
        assert np.array_equal(got, want), ("xstart_from_eps", T, t.tolist(), int((got != want).sum()))
        got = ops.q_sample(_dev(x), _dev(t), noise=_dev(n), mask=_dev(mask_tok)).cpu().numpy()
        want = np.where(keep, x, _tab(s, "sqrt_alphas_cumprod")[ti] * x + _tab(s, "sqrt_one_minus_alphas_cumprod")[ti] * n)
        assert np.array_equal(got, want), ("q_sample", T, t.tolist(), int((got != want).sum()))


@pytest.mark.parametrize("T", [2048, 2049, 4000])
def test_schedule_past_constant_limit(T):
    """T = 2048 is the last table held in __constant__ memory, 2049 and 4000 are read from device memory: the DDPM noise
    scale within 2 ulp of float64 at every index, and every output of md_posterior_step, md_xstart_from_eps and md_q_sample
    bit-identical to its float32 replay."""
    s = _schedule(T)
    sd = _kernel_ddpm_sd(T)
    exact = np.exp(0.5 * _tab(s, "model_log_variance").astype(np.float64))
    ulps = np.abs(sd[1:].astype(np.float64) - exact[1:]) / np.spacing(exact[1:].astype(F32)).astype(np.float64)
    _report("DDPM noise scale", T=T, max_ulp=float(ulps.max()))
    assert sd[0] == 0.0 and ulps.max() <= 2.0, ulps.max()
    _check_steps(s, T, seed=T)
    _check_xstart_and_q_sample(s, T, seed=T)


def test_schedule_route_switches():
    """T = 2000 -> 4000 -> 3000 -> 4000 -> 2000 on one device: 3000 reuses the 4000-entry allocation with its own row
    stride, and each switch changes between __constant__ and device memory.  Every call matches its own replay."""
    for k, T in enumerate((2000, 4000, 3000, 4000, 2000)):
        s = _schedule(T)
        _check_steps(s, T, seed=100 + k, clips=(1,))
        _check_xstart_and_q_sample(s, T, seed=100 + k)


CHAINS_4000 = {
    # as test_reverse_step_gpu.CHAINS: DDIM gap 100 from t = 3999 (6 steps), and DDPM from t = 5 (6 steps)
    "t4000-mod-ddim-eta": dict(mode="modification", D=128, L=64, B=2, T=4000, step=40, strength=6.2 / 40, eta=0.3),
    "t4000-mod-ddpm-central": dict(mode="modification", D=128, L=64, B=3, T=4000, step=4000, strength=6.2 / 4000, top_p=1),
}


@pytest.mark.parametrize("name", list(CHAINS_4000))
def test_fused_loop_at_4000_steps(name):
    """diffusion_steps = 4000: the per-step path fed PhiloxStream agrees with the oracle under the parity rule, and the fused
    loop, graph-replayed and eager, reproduces it bit for bit (test_reverse_step_gpu._check_chain)."""
    _check_chain(name, CHAINS_4000[name])
