"""The reductions that turn model outputs into token ids, checked against exact and float64 references through the C-ABI
ops (`torch.ops.musediff.*`, the path production uses):

  md_round_argmin_tc (mode 0: argmin_v |E_v|^2 - 2 x.E_v, the sampler's rounding; mode 1: argmax_v x.E_v + b_v,
  decode_tokens), md_round_argmin / md_logits_argmax (fp32 CUDA cores, the reference API), md_dist_scores (get_logits
  with logits_mode 2), and the operand preparation md_split_bf16 / md_embed_split(_padded) / the GEMM split epilogue.

  A  operand preparation, bit-exact against round-to-nearest-even (computed on the fp32 bit pattern) and against a
     float32 emulation of |E_v|^2's operation order.
  B  the tensor-core reduction on integer data, where every partial product and partial sum is exact in fp32 in any
     order: ids (lowest id on ties), margins and planted ties must equal the exact result, for both input routes.
  C  the tensor-core reduction on random data against a per-key error bound beta derived from the kernel's arithmetic
     (see `tc_key_bound`), with the per-key error measured directly.
  D  the fp32 kernels, bit-exact against a float32 emulation of `round_kernel<MODE>`'s operation order.
  E  md_dist_scores bit-exact from its own inputs; get_logits exact on integer data; decode_tokens vs get_logits.
  F  non-finite rows: every id any of the four reductions writes lies in [0, V).

Outputs are written into views inside guard regions, which must stay untouched.  Run with -s to see the MEASURED lines.
Exact FMA in float32 is emulated through float64 (`fma32`); float32 adds are torch float32 ops on the GPU (IEEE RN)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

from musediffusion_b200 import _lib, ops  # noqa: E402
from musediffusion_b200.initialization import create_model_and_diffusion  # noqa: E402

DEV = torch.device("cuda:0")
BF16, F32 = torch.bfloat16, torch.float32
K = torch.ops.musediff
U32 = 2.0 ** -24                  # fp32 unit roundoff
INF = float("inf")
IDX_FILL = -7


# ------------------------------------------------------------------------------------------------ shared helpers
def _report(name, **kv):
    print("MEASURED %s %s" % (name, " ".join("%s=%s" % (k, ("%.4g" % v) if isinstance(v, float) else v) for k, v in kv.items())))


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _guarded(n, dtype, fill):
    front, back = 64, 4096
    buf = torch.full((front + n + back,), fill, dtype=dtype, device=DEV)
    return buf, buf[front:front + n]


def _check_guard(buf, n, fill, what):
    ib = torch.int32 if buf.element_size() == 4 else torch.int16
    want = torch.full((1,), fill, dtype=buf.dtype).view(ib).item()
    g = torch.cat([buf[:64], buf[64 + n:]]).view(ib)
    assert bool((g == want).all()), "%s: %d guard elements outside the out= view were written" % (what, int((g != want).sum()))


def fma32(a, b, c):
    """Correctly rounded float32 fmaf(a, b, c) (broadcasting).  a*b is exact in float64; TwoSum gives the error of the
    float64 sum, which is then rounded to odd, so the final cast to float32 rounds once."""
    p = a.double() * b.double()
    c = c.double()
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    fix = (err != 0) & ((s.view(torch.int64) & 1) == 0)
    toward = torch.where(err > 0, torch.full_like(s, INF), torch.full_like(s, -INF))
    return torch.where(fix, torch.nextafter(s, toward), s).float()


def _butterfly(vals):
    """the xor-16 ... 1 shuffle tree on [..., 32] lanes (every lane ends with the same sum); returns lane 0's value"""
    lane = torch.arange(32, device=vals.device)
    for o in (16, 8, 4, 2, 1):
        vals = vals + vals[..., lane ^ o]
    return vals[..., 0]


def _first_min(key):
    """(lowest index of the row minimum, second-smallest minus smallest of the multiset; +inf for one column)"""
    V = key.shape[1]
    best = key.min(1).values
    ar = torch.arange(V, device=key.device).expand_as(key)
    idx = torch.where(key == best[:, None], ar, V).min(1).values
    if V == 1:
        return idx, torch.full_like(best, INF)
    two = key.topk(2, dim=1, largest=False).values
    return idx, two[:, 1] - two[:, 0]


def run_tc(se, mode, cst, x=None, presplit=None):
    """md_round_argmin_tc(_padded) with idx / margin written into guarded views; every row must be written."""
    M = x.shape[0] if presplit is None else presplit.shape[0]
    ibuf, idx = _guarded(M, torch.int32, IDX_FILL)
    mbuf, mg = _guarded(M, F32, float("nan"))
    ws = presplit if presplit is not None else torch.empty((M, 2 * se.Dp), dtype=BF16, device=DEV)
    if se.Dp == se.D:
        K.round_argmin_tc(x, se.E2, cst, ws, idx, mg, se.V, mode)
    else:
        K.round_argmin_tc_padded(x, se.E2, cst, ws, idx, mg, se.V, se.D, mode)
    torch.cuda.synchronize()
    what = "round_tc mode %d M=%d V=%d D=%d" % (mode, M, se.V, se.D)
    _check_guard(ibuf, M, IDX_FILL, what + " idx")
    _check_guard(mbuf, M, float("nan"), what + " margin")
    assert not bool((idx == IDX_FILL).any()), what + ": rows left unwritten"
    return idx.clone(), mg.clone()


def run_fp32(x, E, bias, mode):
    """md_round_argmin (mode 0) / md_logits_argmax (mode 1) into guarded views."""
    M = x.shape[0]
    ibuf, idx = _guarded(M, torch.int32, IDX_FILL)
    mbuf, mg = _guarded(M, F32, float("nan"))
    if mode == 0:
        K.round_argmin(x, E, idx, mg)
    else:
        K.logits_argmax(x, E, bias, idx, mg)
    torch.cuda.synchronize()
    what = "fp32 round mode %d M=%d V=%d D=%d" % (mode, M, E.shape[0], E.shape[1])
    _check_guard(ibuf, M, IDX_FILL, what + " idx")
    _check_guard(mbuf, M, float("nan"), what + " margin")
    assert not bool((idx == IDX_FILL).any()), what + ": rows left unwritten"
    return idx.clone(), mg.clone()


def presplit_via_gemm(x, Dp):
    """[hi | 0 | lo | 0] of x written by the split epilogue of md_linear_bf16, as the sampler's last Linear writes it:
    y = [xh | xl] @ [I | I]^T = x exactly (x must be hi + lo in bf16), N = Dp."""
    M, D = x.shape
    xp = torch.zeros((M, Dp), dtype=F32, device=DEV)
    xp[:, :D] = x
    xh = xp.to(BF16)
    xl = (xp - xh.float()).to(BF16)
    assert torch.equal(xh.float() + xl.float(), xp), "test construction: x is not hi + lo"
    A = torch.cat([xh, xl], 1).contiguous()
    eye = torch.eye(Dp, dtype=BF16, device=DEV)
    W = torch.cat([eye, eye], 1).contiguous()
    buf, out = _guarded(M * 2 * Dp, BF16, float("nan"))
    ops.linear(A, W, torch.zeros(Dp, device=DEV), _lib.EPI_BIAS_SPLIT, out=out.view(M, 2 * Dp))
    torch.cuda.synchronize()
    _check_guard(buf, M * 2 * Dp, float("nan"), "split epilogue M=%d N=%d" % (M, Dp))
    return out.view(M, 2 * Dp)


def _bits16(t):
    return t.detach().cpu().contiguous().view(torch.int16)


# ------------------------------------------------------------------------------------------------ A. operand preparation
def _split_inputs(rows, D, seed):
    """fp32 rows covering ordinary values, the top of the bf16 range, lo below bf16's normal range, fp32 subnormals,
    exact bf16 values (lo = +0) and signed zeros."""
    g = torch.Generator().manual_seed(seed)
    r = rows // 6
    parts = [
        torch.randn(r, D, generator=g) * torch.exp2(torch.randint(-20, 21, (r, 1), generator=g).float()),
        (torch.rand(r, D, generator=g) * (3.39e38 - 2.0 ** 127) + 2.0 ** 127) * torch.sign(torch.randn(r, D, generator=g)),
        torch.exp2(torch.rand(r, D, generator=g) * 14 - 126) * torch.sign(torch.randn(r, D, generator=g)),
        torch.randn(r, D, generator=g) * 2.0 ** -130,
        (torch.randn(r, D, generator=g) * 100).to(BF16).float(),
    ]
    z = torch.zeros(rows - 5 * r, D)
    z[::2] = -0.0
    x = torch.cat(parts + [z]).float()
    assert bool(torch.isfinite(x).all())
    return x


def _rne_bf16(x_cpu):
    """RNE of finite fp32 values to bf16 on the bit pattern (subnormals included: no flush to zero on any CPU path)"""
    u = x_cpu.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    r = (u + 0x7FFF + ((u >> 16) & 1)) >> 16
    return torch.where(r >= 0x8000, r - 0x10000, r).to(torch.int16).view(BF16)


def _rne_split(x_cpu):
    """hi = RNE(x), lo = RNE(x - hi); x - hi is exact in fp32 (the CPU does not flush subnormals by default)"""
    hi = _rne_bf16(x_cpu)
    lo = _rne_bf16(x_cpu - hi.float())
    return hi, lo


@pytest.mark.parametrize("copies", [1, 2])
@pytest.mark.parametrize("D", [4, 64, 100, 128, 500, 768])
def test_split_bf16_is_rne(D, copies):
    """md_split_bf16: hi = RNE(x), lo = RNE(x - hi) (x - hi is exact in fp32), copies x [hi | lo], bit for bit: lo below
    bf16's normal range is kept (no flush to zero), exact bf16 values give lo = +0."""
    rows = 60
    x = _split_inputs(rows, D, seed=D * 3 + copies)
    buf, out = _guarded(rows * copies * 2 * D, BF16, float("nan"))
    K.split_bf16(x.to(DEV), out.view(rows, copies * 2 * D), copies)
    torch.cuda.synchronize()
    _check_guard(buf, rows * copies * 2 * D, float("nan"), "split_bf16")
    hi, lo = _rne_split(x)
    sub = ((lo.float().abs() < 2.0 ** -126) & (lo.float() != 0)).sum()
    assert int(sub) > 0 and bool((lo.float() == 0).any()), "test construction: no subnormal / zero lo"
    got = out.view(rows, copies, 2, D)
    for k in range(copies):
        assert torch.equal(_bits16(got[:, k, 0]), _bits16(hi)), "hi copy %d" % k
        assert torch.equal(_bits16(got[:, k, 1]), _bits16(lo)), "lo copy %d" % k
    _report("split_bf16", D=D, copies=copies, subnormal_lo=int(sub), bit_exact=rows * D * 2 * copies)


def sqnorm_emulated(E):
    """embed_prepare_kernel's |E_v|^2: thread t (of 128) chains fmaf over d = t, t + 128, ...; the xor-16 ... 1 warp
    tree; then red[0] + red[1] + red[2] + red[3] left to right."""
    V, D = E.shape
    n = -(-D // 128) * 128
    Ep = torch.zeros((V, n), dtype=F32, device=E.device)
    Ep[:, :D] = E
    lanes = torch.zeros((V, 128), dtype=F32, device=E.device)
    for k in range(n // 128):
        col = Ep[:, k * 128:(k + 1) * 128]
        lanes = fma32(col, col, lanes)
    red = [_butterfly(lanes[:, 32 * w:32 * w + 32]) for w in range(4)]
    return ((red[0] + red[1]) + red[2]) + red[3]


@pytest.mark.parametrize("V,D,Dp", [(1, 64, 64), (63, 100, 128), (256, 128, 128), (257, 500, 512), (729, 128, 128),
                                    (729, 16, 64), (200, 768, 768), (63, 64, 128), (1000, 132, 192)])
def test_embed_split_exact(V, D, Dp):
    """md_embed_split(_padded): E2 = [Eh | 0 | El | 0] with zero rows for V <= v < Vp, |E_v|^2 bit-identical to the
    kernel's float32 operation order, +inf on the padding rows, E_clamped = clamp(E, -1, 1) exactly."""
    g = _gen(V + D + Dp)
    E = torch.randn(V, D, generator=g, device=DEV) * 1.7
    E[:, ::7] *= 300.0                                      # large entries: |E_v|^2 rounds in every order
    Vp = _lib.lib.md_round_tc_padded_vocab(V)
    E2 = torch.full((Vp, 2 * Dp), float("nan"), dtype=BF16, device=DEV)
    sbuf, sq = _guarded(Vp, F32, float("nan"))
    Ec = torch.full_like(E, float("nan"))
    if Dp == D:
        K.embed_split(E, E2, sq, Ec)
    else:
        K.embed_split_padded(E, E2, sq, Ec)
    torch.cuda.synchronize()
    _check_guard(sbuf, Vp, float("nan"), "sqnorm")
    hi, lo = _rne_split(E.cpu())
    want = torch.zeros((Vp, 2 * Dp), dtype=BF16)
    want[:V, :D] = hi
    want[:V, Dp:Dp + D] = lo
    assert torch.equal(_bits16(E2), _bits16(want)), "E2 layout / rounding"
    ref = sqnorm_emulated(E)
    assert torch.equal(sq[:V].view(torch.int32), ref.view(torch.int32)), \
        "sqnorm: %d of %d rows differ from the emulation" % (int((sq[:V] != ref).sum()), V)
    assert bool((sq[V:] == INF).all())
    assert torch.equal(Ec, E.clamp(-1.0, 1.0))
    rel = float(((sq[:V].double() - (E.double() ** 2).sum(1)).abs() / (E.double() ** 2).sum(1)).max())
    _report("embed_split", V=V, D=D, Dp=Dp, sqnorm_rel_err_vs_f64=rel)


@pytest.mark.parametrize("N", [64, 128, 512])
def test_gemm_split_epilogue_is_rne(N):
    """MD_EPI_BIAS_SPLIT against RNE directly: dyadic operands make y exact in fp32 with up to 22 significant bits."""
    M, Kd = 4192, 768
    g = _gen(N)
    A = torch.randint(-255, 256, (M, Kd), generator=g, device=DEV).to(BF16)
    W = (torch.randint(-15, 16, (N, Kd), generator=g, device=DEV) * 2.0 ** -4).to(BF16)
    bias = torch.randint(-4096, 4097, (N,), generator=g, device=DEV) * 2.0 ** -4
    buf, out = _guarded(M * 2 * N, BF16, float("nan"))
    ops.linear(A, W, bias, _lib.EPI_BIAS_SPLIT, out=out.view(M, 2 * N))
    torch.cuda.synchronize()
    _check_guard(buf, M * 2 * N, float("nan"), "split epilogue")
    y64 = A.double() @ W.double().T + bias.double()
    y = y64.float()
    assert torch.equal(y.double(), y64), "test construction: y not exact in fp32"
    hi, lo = _rne_split(y.cpu())
    assert bool((lo.float() != 0).any())
    got = out.view(M, 2 * N)
    assert torch.equal(_bits16(got[:, :N]), _bits16(hi))
    assert torch.equal(_bits16(got[:, N:]), _bits16(lo))


# ------------------------------------------------------------------------------------------------ B. tensor core, exact data
WIDTHS = [(64, 64), (128, 128), (768, 768), (16, 64), (100, 128), (500, 512)]
VOCABS = [1, 200, 256, 257, 512, 729, 1000]
ROWS = [1, 127, 128, 129]
BIG = 1023                    # 10 significant bits: hi = 1024, lo = -1


def tie_pairs(V):
    """(c, c') column pairs made equal: one column half; halves c and c + 128 of a tile; half 1 of tile 0 against half 0
    of tile 1 (the higher index sits in the lower half); tiles; column 0 and V - 1."""
    cand = [(3, 9), (17, 145), (130, 261), (40, 296), (0, V - 1)]
    out, used = [], set()
    for c, d in cand:
        if d < V and c < d and c not in used and d not in used:
            out.append((c, d))
            used |= {c, d}
    return out


def _sparse(n, D, g, lo=257, hi=BIG + 1, nnz=3):
    """rows with nnz entries of 9 to 10 significant bits (lo and hi both nonzero), random signs and positions"""
    r = torch.zeros((n, D), device=DEV)
    pos = torch.rand((n, D), generator=g, device=DEV).argsort(1)[:, :nnz]
    val = torch.randint(lo, hi, (n, nnz), generator=g, device=DEV).float()
    sgn = torch.randint(0, 2, (n, nnz), generator=g, device=DEV).float() * 2 - 1
    r.scatter_(1, pos, val * sgn)
    return r


def exact_embedding(V, D, seed):
    """integer E [V, D] (dense rows in [-3, 3], every fifth row sparse), bias [V] in [-50000, -20000] (so dense x rows
    have only negative logits); the columns of `tie_pairs(V)` are duplicated (rows of +-1023 entries, bias = the maximum)"""
    g = _gen(seed)
    E = torch.randint(-3, 4, (V, D), generator=g, device=DEV).float()
    sp = torch.arange(V, device=DEV) % 5 == 2
    E[sp] = _sparse(int(sp.sum()), D, g)
    bias = torch.randint(-50000, -19999, (V,), generator=g, device=DEV).float()
    pairs = tie_pairs(V)
    if pairs:
        top = _sparse(len(pairs), D, g, lo=BIG, hi=BIG + 1)
        bmax = bias.max()
        for k, (c, d) in enumerate(pairs):
            E[c] = E[d] = top[k]
            bias[c] = bias[d] = bmax
    return E, bias, pairs


def exact_rows(M, E, pairs, seed):
    """integer x [M, D]: the planted-tie rows x = E_c first, then dense rows, sparse rows and exact hits x = E_v"""
    V, D = E.shape
    g = _gen(seed)
    x = torch.randint(-3, 4, (M, D), generator=g, device=DEV).float()
    r = torch.arange(M, device=DEV)
    sp = r % 4 == 1
    x[sp] = _sparse(int(sp.sum()), D, g)
    hit = r % 4 == 3
    x[hit] = E[torch.randint(0, V, (int(hit.sum()),), generator=g, device=DEV)]
    for k, (c, _) in enumerate(pairs[:M]):
        x[k] = E[c]
    return x


def exact_keys(x, E, bias, mode):
    """float64 keys (exact here): mode 0 |E_v|^2 - 2 x.E_v (unclamped), mode 1 -(x.E_v + b_v)"""
    dot = x.double() @ E.double().T
    if mode == 0:
        key = (E.double() ** 2).sum(1)[None, :] - 2 * dot
    else:
        key = -(dot + bias.double()[None, :])
    s = x.double().abs() @ E.double().abs().T
    assert float(key.abs().max()) < 2 ** 24 and float(s.max()) * 1.02 < 2 ** 24, "test construction: keys not exact in fp32"
    return key


def _check_exact(x, E, bias, se, mode, pairs, presplit, what):
    cst = se.sqnorm if mode == 0 else se.logit_cst(bias)
    if presplit:
        idx, mg = run_tc(se, mode, cst, presplit=presplit_via_gemm(x, se.Dp))
    else:
        idx, mg = run_tc(se, mode, cst, x=x)
    key = exact_keys(x, E, bias, mode)
    ref_idx, ref_mg = _first_min(key)
    for k, (c, d) in enumerate(pairs[:x.shape[0]]):        # the planted ties are ties at the top
        assert int(ref_idx[k]) == c and float(ref_mg[k]) == 0.0, "test construction: pair (%d, %d)" % (c, d)
    bad = idx.long() != ref_idx
    if bool(bad.any()):
        i = int(bad.nonzero()[0])
        raise AssertionError("%s: %d ids differ from the exact argmin; first row %d: got %d, want %d (margin %g)"
                             % (what, int(bad.sum()), i, int(idx[i]), int(ref_idx[i]), float(ref_mg[i])))
    badm = mg.double() != ref_mg
    if bool(badm.any()):
        i = int(badm.nonzero()[0])
        raise AssertionError("%s: %d margins differ from the exact one; first row %d: got %r, want %r"
                             % (what, int(badm.sum()), i, float(mg[i]), float(ref_mg[i])))
    return int((ref_mg == 0).sum())


@pytest.mark.parametrize("V", VOCABS)
@pytest.mark.parametrize("D,Dp", WIDTHS, ids=["D%d-Dp%d" % w for w in WIDTHS])
def test_tc_exact(D, Dp, V):
    """ids, margins and planted ties bit-exact at M = 1, 127, 128, 129, both modes, fp32 x and the GEMM-written presplit."""
    E, bias, pairs = exact_embedding(V, D, seed=V * 7 + D)
    se = ops.SplitEmbedding(E)
    assert se.Dp == Dp
    ties = 0
    for M in ROWS:
        x = exact_rows(M, E, pairs, seed=M + V + D)
        if V % 256 and M > 1:                       # dense rows: every real logit negative, so a 0 padding constant would win
            assert bool(((x.double() @ E.double().T + bias.double()) < 0).all(1).any())
        for mode in (0, 1):
            for presplit in (False, True):
                ties += _check_exact(x, E, bias, se, mode, pairs, presplit,
                                     "D=%d V=%d M=%d mode %d %s" % (D, V, M, mode, "presplit" if presplit else "fp32 x"))
    _report("tc_exact", D=D, V=V, tied_rows=ties)


def _persistent_M():
    sms = torch.cuda.get_device_properties(DEV).multi_processor_count
    return 3 * sms * 128 + 77, sms                 # 3 sms + 1 row blocks: every CTA walks >= 3, the last one partial


@pytest.mark.parametrize("D,Dp,V", [(128, 128, 729), (100, 128, 257)])
def test_tc_exact_persistent(D, Dp, V):
    """every CTA walks at least three 128-row blocks (the two TMEM accumulators' phases carry across blocks)."""
    M, sms = _persistent_M()
    E, bias, pairs = exact_embedding(V, D, seed=V + 3)
    se = ops.SplitEmbedding(E)
    x = exact_rows(M, E, pairs, seed=M)
    for mode in (0, 1):
        for presplit in (False, True):
            _check_exact(x, E, bias, se, mode, pairs, presplit, "persistent M=%d mode %d" % (M, mode))
    _report("tc_exact_persistent", M=M, sms=sms, D=D, V=V)


def test_tc_exact_production_pass():
    """M = 256 x 2096 at V = 729, D = 128; the float64 reference in row chunks on the GPU (exact for this data)."""
    M, V, D = 256 * 2096, 729, 128
    E, bias, pairs = exact_embedding(V, D, seed=99)
    se = ops.SplitEmbedding(E)
    x = exact_rows(M, E, pairs, seed=2096)
    for mode in (0, 1):
        for presplit in ((False, True) if mode == 0 else (False,)):
            cst = se.sqnorm if mode == 0 else se.logit_cst(bias)
            if presplit:
                idx, mg = run_tc(se, mode, cst, presplit=presplit_via_gemm(x, se.Dp))
            else:
                idx, mg = run_tc(se, mode, cst, x=x)
            for r0 in range(0, M, 65536):
                key = exact_keys(x[r0:r0 + 65536], E, bias, mode)
                ref_idx, ref_mg = _first_min(key)
                assert torch.equal(idx[r0:r0 + 65536].long(), ref_idx), "mode %d rows %d.." % (mode, r0)
                assert torch.equal(mg[r0:r0 + 65536].double(), ref_mg), "mode %d margins rows %d.." % (mode, r0)
    _report("tc_exact_production_pass", M=M, V=V, D=D)


# ------------------------------------------------------------------------------------------------ C. tensor core, random data
def tc_key_bound(x, E, bias, mode, Dp):
    """beta(m, v) >= |fp32 key the kernel computes - float64 key of the same fp32 inputs|.  S = sum_d |x_d||E_vd|.

    1. Split residuals.  xh = RNE_bf16(x), |x - xh| <= u|x| with u = 2^-8; xl = RNE_bf16(x - xh), so the dropped
       residual |x - xh - xl| <= u^2|x| = 2^-16|x|, likewise for E.  x.E - (xh + xl).(Eh + El) therefore stays within
       (2 * 2^-16 + 2^-32)(1 + 2^-16) S <= 2^-15 (1 + 2^-14) S.
    2. Accumulation.  The 4 Dp products of bf16 values are exact in fp32; tcgen05 adds them in an order and with a
       rounding the PTX ISA does not specify, so each add is charged a full ulp (2^-23 relative, truncation), over
       n = 4 Dp adds: gamma = n 2^-23 / (1 - n 2^-23) times sum |products| <= (1 + 2^-8)^4 S <= (1 + 2^-5) S.
    3. |E_v|^2 (mode 0) in fp32 by IEEE fmaf / adds over D terms: gamma_D = D 2^-24 / (1 - D 2^-24) times |E_v|^2.
    4. The final fmaf(-2, dot, cst) (mode 0) or add (mode 1): one rounding, 2^-24 of the computed operands' magnitude.
    mode 0: beta = 2 (1 + 2) + 3 + 4;   mode 1: beta = (1 + 2) + 4 (the bias is exact)."""
    x64, E64 = x.double(), E.double()
    S = x64.abs() @ E64.abs().T
    n = 4 * Dp
    g_acc = n * 2.0 ** -23 / (1 - n * 2.0 ** -23)
    dot_err = 2.0 ** -15 * (1 + 2.0 ** -14) * S + g_acc * (1 + 2.0 ** -5) * S
    if mode == 0:
        D = E.shape[1]
        sq = (E64 ** 2).sum(1)[None, :]
        cst_err = D * U32 / (1 - D * U32) * sq
        return 2 * dot_err + cst_err + U32 * (1 + 2.0 ** -20) * (sq + cst_err + 2 * (S + dot_err))
    return dot_err + U32 * (1 + 2.0 ** -20) * (S + dot_err + bias.double().abs()[None, :])


def random_case(kind, M, V, D, seed):
    g = _gen(seed)
    E = torch.randn(V, D, generator=g, device=DEV)
    bias = torch.randn(V, generator=g, device=DEV)
    if kind == "gauss":
        x = torch.randn(M, D, generator=g, device=DEV) * 0.8
    else:                                              # near-ties: near-duplicate rows, x = E_v + small noise
        E[1::2] = E[0::2][:V // 2] + 1e-4 * torch.randn(V // 2, D, generator=g, device=DEV)
        x = E[torch.randint(0, V, (M,), generator=g, device=DEV)] + 1e-3 * torch.randn(M, D, generator=g, device=DEV)
    return x, E, bias


def check_bound(x, E, bias, se, mode, what):
    cst = se.sqnorm if mode == 0 else se.logit_cst(bias)
    idx, mg = run_tc(se, mode, cst, x=x)
    key = exact_keys_any(x, E, bias, mode)
    beta = tc_key_bound(x, E, bias, mode, se.Dp)
    ref_idx, ref_mg = _first_min(key)
    rows = torch.arange(x.shape[0], device=DEV)
    il = idx.long()
    gap = key[rows, il] - key[rows, ref_idx]
    allow = beta[rows, il] + beta[rows, ref_idx]
    if not bool((gap <= allow).all()):
        i = int((gap - allow).argmax())
        raise AssertionError("%s: row %d: id %d is %g above the optimum %d, bound %g" % (what, i, int(il[i]), float(gap[i]),
                                                                                       int(ref_idx[i]), float(allow[i])))
    bmax = beta.max(1).values
    sure = ref_mg > beta[rows, ref_idx] + bmax
    assert bool((il[sure] == ref_idx[sure]).all()), "%s: %d ids differ where the margin exceeds the bounds" % (what, int((il[sure] != ref_idx[sure]).sum()))
    if E.shape[0] > 1:
        merr = (mg.double() - ref_mg).abs()
        mallow = 2 * bmax + U32 * (ref_mg + 2 * bmax)
        assert bool((merr <= mallow).all()), "%s: margin error %g > %g" % (what, float(merr.max()), float(mallow[merr.argmax()]))
        mfrac = float((merr / (2 * bmax)).max())
    else:
        assert bool((mg == INF).all())
        mfrac = 0.0
    return float((gap / allow).max()), mfrac, float(sure.float().mean()), int((il != ref_idx).sum())


def exact_keys_any(x, E, bias, mode):
    dot = x.double() @ E.double().T
    if mode == 0:
        return (E.double() ** 2).sum(1)[None, :] - 2 * dot
    return -(dot + bias.double()[None, :])


@pytest.mark.parametrize("V", VOCABS)
@pytest.mark.parametrize("D,Dp", WIDTHS, ids=["D%d-Dp%d" % w for w in WIDTHS])
def test_tc_random_within_bound(D, Dp, V):
    """ids near-optimal within beta(id) + beta(best), equal to the float64 argmin / argmax wherever the float64 margin
    exceeds beta(best) + max_v beta, margins within 2 max_v beta; Gaussian data and near-ties; M = 1, 129, 1000."""
    worst = [0.0, 0.0]
    flips, decided = 0, []
    for kind in ("gauss", "near"):
        for M in (1, 129, 1000):
            x, E, bias = random_case(kind, M, V, D, seed=M * 11 + V + D + (kind == "near"))
            se = ops.SplitEmbedding(E)
            for mode in (0, 1):
                gfrac, mfrac, sure, fl = check_bound(x, E, bias, se, mode, "%s D=%d V=%d M=%d mode %d" % (kind, D, V, M, mode))
                worst = [max(worst[0], gfrac), max(worst[1], mfrac)]
                flips += fl
                decided.append(sure)
    _report("tc_random", D=D, V=V, id_gap_over_bound=worst[0], margin_err_over_bound=worst[1], ids_not_argmin=flips,
            rows_decided_min=min(decided))


@pytest.mark.parametrize("D", [128, 500, 768])
def test_tc_key_error_measured(D):
    """The per-key error itself: with V = 2 and E = [0 ; E_v] (bias [0, b_v]) the zero column's key is exactly 0, so
    the margin is |k_v| and the id gives its sign: the kernel's fp32 key, against float64, as a fraction of beta."""
    g = _gen(D)
    Efull = torch.randn(64, D, generator=g, device=DEV)
    bfull = torch.randn(64, generator=g, device=DEV)
    x = torch.randn(4096, D, generator=g, device=DEV) * 0.8
    x[:64] = Efull + 1e-3 * torch.randn(64, D, generator=g, device=DEV)
    worst = {0: 0.0, 1: 0.0}
    for v in range(64):
        E = torch.zeros(2, D, device=DEV)
        E[1] = Efull[v]
        bias = torch.zeros(2, device=DEV)
        bias[1] = bfull[v]
        se = ops.SplitEmbedding(E)
        for mode in (0, 1):
            idx, mg = run_tc(se, mode, se.sqnorm if mode == 0 else se.logit_cst(bias), x=x)
            k = torch.where(idx == 1, -mg, mg).double()
            key = exact_keys_any(x, E, bias, mode)[:, 1]
            beta = tc_key_bound(x, E, bias, mode, se.Dp)[:, 1]
            frac = float(((k - key).abs() / beta).max())
            assert frac <= 1.0, "D=%d v=%d mode %d: key error %.3g of beta" % (D, v, mode, frac)
            worst[mode] = max(worst[mode], frac)
    _report("tc_key_error", D=D, mode0_err_over_beta=worst[0], mode1_err_over_beta=worst[1])


# ------------------------------------------------------------------------------------------------ D. fp32 kernels, bit-exact
def round_kernel_emulated(x, E, bias):
    """float32 emulation of round_kernel<MODE> (rounding.cu) for both modes: (keys mode 0, keys mode 1)."""
    M, D = x.shape
    V = E.shape[0]
    acc = torch.zeros((M, V), dtype=F32, device=DEV)
    for d in range(D):                                       # per-thread fmaf chain over d, in order, across slices
        acc = fma32(x[:, d:d + 1], E[:, d][None, :], acc)
    xsq = torch.zeros(M, dtype=F32, device=DEV)
    esq = torch.zeros(V, dtype=F32, device=DEV)
    for s0 in range(0, D, 128):
        h = []
        for c0 in (s0, s0 + 64):                              # |x|^2: two 64-column halves, xor-1 shuffle
            s = torch.zeros(M, dtype=F32, device=DEV)
            for c in range(c0, min(c0 + 64, D)):
                s = fma32(x[:, c], x[:, c], s)
            h.append(s)
        xsq = xsq + (h[0] + h[1])
        q = []
        for c0 in (s0, s0 + 32, s0 + 64, s0 + 96):           # |E_v|^2: four 32-column quarters, (q0 + q1) + (q2 + q3)
            s = torch.zeros(V, dtype=F32, device=DEV)
            for c in range(c0, min(c0 + 32, D)):
                s = fma32(E[:, c], E[:, c], s)
            q.append(s)
        esq = esq + ((q[0] + q[1]) + (q[2] + q[3]))
    key0 = torch.clamp_min((esq[None, :] + xsq[:, None]) - 2.0 * acc, 0.0)
    key1 = -(acc + bias[None, :])
    return key0, key1


def _first_min32(key):
    """as the kernel: lowest id of the minimum, margin = second - best in fp32"""
    V = key.shape[1]
    best = key.min(1).values
    ar = torch.arange(V, device=key.device).expand_as(key)
    idx = torch.where(key == best[:, None], ar, V).min(1).values
    if V == 1:
        return idx, torch.full_like(best, INF)
    two = key.topk(2, dim=1, largest=False).values
    return idx, two[:, 1] - two[:, 0]


@pytest.mark.parametrize("V", [1, 63, 64, 65, 729])
@pytest.mark.parametrize("D", [4, 100, 128, 132, 256, 500, 768])
def test_fp32_kernels_bit_exact(D, V):
    """md_round_argmin / md_logits_argmax: ids and margins identical to the emulation at M = 1, 127, 128, 129, 5000,
    including clamp-to-0 ties (x = E_v with near-duplicate rows) and duplicate rows across the 16 vocabulary lanes."""
    g = _gen(D * 5 + V)
    M = 5000
    E = torch.randn(V, D, generator=g, device=DEV)
    if V >= 64:
        E[1] = E[0]                                           # lanes 0 / 1 of one chunk
        E[16] = E[2]                                          # the same lane
        E[V - 1] = E[5]                                       # another chunk
        E[7] = E[6]
        E[7, 0] = torch.nextafter(E[6, 0], torch.tensor(INF, device=DEV))     # a near-duplicate
    bias = torch.randn(V, generator=g, device=DEV)
    if V >= 64:
        bias[1], bias[16], bias[V - 1], bias[7] = bias[0], bias[2], bias[5], bias[6]
    x = torch.randn(M, D, generator=g, device=DEV) * 0.8
    pick = torch.randint(0, V, (M // 4,), generator=g, device=DEV)
    x[0::4] = E[pick]                                         # exact hits
    x[2::8] = 3 * E[pick[: x[2::8].shape[0]]]                 # dominant logits on the duplicated rows
    if V >= 64:
        x[1:40:2] = E[torch.tensor([0, 1, 2, 16, 5, V - 1, 6, 7] * 3, device=DEV)[:20]]
    key0, key1 = round_kernel_emulated(x, E, bias)
    counts = {}
    for mode, key in ((0, key0), (1, key1)):
        ref_idx, ref_mg = _first_min32(key)
        for m in (1, 127, 128, 129, M):
            idx, mg = run_fp32(x[:m].contiguous(), E, bias, mode)
            bad = idx.long() != ref_idx[:m]
            assert not bool(bad.any()), "mode %d M=%d: %d ids differ from the emulation (first row %d)" % (
                mode, m, int(bad.sum()), int(bad.nonzero()[0]))
            badm = mg != ref_mg[:m]
            assert not bool(badm.any()), "mode %d M=%d: %d margins differ (first row %d: %r vs %r)" % (
                mode, m, int(badm.sum()), int(badm.nonzero()[0]), float(mg[badm][0]), float(ref_mg[:m][badm][0]))
        counts[mode] = int((ref_mg == 0).sum())
    _report("fp32_bit_exact", D=D, V=V, rows=M, tied_rows_mode0=counts[0], tied_rows_mode1=counts[1],
            clamped_ties=int(((key0.min(1).values == 0) & (_first_min32(key0)[1] == 0)).sum()))


# ------------------------------------------------------------------------------------------------ E. dist_scores, get_logits
@pytest.mark.parametrize("D", [100, 128, 768])
def test_dist_scores_bit_exact(D):
    """md_dist_scores from its own dot / esq inputs: lane-strided fmaf chain for |x|^2, xor-16 ... 1 tree,
    __fadd_rn / __fsub_rn / __fmul_rn, IEEE sqrtf; dot_stride > V; some d^2 < 0 (clamped to 0)."""
    M, V, stride = 300, 729, 736
    g = _gen(D)
    x = torch.randn(M, D, generator=g, device=DEV)
    esq = torch.rand(V, generator=g, device=DEV) * 150 + 50
    dot = torch.randn(M, stride, generator=g, device=DEV) * 10
    q64 = (x.double() ** 2).sum(1)
    dot[::5, :V] = ((esq.double()[None, :] + q64[::5, None]) / 2).float()   # d^2 near 0, both signs
    buf, out = _guarded(M * V, F32, float("nan"))
    K.dist_scores(x, dot, esq, out.view(M, V))
    torch.cuda.synchronize()
    _check_guard(buf, M * V, float("nan"), "dist_scores")
    n = -(-D // 32) * 32
    xp = torch.zeros((M, n), dtype=F32, device=DEV)
    xp[:, :D] = x
    lanes = torch.zeros((M, 32), dtype=F32, device=DEV)
    for k in range(n // 32):
        col = xp[:, 32 * k:32 * k + 32]
        lanes = fma32(col, col, lanes)
    q = _butterfly(lanes)
    d2 = (esq[None, :] + q[:, None]) - 2.0 * dot[:, :V]
    ref = -(torch.clamp_min(d2, 0.0).double().sqrt().float())
    got = out.view(M, V)
    assert int((d2 < 0).sum()) > 0
    assert torch.equal(got.view(torch.int32), ref.view(torch.int32)), "%d of %d scores differ" % (int((got != ref).sum()), M * V)
    _report("dist_scores", D=D, clamped=int((d2 < 0).sum()), bit_exact=M * V)


def _model(V, D, E, bias):
    targs = dict(hidden_dim=D, hidden_t_dim=128, vocab_size=V, seq_len=64, dropout=0.1, noise_schedule="sqrt",
                 diffusion_steps=20, timestep_respacing="", rescale_timesteps=True, predict_xstart=True,
                 encoder_config=dict(num_hidden_layers=1))
    torch.manual_seed(0)
    model, _ = create_model_and_diffusion(**targs)
    model.eval().requires_grad_(False).to(DEV)
    with torch.no_grad():
        model.word_embedding.weight.copy_(E)
        model.lm_head.bias.copy_(bias)
    return model


@pytest.mark.parametrize("D", [128, 100])
def test_get_logits_exact(D):
    """logits_mode 1: x.E_v + b_v exactly; logits_mode 2: RN(-sqrt(d^2)) of the exact squared distance."""
    V = 729
    E, bias, pairs = exact_embedding(V, D, seed=D + 1)
    model = _model(V, D, E, bias)
    x = exact_rows(2 * 64, E, pairs, seed=D).view(2, 64, D)
    logits = model.get_logits(x)
    ref = x.view(-1, D).double() @ E.double().T + bias.double()
    assert torch.equal(logits.view(-1, V).double(), ref)
    model.logits_mode = 2
    d2 = (E.double() ** 2).sum(1)[None, :] + (x.view(-1, D).double() ** 2).sum(1)[:, None] - 2 * (x.view(-1, D).double() @ E.double().T)
    assert float(d2.max()) < 2 ** 24 and float(d2.min()) >= 0
    scores = model.get_logits(x)
    assert torch.equal(scores.view(-1, V).view(torch.int32), (-(d2.sqrt())).float().view(torch.int32))
    model.logits_mode = 1
    tok = model.decode_tokens(x)
    assert torch.equal(tok.view(-1), _first_min(-ref)[0])


@pytest.mark.parametrize("D", [128, 100])
def test_decode_tokens_vs_get_logits(D):
    """decode_tokens == argmax(get_logits) == the float64 argmax wherever the float64 gap exceeds the mode-1 bound."""
    V = 729
    g = _gen(D + 5)
    E = torch.randn(V, D, generator=g, device=DEV)
    bias = torch.randn(V, generator=g, device=DEV)
    model = _model(V, D, E, bias)
    x = torch.randn(4, 64, D, generator=g, device=DEV)
    tok = model.decode_tokens(x).view(-1)
    lg = model.get_logits(x).view(-1, V)
    x2 = x.view(-1, D)
    key = exact_keys_any(x2, E, bias, 1)
    beta = tc_key_bound(x2, E, bias, 1, ops.padded_width(D))
    ref_idx, ref_mg = _first_min(key)
    rows = torch.arange(x2.shape[0], device=DEV)
    sure = ref_mg > beta[rows, ref_idx] + beta.max(1).values
    assert float(sure.float().mean()) > 0.9
    assert torch.equal(tok[sure], ref_idx[sure])
    assert torch.equal(lg.argmax(1)[sure], ref_idx[sure])
    _report("decode_vs_get_logits", D=D, rows_decided=float(sure.float().mean()), agree_all=float((tok == lg.argmax(1)).float().mean()))


# ------------------------------------------------------------------------------------------------ F. non-finite rows
def _nonfinite_x(M, D, g):
    x = torch.randn(M, D, generator=g, device=DEV)
    x[0] = float("nan")
    x[1, 3] = float("nan")
    x[2, 5] = INF
    x[3, D - 1] = -INF
    x[4, 0], x[4, 1] = float("nan"), INF
    x[5] = INF
    return x


@pytest.mark.parametrize("D", [128, 100])
@pytest.mark.parametrize("V", [729, 200])
def test_nonfinite_rows_give_valid_ids(V, D):
    """Every id the four reductions write lies in [0, V): NaN / +-inf in x, in E rows and in bias entries.  A row whose
    keys are all NaN or +inf (the tensor-core kernels: any non-finite x; mode 1: every bias -inf or NaN) gets id 0, as
    torch.argmax gives.  Finite rows are unaffected by the non-finite rows launched with them.  Only the ids are used."""
    g = _gen(V + D)
    M = 300
    x = _nonfinite_x(M, D, g)
    E = torch.randn(V, D, generator=g, device=DEV)
    bias = torch.randn(V, generator=g, device=DEV)
    Ebad = E.clone()
    Ebad[5, 7], Ebad[150, 0], Ebad[V - 2, 1] = float("nan"), INF, -INF
    bbad = bias.clone()
    bbad[7], bbad[8], bbad[9] = float("nan"), INF, -INF
    cases = [("x", E, bias), ("E", Ebad, bias), ("bias", E, bbad), ("all", Ebad, bbad),
             ("bias -inf", E, torch.full_like(bias, -INF)), ("bias nan", E, torch.full_like(bias, float("nan")))]
    fin = torch.isfinite(x).all(1)
    for name, Ec, bc in cases:
        se = ops.SplitEmbedding(Ec)
        res = {}
        for mode in (0, 1):
            if mode == 0 and name.startswith("bias"):
                continue
            cst = se.sqnorm if mode == 0 else se.logit_cst(bc)
            res["tc%d" % mode] = run_tc(se, mode, cst, x=x)[0]
            assert torch.equal(run_tc(se, mode, cst, x=x)[0], res["tc%d" % mode]), "not deterministic"
            res["fp32_%d" % mode] = run_fp32(x, Ec, bc, mode)[0]
            for k in ("tc%d" % mode, "fp32_%d" % mode):
                ids = res[k]
                assert bool(((ids >= 0) & (ids < V)).all()), "%s / %s: ids outside [0, %d): %s" % (
                    name, k, V, ids[(ids < 0) | (ids >= V)][:8].tolist())
                assert int(ids[0]) == 0, "%s / %s: the all-NaN row got id %d" % (name, k, int(ids[0]))
            tc = res["tc%d" % mode]
            assert bool((tc[~fin] == 0).all()), "%s / tc%d: a non-finite x row did not get id 0" % (name, mode)
            if name in ("bias -inf", "bias nan"):          # every key +inf / NaN (md_logits_argmax takes the lowest id
                assert bool((tc == 0).all())                # of a +inf key, so an inf in x, which mixes NaN and +inf keys,
                assert bool((res["fp32_1"][fin] == 0).all()) and int(res["fp32_1"][0]) == 0     # may give another id)
            xf = x[fin].contiguous()
            assert torch.equal(run_tc(se, mode, cst, x=xf)[0], tc[fin]), "%s / tc%d: finite rows changed" % (name, mode)
            assert torch.equal(run_fp32(xf, Ec, bc, mode)[0], res["fp32_%d" % mode][fin])
    model = _model(V, D, E, bias)
    tok = model.decode_tokens(x.view(3, 100, D)).view(-1)
    assert bool(((tok >= 0) & (tok < V)).all()) and bool((tok[~fin] == 0).all())
