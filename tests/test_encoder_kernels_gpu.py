"""The encoder's three kernel families — `md_linear_bf16` (GEMM + epilogue), `md_attention_bf16`, `md_layernorm_bf16` —
checked element by element against float64 references, through `musediffusion_b200.ops` (the C-ABI path production uses).

Every bf16 output is one round-to-nearest-even (RNE) of a value the kernel computes in fp32.  `assert_rounded` checks each
element against RNE of the float64 reference; where the kernel's fp32 value may differ from the reference by up to `delta`
(derived per kernel below), an element whose reference lies within `delta` of a rounding midpoint may take either
neighbour.  Inputs are built so that this rule is exact wherever it can be:

  A  GEMM on integer / dyadic operands: every partial sum is exact in fp32, so fp32 output is bit-identical to float64 and
     bf16 output is exactly RNE(ref), on every launch path of `md_linear_bf16_cols` (pair, single-CTA BN 256 / 128).
  B  GELU / tanh epilogues on one-hot A rows, so the pre-activation z is known exactly, against float64 GELU / tanh.
  C  attention: exact routing (every query picks one key with all other weights exactly 0), exact masking (a padded key
     that leaks is 2^18.75 times heavier than a real one), and a per-element bound on random data.
  D  LayerNorm at every supported width with a delta derived from the kernel's operation order; constant rows must give
     exactly beta.
  E  the non-default kernel variants (MD_GEMM_PAIR=0, MD_ATT_POLY=1..4, MD_LN_HOIST=0) re-run the structured cases in a
     child process, because the library reads those switches once per process.

References are numpy float64 on the CPU; torch float64 on the GPU is used only for GEMMs whose operands are all
dyadic, where the result is exact in any summation order.  Nothing uses TF32 or an fp32 matmul as a reference."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)

from musediffusion_b200 import _lib, ops  # noqa: E402

DEV = torch.device("cuda:0")
BF16, F32 = torch.bfloat16, torch.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VARIANT_GUARD = "MD_ENCODER_TEST_CHILD"       # set in the child processes of section E: they must not spawn their own
U32 = 2.0 ** -24                              # fp32 unit roundoff


# ------------------------------------------------------------------------------------------------ shared helpers
def _rne(ref64, dtype):
    """RNE of float64 values to `dtype`, on the CPU.  fp32: the IEEE cast.  bf16: torch's double -> bf16 cast rounds
    through float32 first (1 + 2^-8 + 2^-30 becomes 1.0, not 1 + 2^-7), so values that are not exact in fp32 are rounded
    on their float64 bit pattern to 8 significant bits, after which the cast is exact.  (Below bf16's normal range,
    |x| < 2^-126, the cast is used as is; no check here depends on an exact rounding that small.)"""
    if dtype == F32:
        return ref64.to(F32)
    r32 = ref64.to(F32)
    if torch.equal(r32.to(torch.float64), ref64):
        return r32.to(BF16)
    bits = ref64.contiguous().view(torch.int64)
    drop = 52 - 7
    bits = (bits + ((1 << (drop - 1)) - 1) + ((bits >> drop) & 1)) & ~((1 << drop) - 1)
    rounded = bits.view(torch.float64)
    return torch.where(ref64.abs() < 2.0 ** -126, ref64, rounded).to(BF16)


def assert_rounded(out, ref64, delta, what=""):
    """Every element of `out` must equal RNE(ref64) in out's dtype, except that an element whose ref64 lies within
    `delta` of a rounding midpoint may take either neighbour: out must be the RNE of SOME value within delta of ref64,
    i.e. RNE(ref - delta) <= out <= RNE(ref + delta).  delta: scalar or array broadcastable to out (0 = exact).
    Returns (elements that took the other neighbour, max |ref - midpoint| / delta over them)."""
    out = out.detach().cpu()
    ref64 = torch.as_tensor(ref64, dtype=torch.float64).cpu()
    assert out.shape == ref64.shape, (out.shape, ref64.shape)
    want = _rne(ref64, out.dtype)
    d = torch.as_tensor(delta, dtype=torch.float64)
    if not bool((d != 0).any()):
        ok = out == want
    else:
        ok = (out >= _rne(ref64 - d, out.dtype)) & (out <= _rne(ref64 + d, out.dtype))
    if not bool(ok.all()):
        bad = ~ok
        err = torch.where(bad, (out.to(torch.float64) - ref64).abs().nan_to_num(float("inf")), torch.zeros((), dtype=torch.float64))
        flat = int(err.argmax())
        cols = out.shape[-1] if out.dim() > 0 else 1
        rc = (flat // cols, flat % cols)
        o, r, w = float(out.reshape(-1)[flat]), float(ref64.reshape(-1)[flat]), float(want.reshape(-1)[flat])
        dd = float(d.expand(out.shape).reshape(-1)[flat]) if d.dim() else float(d)
        raise AssertionError("%s: %d of %d elements are not RNE(ref) within delta; worst at (row, col) = %s: out %r, ref %r, "
                             "RNE(ref) %r, delta %.3g" % (what, int(bad.sum()), out.numel(), rc, o, r, w, dd))
    other = out != want
    n_other = int(other.sum())
    if n_other == 0:
        return 0, 0.0
    mid = (out.to(torch.float64) + want.to(torch.float64)) / 2
    frac = ((ref64 - mid).abs() / d.expand(out.shape))[other]
    return n_other, float(frac.max())


def _report(name, **kv):
    print("MEASURED %s %s" % (name, " ".join("%s=%s" % (k, ("%.4g" % v) if isinstance(v, float) else v) for k, v in kv.items())))


def _guarded(shape, dtype):
    """An output view inside a NaN-filled allocation with guard regions before and after it (the front one keeps the
    view 16-byte aligned, as the TMA store needs)."""
    n = math.prod(shape)
    front, back = 64, 4096 + 8
    buf = torch.full((front + n + back,), float("nan"), dtype=dtype, device=DEV)
    return buf, buf[front:front + n].view(shape), front, n


def _check_guard(buf, front, n, what):
    ib = torch.int16 if buf.dtype == BF16 else torch.int32
    nan_bits = torch.full((1,), float("nan"), dtype=buf.dtype).view(ib).item()
    g = torch.cat([buf[:front], buf[front + n:]]).view(ib)
    assert bool((g == nan_bits).all()), "%s: %d guard elements outside the out= view were written" % (what, int((g != nan_bits).sum()))


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


# ------------------------------------------------------------------------------------------------ A. GEMM, exact
def gemm_path(M, N, out_f32, split=False):
    """The launch path `md_linear_bf16_cols` picks (gemm.cu: BN = 256 if N % 256 == 0 or N > 512 else 128; CTA pair
    when N % 256 == 0, M >= 1024, bf16 output, not the split epilogue) with the default MD_GEMM_PAIR=1."""
    if N % 256 == 0 and M >= 1024 and not out_f32 and not split:
        return "pair"
    return "bn256" if (N % 256 == 0 or N > 512) else "bn128"


def _dyadic(shape, g, bits, scale_log2):
    """integers in (-2^bits, 2^bits) times 2^scale_log2 (fp32; at most `bits` significant bits)"""
    return (torch.randint(-(1 << bits) + 1, 1 << bits, shape, generator=g, device=DEV).float() * 2.0 ** scale_log2)


def _gemm_operands(M, N, K, seed):
    """A: bf16 integers in [-8, 8]; W: bf16 integers in [-8, 8] x 2^-6 (outputs carry up to ~19 significant bits, more
    than bf16 holds); bias: dyadic, |b| < 64, <= 12 significant bits.  Every product is a multiple of 2^-6 with |p| <= 1 and
    every partial sum stays below K < 2^12, so the fp32 tensor-core accumulation and the epilogue adds are exact."""
    g = _gen(seed)
    A = torch.randint(-8, 9, (M, K), generator=g, device=DEV).to(BF16)
    W = (torch.randint(-8, 9, (N, K), generator=g, device=DEV).float() * 2.0 ** -6).to(BF16)
    bias = _dyadic((N,), g, 11, -5)
    return A, W, bias


def _gemm_ref64(A, W, bias, pos=None, temb=None, temb_stride=0, L=1):
    """float64 on the GPU: every operand is dyadic and every sum exact, so the order does not matter."""
    y = A.double() @ W.double().T + bias.double()
    if pos is not None:
        M, N = y.shape
        B = M // L
        t = temb.double()[:B] if temb_stride else temb.double()[:1].expand(B, N)
        y = (y.view(B, L, N) + pos.double()[None] + t[:, None]).view(M, N)
    return y


def _assert_gemm_exact(out, ref64, what, rows_per_chunk=1 << 15):
    """fp32 output bit-identical to float64; bf16 output exactly RNE(ref).  The reference must itself be exact in fp32
    (checked), which is what makes the fp32 comparison an identity test rather than a tolerance."""
    for r0 in range(0, ref64.shape[0], rows_per_chunk):
        ref_c = ref64[r0:r0 + rows_per_chunk]
        assert torch.equal(ref_c.float().double(), ref_c), "%s: reference not exact in fp32 (test construction)" % what
        if out.dtype == F32:
            bad = out[r0:r0 + rows_per_chunk].double() != ref_c
            if bool(bad.any()):
                i = int(bad.flatten().nonzero()[0])
                raise AssertionError("%s: %d fp32 elements differ from float64; first at (row, col) = (%d, %d): %r vs %r"
                                     % (what, int(bad.sum()), r0 + i // ref_c.shape[1], i % ref_c.shape[1],
                                        float(out[r0:r0 + rows_per_chunk].flatten()[i]), float(ref_c.flatten()[i])))
        else:
            assert_rounded(out[r0:r0 + rows_per_chunk], ref_c.cpu(), 0, "%s rows %d.." % (what, r0))


def _run_linear(A, W, bias, epi, out_dtype, out_cols=None, **kw):
    M, N = A.shape[0], W.shape[0]
    cols = (2 * N if epi == _lib.EPI_BIAS_SPLIT else N) if out_cols is None else out_cols
    buf, view, front, n = _guarded((M, cols), out_dtype)
    ops.linear(A, W, bias, epi, out=view, **kw)
    torch.cuda.synchronize()
    _check_guard(buf, front, n, "linear M=%d N=%d epi=%d" % (M, N, epi))
    return view


# (id, M, N, K, out dtype, out_cols or None, launch path per gemm_path)
GEMM_CASES = [
    # pair kernel: M = 1024 / 1025, 2096 x 2 (the second CTA of the last pair has no rows), 2096 x 3 (144-row tail)
    ("pair-M1024", 1024, 768, 768, BF16, None, "pair"),
    ("pair-M1025", 1025, 768, 768, BF16, None, "pair"),
    ("pair-M4192", 4192, 768, 768, BF16, None, "pair"),           # production out-proj and down1 shape (768, 768)
    ("pair-M6288", 6288, 768, 768, BF16, None, "pair"),
    ("pair-qkv", 4192, 2304, 768, BF16, None, "pair"),
    ("pair-ffn1", 4192, 3072, 768, BF16, None, "pair"),
    ("pair-ffn2", 4192, 768, 3072, BF16, None, "pair"),           # K >= 2048: sleeping epilogue waits
    ("pair-up1", 4192, 768, 128, BF16, None, "pair"),
    ("pair-K8", 1100, 768, 8, BF16, None, "pair"),
    ("pair-K136", 2096, 2304, 136, BF16, None, "pair"),
    ("pair-cols504", 2000, 768, 768, BF16, 504, "pair"),          # TMA store clips columns >= out_cols
    # single-CTA BN = 256: N % 256 == 0 with M < 1024 or fp32 output, or N > 512 not a multiple of 256
    ("bn256-M600", 600, 768, 768, BF16, None, "bn256"),
    ("bn256-M1023", 1023, 768, 768, BF16, None, "bn256"),
    ("bn256-f32", 2096, 768, 768, F32, None, "bn256"),
    ("bn256-f32-ffn2", 1100, 768, 3072, F32, None, "bn256"),
    ("bn256-N776", 300, 776, 768, BF16, None, "bn256"),
    ("bn256-N776-f32", 1100, 776, 136, F32, None, "bn256"),
    ("bn256-M1", 1, 768, 768, BF16, None, "bn256"),
    # single-CTA BN = 128
    ("bn128-N128-f32", 2096, 128, 768, F32, None, "bn128"),
    ("bn128-N200", 77, 200, 72, BF16, None, "bn128"),
    ("bn128-N384", 1500, 384, 256, BF16, None, "bn128"),
    ("bn128-M127", 127, 384, 768, BF16, None, "bn128"),
    ("bn128-M129-f32", 129, 384, 768, F32, None, "bn128"),
    ("bn128-K72-f32", 300, 200, 72, F32, None, "bn128"),
    ("bn128-D100-f32", 2096, 128, 768, F32, 100, "bn128"),        # D = 100 in a Dp = 128 GEMM
    ("bn128-cols96", 300, 128, 768, BF16, 96, "bn128"),
]


@pytest.mark.parametrize("case", [pytest.param(c, id=c[0]) for c in GEMM_CASES])
def test_gemm_exact(case):
    name, M, N, K, dt, out_cols, path = case
    assert gemm_path(M, N, dt == F32) == path
    A, W, bias = _gemm_operands(M, N, K, seed=M * 31 + N * 7 + K)
    ref = _gemm_ref64(A, W, bias)
    if out_cols is not None:
        ref = ref[:, :out_cols]
    out = _run_linear(A, W, bias, _lib.EPI_BIAS, dt, out_cols)
    _assert_gemm_exact(out, ref, name)


def test_gemm_exact_production_pass():
    """QKV at the production pass size M = 256 x 2096 (pair kernel, 4192 x 9 tiles over 74 pairs)."""
    M, N, K = 256 * 2096, 2304, 768
    assert gemm_path(M, N, False) == "pair"
    A, W, bias = _gemm_operands(M, N, K, seed=11)
    out = _run_linear(A, W, bias, _lib.EPI_BIAS, BF16)
    ref = _gemm_ref64(A, W, bias)
    del A
    _assert_gemm_exact(out, ref, "qkv M=536576")


# (L, B, N, K, out dtype, path): M = B * L
POS_TIME_CASES = [
    (64, 16, 768, 768, BF16, "pair"),
    (256, 4, 768, 768, BF16, "pair"),
    (2096, 2, 768, 768, BF16, "pair"),        # production: up-projection's second Linear
    (64, 3, 768, 768, BF16, "bn256"),
    (256, 5, 768, 128, F32, "bn256"),
    (2096, 1, 768, 768, F32, "bn256"),
    (64, 5, 384, 72, BF16, "bn128"),
    (256, 3, 128, 768, BF16, "bn128"),
    (2096, 1, 200, 136, F32, "bn128"),
]


@pytest.mark.parametrize("temb_stride_n", [False, True], ids=["temb_shared", "temb_per_seq"])
@pytest.mark.parametrize("case", [pytest.param(c, id="%s-L%d-B%d-N%d-K%d-%s" % (c[5], c[0], c[1], c[2], c[3], "f32" if c[4] == F32 else "bf16"))
                                  for c in POS_TIME_CASES])
def test_gemm_pos_time_exact(case, temb_stride_n):
    """MD_EPI_BIAS_POS_TIME: out[b*L + l] = A W^T + bias + pos[l] + temb[b] (temb_stride 0: temb[0] for every b).  pos and
    temb rows are all distinct, so a row mapped to the wrong (seq_b, seq_l) — in the pair kernel the row also depends on
    the CTA's rank — changes the output exactly."""
    L, B, N, K, dt, path = case
    M = B * L
    assert gemm_path(M, N, dt == F32) == path
    A, W, bias = _gemm_operands(M, N, K, seed=L * 13 + B + N + K + temb_stride_n)
    g = _gen(L + N)
    pos = _dyadic((L, N), g, 11, -6)
    temb = _dyadic((B, N), g, 11, -6)
    assert torch.unique(pos, dim=0).shape[0] == L and torch.unique(temb, dim=0).shape[0] == B
    stride = N if temb_stride_n else 0
    out = _run_linear(A, W, bias, _lib.EPI_BIAS_POS_TIME, dt, pos=pos, temb=temb, temb_stride=stride, L=L)
    _assert_gemm_exact(out, _gemm_ref64(A, W, bias, pos, temb, stride, L), "pos_time L=%d B=%d N=%d" % (L, B, N))


@pytest.mark.parametrize("M,N,K", [(4192, 128, 768), (77, 256, 72), (1023, 384, 136)])
def test_gemm_split_exact(M, N, K):
    """MD_EPI_BIAS_SPLIT writes [hi | lo] with hi = RNE(y), lo = RNE(y - hi); y carries more bits than bf16, so lo != 0."""
    A, W, bias = _gemm_operands(M, N, K, seed=M + N + K)
    out = _run_linear(A, W, bias, _lib.EPI_BIAS_SPLIT, BF16)
    y = _gemm_ref64(A, W, bias).cpu()
    hi = _rne(y, BF16).double()
    assert bool((y != hi).any())
    assert_rounded(out[:, :N], y, 0, "split hi")
    assert_rounded(out[:, N:], y - hi, 0, "split lo")


# ------------------------------------------------------------------------------------------------ B. epilogue functions
GELU_ABS = 3.5e-6                   # the stated bound of gelu_erf_x2 (common.cuh)
TANH_REL = 2.0 ** -10.987           # PTX ISA, tanh.approx.f32: maximum relative error 2^-10.987 over the full range
FTZ_FLOOR = 2.0 ** -126             # subnormal pre-activations may be flushed


def _bf16_sweep(lim):
    """every finite bf16 value in [-lim, lim] (zero once), as float64"""
    allv = torch.arange(-(1 << 15), 1 << 15, dtype=torch.int32).to(torch.int16).view(BF16).double()
    v = allv[torch.isfinite(allv) & (allv.abs() <= lim)]
    return torch.unique(v)


def _epilogue_operands(M, N, K, seed):
    """A: one-hot rows (row r has 1 at column r mod K), so z[r, n] = W[n, r mod K] + bias[n] — one fp32 add, the same one
    the epilogue makes.  Columns n < N/2 have bias 0 and their W entries hold every bf16 value in [-12, 12]; columns
    n >= N/2 hold random bf16 values in [-12, 12] plus a full-precision fp32 bias in (-1/2, 1/2), which puts z between
    the bf16 values."""
    g = torch.Generator().manual_seed(seed)
    sweep = _bf16_sweep(12.0)
    half = N // 2
    assert half * K >= sweep.numel()
    W = ((torch.rand(N, K, generator=g, dtype=torch.float64) * 24 - 12)).to(BF16).double()
    w0 = W[:half].reshape(-1).clone()
    w0[:sweep.numel()] = sweep
    W[:half] = w0[torch.randperm(w0.numel(), generator=g)].view(half, K)
    bias = torch.zeros(N, dtype=F32)
    bias[half:] = torch.rand(N - half, generator=g) - 0.5
    A = torch.zeros(M, K, dtype=BF16)
    A[torch.arange(M), torch.arange(M) % K] = 1.0
    z32 = (W.to(F32)[:, torch.arange(M) % K].T + bias[None, :])        # the epilogue's fp32 add, in numpy-equal IEEE fp32
    return A.to(DEV), W.to(BF16).to(DEV), bias.to(DEV), z32.double().numpy()


def _gelu64(z):
    from scipy.special import ndtr
    return z * ndtr(z)


EPI_CASES = [   # (M, N, K, out dtype, path)
    (1056, 256, 264, BF16, "pair"),
    (792, 256, 264, BF16, "bn256"),
    (1056, 256, 264, F32, "bn256"),
    (1056, 384, 176, F32, "bn128"),
]


@pytest.mark.parametrize("case", [pytest.param(c, id="%s-%s" % (c[4], "f32" if c[3] == F32 else "bf16")) for c in EPI_CASES])
def test_epilogue_gelu(case):
    """erf-GELU (gelu_erf_x2) over every bf16 z in [-12, 12] and fp32 z between them.  fp32 output: |y - gelu64(z)| <=
    3.5e-6 + 2^-22 |gelu64(z)| (the stated polynomial bound plus a few fp32 roundings of the result).  bf16 output:
    assert_rounded with delta 3.5e-6 + 2^-22 |gelu64(z)|."""
    M, N, K, dt, path = case
    assert gemm_path(M, N, dt == F32) == path
    A, W, bias, z = _epilogue_operands(M, N, K, seed=M + N)
    out = _run_linear(A, W, bias, _lib.EPI_BIAS_GELU, dt)
    ref = _gelu64(z)
    tol = GELU_ABS + 2.0 ** -22 * np.abs(ref)
    if dt == F32:
        err = np.abs(out.double().cpu().numpy() - ref)
        worst = np.unravel_index(int(np.argmax(err - tol)), err.shape)
        _report("gelu_f32_%s" % path, max_abs_err=float(err.max()), at_z=float(z[worst]))
        assert (err <= tol).all(), ("GELU error %.3g at z = %r (bound %.3g); %d elements over the bound"
                                    % (err[worst], z[worst], tol[worst], int((err > tol).sum())))
    else:
        n, frac = assert_rounded(out, ref, tol, "gelu bf16 %s" % path)
        _report("gelu_bf16_%s" % path, other_neighbour=n, max_frac_of_delta=frac)


@pytest.mark.parametrize("case", [pytest.param(c, id="%s-%s" % (c[4], "f32" if c[3] == F32 else "bf16")) for c in EPI_CASES])
def test_epilogue_tanh(case):
    """tanh.approx.f32 over the same z: |y - tanh64(z)| <= 2^-10.987 |tanh64(z)| (PTX ISA bound) + 2^-126 (a subnormal z
    may be flushed to zero).  bf16 output: assert_rounded with that delta."""
    M, N, K, dt, path = case
    assert gemm_path(M, N, dt == F32) == path
    A, W, bias, z = _epilogue_operands(M, N, K, seed=M + N + 1)
    out = _run_linear(A, W, bias, _lib.EPI_BIAS_TANH, dt)
    ref = np.tanh(z)
    tol = TANH_REL * np.abs(ref) + FTZ_FLOOR
    if dt == F32:
        y = out.double().cpu().numpy()
        err = np.abs(y - ref)
        nz = np.abs(ref) > 2.0 ** -100
        rel = (err[nz] / np.abs(ref[nz]))
        worst = np.unravel_index(int(np.argmax(err - tol)), err.shape)
        _report("tanh_f32_%s" % path, max_rel_err=float(rel.max()), max_rel_err_log2=float(np.log2(rel.max())))
        assert (err <= tol).all(), ("tanh error %.3g at z = %r (bound %.3g); %d elements over the bound"
                                    % (err[worst], z[worst], tol[worst], int((err > tol).sum())))
    else:
        n, frac = assert_rounded(out, ref, tol, "tanh bf16 %s" % path)
        _report("tanh_bf16_%s" % path, other_neighbour=n, max_frac_of_delta=frac)


# ------------------------------------------------------------------------------------------------ C. attention
# L selects the work-item kinds and tail paths (see tests/test_kernels_gpu.py::test_attention): 64 / 128 SINGLE,
# 130 / 200 / 256 PAIR, 300 / 320 / 385 PAIR + SPLIT with a half-width tail, 2048 PAIR without a tail, 2096 the base shape,
# 2176 SPLIT with a full tail, 4192 SPLIT with a masked full-width tail; B = 24 x 12 heads at 2096: ~18 items per CTA.
ATT_SHAPES = [(1, 64, 2), (2, 128, 12), (2, 130, 3), (2, 200, 12), (1, 256, 3), (3, 300, 4), (2, 320, 2), (2, 385, 5),
              (2, 2048, 3), (2, 2096, 12), (1, 2176, 4), (1, 4192, 2), (24, 2096, 12)]
ATT_IDS = ["B%d-L%d-NH%d" % s for s in ATT_SHAPES]


def _att_poly():
    return int(os.environ.get("MD_ATT_POLY", "0"))


def _codes(n):
    """+-1 code of the 13 bits of j, [n, 13]"""
    j = torch.arange(n)
    return ((j[:, None] >> torch.arange(13)) & 1).float() * 2 - 1


def _qkv(q, k, v):
    """[B, L, NH, 64] each -> the kernel's [B*L, 3*NH*64] bf16 layout"""
    B, L, NH, _ = q.shape
    return torch.stack([q, k, v], dim=2).reshape(B * L, 3 * NH * 64).to(BF16).to(DEV)


@pytest.mark.parametrize("B,L,NH", ATT_SHAPES, ids=ATT_IDS)
def test_attention_routing_exact(B, L, NH):
    """Key j carries the +-1 code of its 13 bits in head dims 0-12; query i is 128 x code(pi(i)) for a random permutation pi
    of each (b, h).  The winning score is 128 x 13 = 1664, every other score <= 1408: after the log2e scale a gap of 369,
    so every other weight is exactly 0 (ex2.approx.ftz underflows; the clamped polynomial variants give 2^-125, far below
    an fp32 ulp of the winner's contribution), also across a lazy rescale and the SPLIT merge.  The winner's weight is
    2^r with |r| < 2^-13 (the fma residual of s log2e - m), which rounds to bf16 1.0, and the output V / (2^r) rounds back
    to V.  So out[b, i, h] must equal V[b, pi(i), h] bit for bit."""
    g = torch.Generator().manual_seed(B * 100003 + L * 7 + NH)
    code = _codes(L)
    perm = torch.argsort(torch.rand(B, NH, L, generator=g), dim=-1)           # [B, NH, L]
    q = torch.zeros(B, L, NH, 64)
    q[..., :13] = 128.0 * code[perm].permute(0, 2, 1, 3)
    k = torch.zeros(B, L, NH, 64)
    k[..., :13] = code[None, :, None, :]
    v = torch.randn(B, L, NH, 64, generator=g).to(BF16).float()
    out = ops.attention(_qkv(q, k, v), B, L, NH).cpu().view(B, L, NH, 64)
    want = torch.gather(v, 1, perm.permute(0, 2, 1)[..., None].expand(B, L, NH, 64)).to(BF16)
    bad = out.view(torch.int16) != want.view(torch.int16)
    if bool(bad.any()):
        b, i, h, d = [int(t) for t in bad.nonzero()[0]]
        raise AssertionError("routing: %d of %d elements differ; first at (b, row, head, dim) = (%d, %d, %d, %d): %r, want %r"
                             % (int(bad.sum()), bad.numel(), b, i, h, d, float(out[b, i, h, d]), float(want[b, i, h, d])))


@pytest.mark.parametrize("B,L,NH", ATT_SHAPES, ids=ATT_IDS)
def test_attention_masking_exact(B, L, NH):
    """All keys carry the same code and q = -code, so every real score is -13 and every weight equal; a padded key past L
    (read as zeros by TMA) would score 0 and weigh 2^18.75 times more.  V holds integers in [-8, 8], so O = sum(v) is exact
    and out = RNE(sum(v) / L) up to the fp32 sum of L equal weights and one division: delta = 2^-18 |sum(v) / L|.
    The polynomial exponential (MD_ATT_POLY >= 1) evaluates 2^0 as 0.99993: those weights round to bf16 1.0 in P but enter
    the fp32 row sum as they are, which scales the output by up to 1 + 7.6e-5 < 1 + 2^-13; delta adds 2^-13 |sum(v) / L|."""
    g = torch.Generator().manual_seed(B * 7919 + L + NH)
    c = _codes(1)[0]
    q = torch.zeros(B, L, NH, 64)
    q[..., :13] = -c
    k = torch.zeros(B, L, NH, 64)
    k[..., :13] = c
    v = torch.randint(-8, 9, (B, L, NH, 64), generator=g).float()
    out = ops.attention(_qkv(q, k, v), B, L, NH).cpu().view(B, L, NH, 64)
    mean = (v.double().sum(1, keepdim=True) / L).expand(B, L, NH, 64)
    rel = 2.0 ** -18 + (2.0 ** -13 if _att_poly() else 0.0)
    assert_rounded(out.reshape(B * L, NH * 64), mean.reshape(B * L, NH * 64), rel * mean.abs().reshape(B * L, NH * 64),
                   "masking B=%d L=%d NH=%d" % (B, L, NH))


ATT_RANDOM = [(1, 64, 2), (2, 200, 12), (3, 300, 4), (2, 385, 5), (1, 2176, 4), (2, 2096, 12), (1, 4192, 2)]


@pytest.mark.parametrize("scale", [(0.5, 1.5), (0.25, 0.25)], ids=["peaky", "high_entropy"])
@pytest.mark.parametrize("B,L,NH", ATT_RANDOM, ids=["B%d-L%d-NH%d" % s for s in ATT_RANDOM])
def test_attention_random_bound(B, L, NH, scale):
    """Random q, k, v (score std ~6 'peaky' as in test_kernels_gpu.py, or ~0.5 'high entropy').  With float64 weights
    p_j = exp(s_j - max s), O = sum p_j v_j / sum p_j and A = sum p_j |v_j| / sum p_j:

        |out - O| <= 2^-8 (A + |O|) (1 + 1/16)   [+ 2^-13 A for the polynomial exponential, MD_ATT_POLY >= 1]

    Derivation.  bf16 has 8 significant bits, so one RNE moves a value by at most 2^-8 of its magnitude (half an ulp of
    2^-7 at the bottom of a binade).  (1) The kernel multiplies V by P rounded to bf16 but divides by the fp32 row sum
    l_sum of the unrounded p (attention.cu, softmax_block): sum_j |p_j - bf16(p_j)| |v_j| / sum p_j <= 2^-8 A.  (2) The
    output rounding adds at most 2^-8 |O_kernel|.  Everything else — fp32 scores (64 exact bf16 products per dot),
    ex2.approx (relative error ~2^-22), the fp32 P V accumulation, the lazy rescale and SPLIT merge multiplies and the
    1 / l_sum — is below 2^-16 relative, which the factor 1 + 1/16 covers with room.  The polynomial 2^x has relative
    error 7.6e-5 < 2^-13 on every weight.  The measured maximum of |out - O| / (2^-9 (A + |O|)) is reported."""
    g = torch.Generator().manual_seed(B * 1000 + L + NH + int(scale[0] * 8))
    H = NH * 64
    qkv = torch.randn(B * L, 3 * H, generator=g)
    qkv[:, :H] *= scale[0]
    qkv[:, H:2 * H] *= scale[1]
    qkv = qkv.to(BF16)
    out = ops.attention(qkv.to(DEV), B, L, NH).cpu().double().view(B, L, NH, 64).numpy()
    x = qkv.double().view(B, L, 3, NH, 64).numpy()
    worst, worst9 = 0.0, 0.0
    for b in range(B):
        for h in range(NH):
            q, k, v = x[b, :, 0, h], x[b, :, 1, h], x[b, :, 2, h]
            s = q @ k.T
            p = np.exp(s - s.max(axis=1, keepdims=True))
            den = p.sum(axis=1, keepdims=True)
            O = (p @ v) / den
            Aa = (p @ np.abs(v)) / den
            err = np.abs(out[b, :, h] - O)
            bound = 2.0 ** -8 * (Aa + np.abs(O)) * (1 + 1 / 16) + (2.0 ** -13 * Aa if _att_poly() else 0.0)
            r = err / bound
            if r.max() > 1:
                i, d = np.unravel_index(int(np.argmax(r)), r.shape)
                raise AssertionError("attention b=%d h=%d row %d dim %d: |out - O| = %.4g > bound %.4g (O = %.6g, A = %.4g); %d elements "
                                     "over" % (b, h, i, d, err[i, d], bound[i, d], O[i, d], Aa[i, d], int((r > 1).sum())))
            worst = max(worst, float(r.max()))
            worst9 = max(worst9, float((err / (2.0 ** -9 * (Aa + np.abs(O)))).max()))
    _report("attention_random_B%d_L%d_NH%d_%s" % (B, L, NH, "peaky" if scale[0] == 0.5 else "flat"), max_err_over_bound=worst,
            max_err_over_2m9=worst9)


# ------------------------------------------------------------------------------------------------ D. LayerNorm
LN_WIDTHS = [256 * k for k in range(1, 9)]


def _ln_reference(x, r, gamma, beta, eps):
    """float64 LN(x + r) and the per-element delta of the kernel's fp32 evaluation (elementwise.cu, layernorm_kernel).

    The kernel: v = fl(x + r); s = sum v (per lane a sequential sum of H/32 values, then 5 butterfly levels: n = H/32 + 5
    rounded adds in any chain); mean = s / H (one rounding); q = sum fma(v - mean, v - mean, .) (same chain length);
    rstd = rsqrtf(q * (1/H) + eps); y = fma((v - mean) * rstd, gamma, beta).  With u = 2^-24, to first order:
      e_v  = u |v| where x + r is inexact in fp32 (0 without r);
      e_s  = n u sum|v|, or 0 when every v is a multiple of 2^g with sum|x| + sum|r| < 2^(24+g) (then every partial
             sum is exact: the constant and large-offset rows);
      e_mu = (e_s + sum e_v) / H + 2u |mu|;
      eps_q = (n + 3) u + 2 rms(e_v) rstd + ((e_mu + max e_v) rstd)^2           (relative error of q)
      eps_r = eps_q / 2 + 5u                                  (q/H, + eps, rsqrtf's 2 ulp: relative error of rstd)
      |d xhat| <= |xhat| (eps_r + 2u) + (e_mu + e_v) rstd
      |d y|    <= |gamma| |d xhat| + u (|gamma xhat| + |beta|)
    delta = 2 |d y| (the factor 2 covers the second-order terms).  Returns (y64, delta, gamma*xhat)."""
    H = x.shape[-1]
    u = U32
    n = H // 32 + 5
    v = x + (r if r is not None else 0.0)
    mu = v.mean(axis=1, keepdims=True)
    var = ((v - mu) ** 2).mean(axis=1, keepdims=True)
    eps64 = float(np.float32(eps))
    rstd = 1.0 / np.sqrt(var + eps64)
    xhat = (v - mu) * rstd
    gx = gamma[None, :] * xhat
    y = gx + beta[None, :]
    # grid exponent of every operand: a bf16 value with exponent e is a multiple of 2^(e - 7)
    parts = [x] if r is None else [x, r]
    g = np.full((x.shape[0], 1), np.inf)
    tot = np.zeros((x.shape[0], 1))
    for t in parts:
        nz = t != 0
        e = np.where(nz, np.floor(np.log2(np.where(nz, np.abs(t), 1.0))) - 7, np.inf)
        g = np.minimum(g, e.min(axis=1, keepdims=True))
        tot += np.abs(t).sum(axis=1, keepdims=True)
    exact = tot < 2.0 ** (24 + np.where(np.isinf(g), 0, g))
    e_v = np.zeros_like(v) if (r is None) else np.where(exact, 0.0, u * np.abs(v))
    e_s = np.where(exact, 0.0, n * u * np.abs(v).sum(axis=1, keepdims=True))
    e_mu = (e_s + e_v.sum(axis=1, keepdims=True)) / H + 2 * u * np.abs(mu)
    rms_ev = np.sqrt((e_v ** 2).mean(axis=1, keepdims=True))
    eps_q = (n + 3) * u + 2 * rms_ev * rstd + ((e_mu + e_v.max(axis=1, keepdims=True)) * rstd) ** 2
    eps_r = eps_q / 2 + 5 * u
    dxhat = np.abs(xhat) * (eps_r + 2 * u) + (e_mu + e_v) * rstd
    delta = 2 * (np.abs(gamma)[None, :] * dxhat + u * (np.abs(gx) + np.abs(beta)[None, :]))
    return y, delta, gx


def _ln_params(H, seed):
    """gamma ~ 1 + 0.1 N(0, 1); beta = +-[1/4, 1) in bf16.  beta is kept away from 0 so that delta, which has a term
    independent of xhat (the rounding of the mean), stays within 2^-12 (|gamma xhat| + |beta|) for elements with xhat ~ 0."""
    g = torch.Generator().manual_seed(seed)
    gamma = (1 + 0.1 * torch.randn(H, generator=g)).float()
    sign = torch.where(torch.rand(H, generator=g) < 0.5, -1.0, 1.0)
    beta = (sign * (0.25 + 0.75 * torch.rand(H, generator=g))).to(BF16).float()
    return gamma, beta


def _check_ln(x, r, gamma, beta, eps, what):
    """run the kernel on bf16 x (and r) and assert_rounded against the float64 reference; delta must stay within
    2^-12 (|gamma xhat| + |beta|), at least 8x tighter than bf16's half ulp."""
    out = ops.layernorm(x.to(DEV), gamma.to(DEV), beta.to(DEV), eps, resid=None if r is None else r.to(DEV)).cpu()
    x64 = x.double().numpy()
    r64 = None if r is None else r.double().numpy()
    g64, b64 = gamma.double().numpy(), beta.double().numpy()
    y, delta, gx = _ln_reference(x64, r64, g64, b64, eps)
    cap = 2.0 ** -12 * (np.abs(gx) + np.abs(b64)[None, :])
    assert (delta <= cap).all(), "%s: derived delta exceeds 2^-12 (|gamma xhat| + |beta|) (test construction)" % what
    n, frac = assert_rounded(out, y, delta, what)
    return n, frac


@pytest.mark.parametrize("M", [1, 7, 333, 4192])
@pytest.mark.parametrize("H", LN_WIDTHS)
def test_layernorm_rows(H, M):
    g = torch.Generator().manual_seed(H * 7 + M)
    gamma, beta = _ln_params(H, H + M)
    x = (torch.randn(M, H, generator=g) * 2 + 0.3).to(BF16)
    r = torch.randn(M, H, generator=g).to(BF16)
    n0, f0 = _check_ln(x, None, gamma, beta, 1e-12, "layernorm H=%d M=%d" % (H, M))
    n1, f1 = _check_ln(x, r, gamma, beta, 1e-12, "layernorm+resid H=%d M=%d" % (H, M))
    _report("layernorm_H%d_M%d" % (H, M), other_neighbour=n0 + n1, max_frac_of_delta=max(f0, f1))


@pytest.mark.parametrize("H", LN_WIDTHS)
def test_layernorm_eps(H):
    """eps = 1e-5 on rows with a small variance (eps matters) and ordinary rows"""
    g = torch.Generator().manual_seed(H + 5)
    gamma, beta = _ln_params(H, H)
    x = torch.randn(64, H, generator=g)
    x[:32] *= 0.004
    x = x.to(BF16)
    for eps in (1e-5, 1e-12):
        _check_ln(x, None, gamma, beta, eps, "layernorm eps=%g H=%d" % (eps, H))


def test_layernorm_production_pass():
    """LN(dense(ctx) + h) at the production pass size: 256 x 2096 rows of H = 768, in chunks of rows for the reference."""
    H, M = 768, 256 * 2096
    g = torch.Generator(device=DEV).manual_seed(3)
    x = (torch.randn(M, H, generator=g, device=DEV) * 2 + 0.3).to(BF16)
    r = torch.randn(M, H, generator=g, device=DEV).to(BF16)
    gamma, beta = _ln_params(H, 17)
    out = ops.layernorm(x, gamma.to(DEV), beta.to(DEV), 1e-12, resid=r).cpu()
    x, r = x.cpu(), r.cpu()
    g64, b64 = gamma.double().numpy(), beta.double().numpy()
    worst = 0.0
    step = 1 << 16
    for r0 in range(0, M, step):
        y, delta, _ = _ln_reference(x[r0:r0 + step].double().numpy(), r[r0:r0 + step].double().numpy(), g64, b64, 1e-12)
        worst = max(worst, assert_rounded(out[r0:r0 + step], y, delta, "layernorm production rows %d.." % r0)[1])
    _report("layernorm_production", max_frac_of_delta=worst)


def _const_sweep():
    """every normal bf16 value c with 2^-60 < |c| < 2^60, and 0"""
    v = _bf16_sweep(2.0 ** 60)
    return torch.cat([v[(v.abs() > 2.0 ** -60) & (v.abs() < 2.0 ** 60)], torch.zeros(1, dtype=torch.float64)])


@pytest.mark.parametrize("H", LN_WIDTHS)
def test_layernorm_constant_rows(H):
    """A constant row c has mean c and variance 0, so the output is exactly beta for every c (beta is bf16 here).  The
    kernel's sum H c is exact; the mean must then come back as exactly c — for H = 1792, fl(H c) * fl(1/H) != c for most
    c, which made dlt = +-1 ulp and rstd ~ 1/ulp, i.e. beta +- gamma x O(1)."""
    c = _const_sweep()
    gamma, beta = _ln_params(H, 99)
    x = c[:, None].expand(c.numel(), H).to(BF16).contiguous()
    want = beta.to(BF16)[None, :].expand(c.numel(), H)
    for eps in (1e-12, 1e-5):
        for r in (None, torch.zeros_like(x)):
            out = ops.layernorm(x.to(DEV), gamma.to(DEV), beta.to(DEV), eps, resid=None if r is None else r.to(DEV)).cpu()
            bad = (out.view(torch.int16) != want.view(torch.int16)).any(dim=1)
            assert not bool(bad.any()), ("H=%d eps=%g resid=%s: %d of %d constant rows do not give beta, e.g. c = %r -> max |out - beta| = %.4g"
                                         % (H, eps, r is not None, int(bad.sum()), c.numel(), float(c[bad][0]),
                                            float((out[bad][0].float() - want[0].float()).abs().max())))


@pytest.mark.parametrize("H", LN_WIDTHS)
def test_layernorm_large_offset_rows(H):
    """x = c + k 2^13 with c = 2^20 (and other offsets), k in {-2..2}: var / mean^2 ~ 2^-13, where a one-pass E[x^2] - mean^2
    in fp32 (relative error ~2^-24 H of 2^40) loses the variance; the two-pass statistics are exact here."""
    g = torch.Generator().manual_seed(H + 1)
    gamma, beta = _ln_params(H, H + 2)
    rows = []
    for c, step in ((2.0 ** 20, 2.0 ** 13), (-3 * 2.0 ** 18, 2.0 ** 12), (2.0 ** 7, 2.0 ** 0), (1.5 * 2.0 ** -10, 2.0 ** -17)):
        k = torch.randint(-2, 3, (8, H), generator=g).double()
        rows.append(c + k * step)
    x = torch.cat(rows).to(BF16)
    assert torch.equal(x.double(), torch.cat(rows))
    _check_ln(x, None, gamma, beta, 1e-12, "layernorm large offset H=%d" % H)
    _check_ln(x, torch.zeros_like(x), gamma, beta, 1e-12, "layernorm large offset + zero resid H=%d" % H)


# ------------------------------------------------------------------------------------------------ E. kernel variants
# Each switch is read once per process by the library, so each variant runs the structured cases of this file in a child
# process.  MD_ATT_POLY=9 is a timing experiment that computes no exponential at all; it is not a kernel and is excluded.
VARIANTS = [
    ("MD_GEMM_PAIR", "0", "test_gemm_exact or test_gemm_pos_time or test_gemm_split or test_epilogue"),
    ("MD_ATT_POLY", "1", "test_attention"),
    ("MD_ATT_POLY", "2", "test_attention"),
    ("MD_ATT_POLY", "3", "test_attention"),
    ("MD_ATT_POLY", "4", "test_attention"),
    ("MD_LN_HOIST", "0", "test_layernorm_rows or test_layernorm_eps or test_layernorm_constant or test_layernorm_large"),
]


@pytest.mark.skipif(os.environ.get(VARIANT_GUARD) == "1", reason="already inside a variant child process")
@pytest.mark.parametrize("var,value,select", VARIANTS, ids=["%s=%s" % v[:2] for v in VARIANTS])
def test_kernel_variant(var, value, select):
    env = dict(os.environ)
    env[var] = value
    env[VARIANT_GUARD] = "1"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [
        "-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-p", "no:cacheprovider", "-x", "-k",
        "(%s) and not production and not B24" % select]
    try:
        res = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    except subprocess.TimeoutExpired as e:       # subprocess.run has killed the child
        raise AssertionError("%s=%s: child pytest exceeded %d s" % (var, value, e.timeout))
    tail = "\n".join(res.stdout.splitlines()[-40:])
    assert res.returncode == 0, "%s=%s: child pytest failed (exit %d):\n%s" % (var, value, res.returncode, tail)
    assert " passed" in tail and " failed" not in tail, tail
