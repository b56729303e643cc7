"""Tensor-level wrappers over the custom ops `torch.ops.musediff.*` (custom_ops.py: one op per `md_*` kernel entry of
include/musediff_b200.h, CUDA dispatch key only).  The wrappers allocate outputs, check dtype / layout / device and
then dispatch; every op launches hand-written sm_100a kernels on the current CUDA stream.  Inputs must be CUDA tensors
(a CPU tensor raises — there is no fallback)."""
import numpy as np
import torch

from . import _lib, custom_ops
from .custom_ops import _s64

BF16 = torch.bfloat16
K = custom_ops.ops          # torch.ops.musediff

_LAUNCHES = custom_ops._LAUNCHES
_PROFILE = custom_ops._PROFILE      # list of (name, detail, start_event, end_event) while profile_step() is active


def launch_count():
    return _LAUNCHES[0]


def add_launches(n):
    """kernels launched by a CUDA-graph replay (they do not pass through the op layer)."""
    _LAUNCHES[0] += int(n)


def profile_step(fn):
    """run fn() with CUDA events around every kernel launch; returns [(kernel, detail, ms)]."""
    _PROFILE[0] = []
    try:
        fn()
        torch.cuda.synchronize()
        return [(n, d, e0.elapsed_time(e1)) for n, d, e0, e1 in _PROFILE[0]]
    finally:
        _PROFILE[0] = None


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _cu(*tensors):
    """every tensor handed to an op lives on a CUDA device (the ops have no other backend)."""
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise _lib.MuseDiffLibraryError("musediffusion_b200 ops need CUDA tensors (got a %s tensor)" % t.device)


def _c(t, dtype=None):
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t if t.is_contiguous() else t.contiguous()


# ------------------------------------------------------------------------------------------------ schedule
TABLE_ORDER = ["posterior_mean_coef1", "posterior_mean_coef2", "model_log_variance", "sqrt_recip_alphas_cumprod",
               "sqrt_recipm1_alphas_cumprod", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_alphas_cumprod",
               "sqrt_one_minus_alphas_cumprod"]
_current_schedule_key = {}      # CUDA device index -> key of the schedule resident in that device's tables


def current_schedule_key():
    return _current_schedule_key.get(torch.cuda.current_device())


def set_schedule(tables64, key=None):
    """tables64: dict name -> float64 numpy [T].  Cast to fp32 exactly like _extract_into_tensor
    (MuseDiffusion/models/diffusion.py:914) and uploaded once; `key` lets callers skip redundant uploads."""
    if key is not None and current_schedule_key() is key:
        return
    T = len(tables64[TABLE_ORDER[0]])
    host = np.ascontiguousarray(np.stack([np.asarray(tables64[n], dtype=np.float64).astype(np.float32)
                                          for n in TABLE_ORDER]))
    _lib.call("md_set_schedule", host.ctypes.data, T, _stream())      # host -> device table copy, not a kernel op
    _current_schedule_key[torch.cuda.current_device()] = key


def padded_width(D):
    """Dp: the width of the bf16 tensor-core operands that stand for a D-wide state or embedding (the first Linear's A
    operand, the [hi | lo] rounding operands, W_up1's columns, W_dn2's rows).  D rounded up to a multiple of 64; the
    columns D..Dp-1 hold zeros, which leaves every contraction unchanged."""
    return -(-int(D) // 64) * 64


# ------------------------------------------------------------------------------------------------ elementwise
def cast_bf16(x, width=None):
    """fp32 [..., D] -> bf16 [..., width] (width defaults to D; columns D..width-1 are zero)."""
    x = _c(x, torch.float32)
    D = x.shape[-1]
    _cu(x)
    if width is None or width == D:
        out = torch.empty(x.shape, dtype=BF16, device=x.device)
        K.cast_f32_bf16(x, out)
    else:
        out = torch.zeros(x.shape[:-1] + (width,), dtype=BF16, device=x.device)
        K.cast_f32_bf16_ld(x, out)
    return out


def cast_f32(x, out=None):
    """bf16 -> fp32 (md_cast_bf16_f32)."""
    assert x.dtype == BF16 and x.is_contiguous()
    if out is None:
        out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    _cu(x, out)
    K.cast_bf16_f32(x, out)
    return out


def add_pos_time(x, pos, temb, temb_stride, L, out):
    """out = bf16((pos[l] + x) + temb[b]) for hidden_dim == hidden_size models (md_add_pos_time)."""
    x = _c(x, torch.float32)
    _cu(x, pos, temb, out)
    K.add_pos_time(x, pos, temb, temb_stride, L, out)
    return out


def embed_gather(E, ids):
    E = _c(E, torch.float32)
    if ids.dtype not in (torch.int32, torch.int64):
        ids = ids.to(torch.int64)
    ids = _c(ids)
    out = torch.empty(tuple(ids.shape) + (E.shape[1],), dtype=torch.float32, device=E.device)
    _cu(E, ids)
    K.embed_gather(E, ids, out)
    return out


def timestep_mlp(t, W0, b0, W2, b2):
    t = _c(t, torch.float32)
    _cu(t, W0, b0, W2, b2)
    out = torch.empty((t.numel(), W2.shape[0]), dtype=torch.float32, device=t.device)
    hid = torch.empty((t.numel(), W0.shape[0]), dtype=torch.float32, device=t.device)
    K.timestep_mlp(t, W0, b0, W2, b2, out, hid)
    return out


def layernorm(x, gamma, beta, eps, resid=None, out=None):
    """LayerNorm(x + resid) (resid optional), bf16 in/out."""
    assert x.dtype == BF16 and x.is_contiguous()
    assert resid is None or (resid.dtype == BF16 and resid.is_contiguous() and resid.shape == x.shape)
    H = x.shape[-1]
    if out is None:
        out = torch.empty_like(x)
    if H % 256 != 0 or H > 2048:
        raise _lib.MuseDiffLibraryError("md_layernorm_bf16: H=%d must be a multiple of 256, <= 2048" % H)
    _cu(x, resid, gamma, beta, out)
    K.layernorm_bf16(x, resid, gamma, beta, float(eps), out)
    return out


# ------------------------------------------------------------------------------------------------ contractions
def linear(A, W, bias, epilogue=_lib.EPI_BIAS, out_dtype=BF16, pos=None, temb=None, temb_stride=0, L=0, out=None):
    """out[M,N] = epi(A[M,K] @ W[N,K]^T + bias).  An `out` narrower than N receives the first out.shape[-1] columns
    (md_linear_bf16_cols: how a model whose width is padded to Dp writes its D real output columns)."""
    assert A.dtype == BF16 and W.dtype == BF16 and A.is_contiguous() and W.is_contiguous()
    M, Kd = A.shape
    N = W.shape[0]
    assert W.shape[1] == Kd
    if out is None:
        out = torch.empty((M, 2 * N if epilogue == _lib.EPI_BIAS_SPLIT else N), dtype=out_dtype, device=A.device)
    if epilogue == _lib.EPI_BIAS_SPLIT and (out.dtype != BF16 or out.shape[-1] != 2 * N):
        raise _lib.MuseDiffLibraryError("md_linear_bf16: the split epilogue writes bf16 [M, 2N]")
    _cu(A, W, bias, out, pos, temb)
    if epilogue != _lib.EPI_BIAS_SPLIT and out.shape[-1] != N:
        K.linear_bf16_cols(A, W, bias, out, epilogue, pos, temb, temb_stride, L)
    else:
        K.linear_bf16(A, W, bias, out, epilogue, pos, temb, temb_stride, L)
    return out


def attention(qkv, B, L, NH, out=None):
    assert qkv.dtype == BF16 and qkv.is_contiguous()
    H = qkv.shape[-1] // 3
    if out is None:
        out = torch.empty((B * L, H), dtype=BF16, device=qkv.device)
    if H // NH != 64:
        raise _lib.MuseDiffLibraryError("md_attention_bf16: head dim %d unsupported (kernel is specialised for 64)" % (H // NH))
    _cu(qkv, out)
    K.attention_bf16(qkv, out, B, L, NH)
    return out


# ------------------------------------------------------------------------------------------------ rounding / decode
def round_argmin(x, E, want_margin=False):
    x = _c(x, torch.float32)
    E = _c(E, torch.float32)
    D = E.shape[1]
    M = x.numel() // D
    idx = torch.empty((M,), dtype=torch.int32, device=x.device)
    margin = torch.empty((M,), dtype=torch.float32, device=x.device) if want_margin else None
    _cu(x, E)
    K.round_argmin(x, E, idx, margin)
    return (idx, margin) if want_margin else idx


def logits_argmax(x, E, bias, want_margin=False):
    x = _c(x, torch.float32)
    E = _c(E, torch.float32)
    bias = _c(bias, torch.float32)
    D = E.shape[1]
    M = x.numel() // D
    tok = torch.empty((M,), dtype=torch.int32, device=x.device)
    margin = torch.empty((M,), dtype=torch.float32, device=x.device) if want_margin else None
    _cu(x, E, bias)
    K.logits_argmax(x, E, bias, tok, margin)
    return (tok, margin) if want_margin else tok


def split_bf16(x, copies=1):
    """fp32 [..., D] -> bf16 [rows, copies * 2D] = copies x [hi | lo]."""
    x = _c(x, torch.float32)
    D = x.shape[-1]
    rows = x.numel() // D
    out = torch.empty((rows, copies * 2 * D), dtype=BF16, device=x.device)
    _cu(x)
    K.split_bf16(x, out, copies)
    return out


def dist_scores(x, dot, esq, V):
    """md_dist_scores: -sqrt(clamp(|E_v|^2 + |x|^2 - 2 x.E_v, 0)) -> fp32 [M, V] (get_logits, logits_mode 2)."""
    x = _c(x, torch.float32)
    dot = _c(dot, torch.float32)
    _cu(x, dot, esq)
    out = torch.empty((dot.shape[0], V), dtype=torch.float32, device=x.device)
    K.dist_scores(x.reshape(dot.shape[0], -1), dot, esq, out)
    return out


class SplitEmbedding:
    """bf16 [Vp, 2Dp] = [Eh | 0 | El | 0] split of an embedding matrix (Dp = padded_width(D)) + |E_v|^2, built once per
    matrix version (md_embed_split, md_embed_split_padded when D is not a multiple of 64); `logit_cst(bias)` gives the
    padded per-column constants of the argmax-logits mode."""

    def __init__(self, E):
        E = _c(E.detach(), torch.float32)
        self.V, self.D = E.shape
        self.Dp = padded_width(self.D)
        self.Vp = _lib.lib.md_round_tc_padded_vocab(self.V)
        self.E2 = torch.empty((self.Vp, 2 * self.Dp), dtype=BF16, device=E.device)
        self.sqnorm = torch.empty((self.Vp,), dtype=torch.float32, device=E.device)
        self.E_clamped = torch.empty_like(E)      # clamp(E, -1, 1): what clip_denoised makes of a rounded x0 (diffusion.py:323-324)
        _cu(E)
        if self.Dp == self.D:
            K.embed_split(E, self.E2, self.sqnorm, self.E_clamped)
        else:
            K.embed_split_padded(E, self.E2, self.sqnorm, self.E_clamped)
        self._ws = {}

    def logit_cst(self, bias):
        c = torch.full((self.Vp,), float("-inf"), dtype=torch.float32, device=self.E2.device)
        c[:self.V] = bias.detach().float()
        return c

    def workspace(self, M):
        ws = self._ws.get(M)
        if ws is None:
            self._ws = {M: torch.empty((M, 2 * self.Dp), dtype=BF16, device=self.E2.device)}
            ws = self._ws[M]
        return ws


_split_cache = {}


def split_embedding(E):
    """cached SplitEmbedding for a weight tensor, keyed by storage address + version.  The entry keeps a reference to the
    tensor it was built from: while it is cached its memory cannot be freed and handed to another embedding table, so an
    equal key always means the same contents (a freed table's address IS reused by the caching allocator)."""
    key = (E.data_ptr(), E._version, tuple(E.shape), str(E.device))
    hit = _split_cache.get(key)
    if hit is None:
        if len(_split_cache) > 8:
            _split_cache.clear()
        hit = (SplitEmbedding(E), E)
        _split_cache[key] = hit
    return hit[0]


def round_argmin_tc(x, se, cst=None, mode=0, want_margin=False, out=None, presplit=None, margin_out=None):
    """tensor-core nearest-embedding ids (mode 0, cst = |E|^2) or argmax-logit ids (mode 1, cst = padded bias).
    x: fp32 [..., D].  `presplit`: bf16 [M, 2Dp] = [hi | 0 | lo | 0] of x already written by the producing GEMM
    (EPI_BIAS_SPLIT with N = Dp); x is then ignored.  `margin_out`: fp32 [M] that receives the top-2 margins (as
    want_margin does, into a buffer the caller owns)."""
    if presplit is not None:
        assert presplit.dtype == BF16 and presplit.is_contiguous() and presplit.shape[-1] == 2 * se.Dp
        M = presplit.numel() // (2 * se.Dp)
        x, ws, dev = None, presplit.view(M, 2 * se.Dp), presplit.device
    else:
        x = _c(x, torch.float32)
        M = x.numel() // se.D
        ws, dev = se.workspace(M), x.device
    idx = out if out is not None else torch.empty((M,), dtype=torch.int32, device=dev)
    if margin_out is not None:
        assert margin_out.dtype == torch.float32 and margin_out.is_contiguous() and margin_out.numel() == M
    margin = margin_out if margin_out is not None else (torch.empty((M,), dtype=torch.float32, device=dev) if want_margin else None)
    _cu(x, ws, margin)
    cst = se.sqnorm if cst is None else cst
    if se.Dp == se.D:
        K.round_argmin_tc(x, se.E2, cst, ws, idx, margin, se.V, mode)
    else:
        K.round_argmin_tc_padded(x, se.E2, cst, ws, idx, margin, se.V, se.D, mode)
    return (idx, margin) if want_margin else idx


# ------------------------------------------------------------------------------------------------ posterior step
def _mask_args(mask, B, L, D):
    """mask: None, or an int tensor broadcastable to [B, L, D] (the reference passes a stride-0 expand of [B, L, 1])."""
    if mask is None:
        return None, None, 0, 0
    if mask.dim() == 2:
        mask = mask.unsqueeze(-1)
    m = torch.broadcast_to(mask, (B, L, D))
    if m.stride(-1) == 0 or D == 1:
        tok = m[..., 0]
        tok = tok.to(torch.int32) if tok.dtype != torch.int32 else tok
        tok = tok.contiguous()
        return tok, tok, 1, 0
    full = m.to(torch.int32).contiguous()
    return full, full, D, 1


def _t_args(t, B):
    """t: int tensor with B entries (one schedule index per sequence) or 1 entry (shared by the batch)."""
    t = _c(t.reshape(-1), torch.int32)
    if t.numel() == B and B != 1:
        return t, 1
    if t.numel() == 1:
        return t, 0
    raise ValueError("timestep tensor has %d entries for a batch of %d" % (t.numel(), B))


def posterior_step(x_t, t, mode, idx=None, pred=None, E=None, noise=None, seed=0, step_counter=0, seq_offset=0,
                   mask=None, x_start=None, eta=0.0, clip=True, top_p=0.0, out=None, out_bf16=None, pred_out=None,
                   mean_out=None, step_counter_dev=None):
    """clip: False / True as diffusion.py:323-324, or 2 = `E` already holds clamp(E, -1, 1) (SplitEmbedding.E_clamped).
    out_bf16: bf16 [B, L, D], or [B, L, Dp] with zeroed columns D..Dp-1 (the padded first-GEMM operand)."""
    x_t = _c(x_t, torch.float32)
    B, L, D = x_t.shape
    t, t_stride = _t_args(t, B)
    keep, mask_t, ts, ds = _mask_args(mask, B, L, D)
    if out is None:
        out = torch.empty_like(x_t)
    if pred is not None:
        pred = _c(pred, torch.float32)
    if noise is not None:
        noise = _c(noise, torch.float32)
    if x_start is not None:
        x_start = _c(x_start, torch.float32)
    if idx is not None:
        idx = _c(idx, torch.int32)
    if (idx is None) == (pred is None):
        raise _lib.MuseDiffLibraryError("md_posterior_step: exactly one of idx / pred_in")
    _cu(x_t, idx, pred, E, noise, t, mask_t, x_start, out, out_bf16, pred_out, mean_out, step_counter_dev)
    step = K.posterior_step if out_bf16 is None or out_bf16.shape[-1] == D else K.posterior_step_ld
    step(x_t, idx, pred, E, noise, _s64(seed), _s64(step_counter), int(seq_offset), t, t_stride, mask_t, ts, ds, x_start,
                     out, out_bf16, pred_out, mean_out, mode, float(eta), int(clip), float(top_p or 0.0), step_counter_dev)
    return out


def dpm_solver_step(x_t, coef, pred_hist, idx=None, pred=None, E=None, cursor=None, mask=None, x_start=None, clip=True, out=None,
                    out_bf16=None):
    """One DPM-Solver++(2M) update (md_dpm_solver_step).  coef: fp32 [n, 4] rows (a, b, c0, c1); without `cursor` it has one
    row, with it the kernel takes row *cursor - 1.  pred_hist: fp32 [B, L, D], read where c1 != 0 and overwritten with this
    step's processed x0.  `out` may be x_t itself.  clip and out_bf16 as in posterior_step."""
    x_t = _c(x_t, torch.float32)
    B, L, D = x_t.shape
    keep, mask_t, ts, ds = _mask_args(mask, B, L, D)
    if out is None:
        out = torch.empty_like(x_t)
    if pred is not None:
        pred = _c(pred, torch.float32)
    if idx is not None:
        idx = _c(idx, torch.int32)
    if x_start is not None:
        x_start = _c(x_start, torch.float32)
    if (idx is None) == (pred is None):
        raise _lib.MuseDiffLibraryError("md_dpm_solver_step: exactly one of idx / pred_in")
    if coef.dtype != torch.float32 or coef.dim() != 2 or coef.shape[1] != 4 or not coef.is_contiguous():
        raise _lib.MuseDiffLibraryError("md_dpm_solver_step: coef must be a contiguous fp32 [n, 4] table")
    if pred_hist.dtype != torch.float32 or pred_hist.shape != x_t.shape or not pred_hist.is_contiguous():
        raise _lib.MuseDiffLibraryError("md_dpm_solver_step: pred_hist must be a contiguous fp32 tensor shaped like x_t")
    if cursor is not None and (cursor.dtype != torch.int32 or cursor.numel() != 1):
        raise _lib.MuseDiffLibraryError("md_dpm_solver_step: cursor must be one int32")
    _cu(x_t, idx, pred, E, pred_hist, coef, cursor, mask_t, x_start, out, out_bf16)
    K.dpm_solver_step(x_t, idx, pred, E, pred_hist, coef, cursor, mask_t, ts, ds, x_start, out, out_bf16, int(clip))
    return out


def xstart_from_eps(x_t, eps, t):
    x_t = _c(x_t, torch.float32)
    eps = _c(eps, torch.float32)
    B, L, D = x_t.shape
    out = torch.empty_like(x_t)
    t, t_stride = _t_args(t, B)
    _cu(x_t, eps, t)
    K.xstart_from_eps(x_t, eps, t, t_stride, out)
    return out


def q_sample(x0, t=None, noise=None, seed=0, step_counter=0, seq_offset=0, mask=None, out_bf16=None):
    """t=None -> pure-noise initialisation (generation mode).  out_bf16 as in posterior_step."""
    x0 = _c(x0, torch.float32)
    B, L, D = x0.shape
    keep, mask_t, ts, ds = _mask_args(mask, B, L, D)
    out = torch.empty_like(x0)
    if noise is not None:
        noise = _c(noise, torch.float32)
    tt, t_stride = _t_args(t, B) if t is not None else (None, 0)
    _cu(x0, noise, tt, mask_t, out_bf16)
    qs = K.q_sample if out_bf16 is None or out_bf16.shape[-1] == D else K.q_sample_ld
    qs(x0, noise, _s64(seed), _s64(step_counter), int(seq_offset), tt, t_stride, mask_t, ts, ds, out, out_bf16)
    return out


def fill_normal(shape, device, seed=0, step_counter=0, elem_offset=0, top_p=0.0):
    out = torch.empty(shape, dtype=torch.float32, device=device)
    if int(elem_offset) % 4 != 0:
        raise _lib.MuseDiffLibraryError("md_fill_normal: elem_offset must be a multiple of 4")
    _cu(out)
    K.fill_normal(out, _s64(seed), _s64(step_counter), int(elem_offset), float(top_p))
    return out


def decode_prepare(tokens, mask, strict=False):
    """md_decode_prepare: the token-level half of SequenceToMidi.decode (decode_util.py:72-199) for a whole batch.
    tokens / mask: integer [B, L] CUDA tensors.  Returns (status [B], note_len [B], notes [B, 2L], meta [B, 11]), int32."""
    B, L = tokens.shape
    tok = tokens.to(torch.int32).contiguous()
    msk = mask.to(torch.int32).contiguous()
    dev = tok.device
    status = torch.empty((B,), dtype=torch.int32, device=dev)
    note_len = torch.empty((B,), dtype=torch.int32, device=dev)
    notes = torch.empty((B, 2 * L), dtype=torch.int32, device=dev)
    meta = torch.empty((B, 11), dtype=torch.int32, device=dev)
    _cu(tok, msk)
    K.decode_prepare(tok, msk, bool(strict), status, note_len, notes, meta)
    return status, note_len, notes, meta


def merge_and_mask(src, src_len, trg, trg_len, seq_len, end_token=1):
    """md_merge_and_mask: preprocess.py:30-58 + :73-81 + wrapper.py:90-126 for a padded batch of raw (src, trg) rows.
    Returns (input_ids [B, seq_len], input_mask [B, seq_len], length [B]), int32; rows with length > seq_len are padding."""
    B = src_len.shape[0]
    dev = trg.device
    i32 = lambda t: t.to(torch.int32).contiguous()
    src, src_len, trg, trg_len = i32(src), i32(src_len), i32(trg), i32(trg_len)
    Ls = src.shape[1] if src.dim() == 2 else 0
    Lt = trg.shape[1]
    input_ids = torch.empty((B, seq_len), dtype=torch.int32, device=dev)
    input_mask = torch.empty((B, seq_len), dtype=torch.int32, device=dev)
    length = torch.empty((B,), dtype=torch.int32, device=dev)
    _cu(src_len, trg, trg_len)
    K.merge_and_mask(src if Ls else None, src_len, trg, trg_len, int(seq_len), int(end_token), input_ids, input_mask, length)
    return input_ids, input_mask, length


def sequence_metrics(notes, note_len, meta):
    """md_sequence_metrics (metric.py:4-75, 131-169): notes [B, Ln], note_len [B], meta [B, 11] integer CUDA tensors ->
    (vectors f32 [B, 56] = rhythm | melody | harmony, status int32 [B], stats int32 [B, 4])."""
    i32 = lambda t: t.to(torch.int32).contiguous()
    notes, note_len, meta = i32(notes), i32(note_len), i32(meta)
    B, Ln = notes.shape
    dev = notes.device
    vectors = torch.empty((B, 56), dtype=torch.float32, device=dev)
    status = torch.empty((B,), dtype=torch.int32, device=dev)
    stats = torch.empty((B, 4), dtype=torch.int32, device=dev)
    _cu(notes, note_len, meta)
    K.sequence_metrics(notes, note_len, meta, vectors, status, stats)
    return vectors, status, stats


def onnc_nearest(vectors, want_msim=False):
    """md_onnc (metric.py:99-107): vectors f32 [N, 56] -> (most_sim int32 [N], msim f32 [N, N] or None)."""
    vectors = vectors.to(torch.float32).contiguous()
    N = vectors.shape[0]
    most = torch.empty((N,), dtype=torch.int32, device=vectors.device)
    msim = torch.empty((N, N), dtype=torch.float32, device=vectors.device) if want_msim else None
    _cu(vectors)
    K.onnc(vectors, msim, most)
    return most, msim


def step_advance(cursor, t_idx, t_model, t_cur, tm_cur, ctr_cur, ctr_base):
    """md_step_advance: device-resident loop state of the CUDA-graph replay (see diffusion.GaussianDiffusion._loop)."""
    _cu(cursor, t_idx, t_model, t_cur, tm_cur, ctr_cur)
    K.step_advance(cursor, t_idx, t_model, t_cur, tm_cur, ctr_cur, _s64(ctr_base))
