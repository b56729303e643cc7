"""PyTorch custom ops of the B200 sampling path: `torch.ops.musediff.*`.

Each op is one entry point of the C-ABI library (include/musediff_b200.h) registered with `torch.library` for the CUDA
dispatch key only — there is no CPU (or any other) backend, so a CPU tensor reaching an op is a dispatcher error, never a
silent fallback.  The schemas spell out what every call mutates (`Tensor(a!)`), outputs and scratch buffers are always
passed in by the caller (nothing is allocated inside an op), and every op enqueues its kernel on the current CUDA
stream through ctypes (`_lib.call`): the "thin C-ABI extension" of BASELINE.json's north star.

`musediffusion_b200.ops` holds the tensor-level wrappers (allocation, dtype / layout checks) that the host mirror of the
reference's classes calls; they all end in one of these ops.
"""
import torch

from . import _lib

NAMESPACE = "musediff"
_LIBRARY = torch.library.Library(NAMESPACE, "DEF")

_LAUNCHES = [0]
_PROFILE = [None]      # list of (name, detail, start_event, end_event) while ops.profile_step() is active
_U64 = (1 << 64) - 1


def launch(name, *args, detail=""):
    """one C-ABI call == one kernel launch of ours (a few entries launch two small kernels back to back)."""
    prof = _PROFILE[0]
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.call(name, *args)
        e1.record()
        prof.append((name, detail, e0, e1))
    else:
        _lib.call(name, *args)
    _LAUNCHES[0] += 1


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _s64(v):
    """uint64 seeds / counters travel through the int64 `int` of the op schema."""
    v = int(v) & _U64
    return v - (1 << 64) if v >= (1 << 63) else v


def _define(schema, fn):
    _LIBRARY.define(schema)
    _LIBRARY.impl(schema.split("(", 1)[0], fn, "CUDA")


# ------------------------------------------------------------------------------------------------ elementwise
def _cast_f32_bf16(x, out):
    launch("md_cast_f32_bf16", _p(x), _p(out), x.numel(), _stream())


def _cast_f32_bf16_ld(x, out):
    D = x.shape[-1]
    launch("md_cast_f32_bf16_ld", _p(x), _p(out), x.numel() // D, D, out.shape[-1], _stream())


def _cast_bf16_f32(x, out):
    launch("md_cast_bf16_f32", _p(x), _p(out), x.numel(), _stream())


def _add_pos_time(x, pos, temb, temb_stride, L, out):
    H = x.shape[-1]
    launch("md_add_pos_time", _p(x), _p(pos), _p(temb), temb_stride, L, H, _p(out), x.numel() // H, _stream())


def _embed_gather(E, ids, out):
    launch("md_embed_gather", _p(E), _p(ids), int(ids.dtype == torch.int64), _p(out), ids.numel(), E.shape[0], E.shape[1], _stream())


def _timestep_mlp(t, W0, b0, W2, b2, out, hid):
    launch("md_timestep_mlp", _p(t), _p(W0), _p(b0), _p(W2), _p(b2), _p(out), _p(hid), t.numel(), W0.shape[1], W0.shape[0],
           W2.shape[0], _stream())


def _layernorm_bf16(x, resid, gamma, beta, eps, out):
    H = x.shape[-1]
    launch("md_layernorm_bf16", _p(x), _p(resid), _p(gamma), _p(beta), float(eps), _p(out), x.numel() // H, H, _stream())


# ------------------------------------------------------------------------------------------------ contractions
def _linear_bf16(A, W, bias, out, epilogue, pos, temb, temb_stride, L):
    M, K = A.shape
    N = W.shape[0]                                     # (the split epilogue writes out = bf16 [M, 2N])
    launch("md_linear_bf16", _p(A), _p(W), _p(bias), _p(out), M, N, K, epilogue, int(out.dtype == torch.float32), _p(pos), _p(temb),
           temb_stride, L, _stream(), detail="%dx%dx%d epi=%d" % (M, N, K, epilogue))


def _linear_bf16_cols(A, W, bias, out, epilogue, pos, temb, temb_stride, L):
    M, K = A.shape
    N = W.shape[0]
    launch("md_linear_bf16_cols", _p(A), _p(W), _p(bias), _p(out), M, N, K, out.shape[-1], epilogue, int(out.dtype == torch.float32),
           _p(pos), _p(temb), temb_stride, L, _stream(), detail="%dx%dx%d epi=%d cols=%d" % (M, N, K, epilogue, out.shape[-1]))


def _attention_bf16(qkv, out, B, L, NH):
    launch("md_attention_bf16", _p(qkv), _p(out), B, L, NH, qkv.shape[-1] // (3 * NH), _stream())


# ------------------------------------------------------------------------------------------------ rounding / decode
def _round_argmin(x, E, idx, margin):
    launch("md_round_argmin", _p(x), _p(E), _p(idx), _p(margin), idx.numel(), E.shape[0], E.shape[1], _stream())


def _logits_argmax(x, E, bias, tok, margin):
    launch("md_logits_argmax", _p(x), _p(E), _p(bias), _p(tok), _p(margin), tok.numel(), E.shape[0], E.shape[1], _stream())


def _split_bf16(x, out, copies):
    D = x.shape[-1]
    launch("md_split_bf16", _p(x), _p(out), x.numel() // D, D, copies, _stream())


def _dist_scores(x, dot, esq, out):
    launch("md_dist_scores", _p(x), _p(dot), _p(esq), _p(out), out.shape[0], out.shape[1], dot.shape[1], x.shape[-1], _stream())


def _embed_split(E, E2, sqnorm, E_clamped):
    launch("md_embed_split", _p(E), E.shape[0], E.shape[1], _p(E2), _p(sqnorm), _p(E_clamped), _stream())


def _round_argmin_tc(x, E2, cst, ws, idx, margin, V, mode):
    D = E2.shape[1] // 2
    launch("md_round_argmin_tc", _p(x), _p(E2), _p(cst), _p(ws), _p(idx), _p(margin), idx.numel(), V, D, mode, _stream())


def _embed_split_padded(E, E2, sqnorm, E_clamped):
    launch("md_embed_split_padded", _p(E), E.shape[0], E.shape[1], E2.shape[1] // 2, _p(E2), _p(sqnorm), _p(E_clamped), _stream())


def _round_argmin_tc_padded(x, E2, cst, ws, idx, margin, V, D, mode):
    launch("md_round_argmin_tc_padded", _p(x), _p(E2), _p(cst), _p(ws), _p(idx), _p(margin), idx.numel(), V, D, E2.shape[1] // 2, mode,
           _stream())


# ------------------------------------------------------------------------------------------------ diffusion steps
def _posterior_step(x_t, idx, pred, E, noise, seed, step_counter, seq_offset, t, t_stride, mask, mask_tok_stride, mask_d_stride,
                    x_start, out, out_bf16, pred_out, mean_out, mode, eta, clip, top_p, step_counter_dev):
    B, L, D = x_t.shape
    launch("md_posterior_step", _p(x_t), _p(idx), _p(pred), _p(E), _p(noise), seed & _U64, step_counter & _U64, seq_offset, _p(t),
           t_stride, _p(mask), mask_tok_stride, mask_d_stride, _p(x_start), _p(out), _p(out_bf16), _p(pred_out), _p(mean_out),
           B, L, D, mode, float(eta), int(clip), float(top_p), _p(step_counter_dev), _stream())


def _posterior_step_ld(x_t, idx, pred, E, noise, seed, step_counter, seq_offset, t, t_stride, mask, mask_tok_stride, mask_d_stride,
                       x_start, out, out_bf16, pred_out, mean_out, mode, eta, clip, top_p, step_counter_dev):
    B, L, D = x_t.shape
    launch("md_posterior_step_ld", _p(x_t), _p(idx), _p(pred), _p(E), _p(noise), seed & _U64, step_counter & _U64, seq_offset, _p(t),
           t_stride, _p(mask), mask_tok_stride, mask_d_stride, _p(x_start), _p(out), _p(out_bf16),
           out_bf16.shape[-1] if out_bf16 is not None else D, _p(pred_out), _p(mean_out), B, L, D, mode, float(eta), int(clip),
           float(top_p), _p(step_counter_dev), _stream())


def _xstart_from_eps(x_t, eps, t, t_stride, out):
    B, L, D = x_t.shape
    launch("md_xstart_from_eps", _p(x_t), _p(eps), _p(t), t_stride, _p(out), B, L, D, _stream())


def _q_sample(x0, noise, seed, step_counter, seq_offset, t, t_stride, mask, mask_tok_stride, mask_d_stride, out, out_bf16):
    B, L, D = x0.shape
    launch("md_q_sample", _p(x0), _p(noise), seed & _U64, step_counter & _U64, seq_offset, _p(t), t_stride, _p(mask), mask_tok_stride,
           mask_d_stride, _p(out), _p(out_bf16), B, L, D, _stream())


def _q_sample_ld(x0, noise, seed, step_counter, seq_offset, t, t_stride, mask, mask_tok_stride, mask_d_stride, out, out_bf16):
    B, L, D = x0.shape
    launch("md_q_sample_ld", _p(x0), _p(noise), seed & _U64, step_counter & _U64, seq_offset, _p(t), t_stride, _p(mask), mask_tok_stride,
           mask_d_stride, _p(out), _p(out_bf16), out_bf16.shape[-1] if out_bf16 is not None else D, B, L, D, _stream())


def _fill_normal(out, seed, step_counter, elem_offset, top_p):
    launch("md_fill_normal", _p(out), out.numel(), seed & _U64, step_counter & _U64, elem_offset, float(top_p), _stream())


def _step_advance(cursor, t_idx, t_model, t_cur, tm_cur, ctr_cur, ctr_base):
    launch("md_step_advance", _p(cursor), _p(t_idx), _p(t_model), t_idx.numel(), _p(t_cur), _p(tm_cur), _p(ctr_cur), ctr_base & _U64,
           _stream())


def _dpm_solver_step(x_t, idx, pred, E, pred_hist, coef, cursor, mask, mask_tok_stride, mask_d_stride, x_start, out, out_bf16, clip):
    B, L, D = x_t.shape
    launch("md_dpm_solver_step", _p(x_t), _p(idx), _p(pred), _p(E), _p(pred_hist), _p(coef), coef.shape[0], _p(cursor), _p(mask),
           mask_tok_stride, mask_d_stride, _p(x_start), _p(out), _p(out_bf16), out_bf16.shape[-1] if out_bf16 is not None else D,
           B, L, D, int(clip), _stream())


# ------------------------------------------------------------------------------------------------ rows either side of the path
def _decode_prepare(tokens, mask, strict, status, note_len, notes, meta):
    B, L = tokens.shape
    launch("md_decode_prepare", _p(tokens), _p(mask), B, L, int(strict), _p(status), _p(note_len), _p(notes), _p(meta), _stream())


def _merge_and_mask(src, src_len, trg, trg_len, seq_len, end_token, input_ids, input_mask, length):
    B = src_len.shape[0]
    Ls = src.shape[1] if (src is not None and src.dim() == 2) else 0
    launch("md_merge_and_mask", _p(src) if Ls else None, _p(src_len), _p(trg), _p(trg_len), B, Ls, trg.shape[1], seq_len, end_token,
           _p(input_ids), _p(input_mask), _p(length), _stream())


def _sequence_metrics(notes, note_len, meta, vectors, status, stats):
    B, Ln = notes.shape
    launch("md_sequence_metrics", _p(notes), _p(note_len), _p(meta), B, Ln, _p(vectors), _p(status), _p(stats), _stream())


def _onnc(vectors, msim, most_sim):
    launch("md_onnc", _p(vectors), vectors.shape[0], _p(msim), _p(most_sim), _stream())


_define("cast_f32_bf16(Tensor x, Tensor(a!) out) -> ()", _cast_f32_bf16)
_define("cast_f32_bf16_ld(Tensor x, Tensor(a!) out) -> ()", _cast_f32_bf16_ld)
_define("cast_bf16_f32(Tensor x, Tensor(a!) out) -> ()", _cast_bf16_f32)
_define("add_pos_time(Tensor x, Tensor pos, Tensor temb, int temb_stride, int L, Tensor(a!) out) -> ()", _add_pos_time)
_define("embed_gather(Tensor E, Tensor ids, Tensor(a!) out) -> ()", _embed_gather)
_define("timestep_mlp(Tensor t, Tensor W0, Tensor b0, Tensor W2, Tensor b2, Tensor(a!) out, Tensor(b!) hid) -> ()", _timestep_mlp)
_define("layernorm_bf16(Tensor x, Tensor? resid, Tensor gamma, Tensor beta, float eps, Tensor(a!) out) -> ()", _layernorm_bf16)
_define("linear_bf16(Tensor A, Tensor W, Tensor? bias, Tensor(a!) out, int epilogue, Tensor? pos, Tensor? temb, int temb_stride, "
        "int L) -> ()", _linear_bf16)
_define("linear_bf16_cols(Tensor A, Tensor W, Tensor? bias, Tensor(a!) out, int epilogue, Tensor? pos, Tensor? temb, "
        "int temb_stride, int L) -> ()", _linear_bf16_cols)
_define("attention_bf16(Tensor qkv, Tensor(a!) out, int B, int L, int NH) -> ()", _attention_bf16)
_define("round_argmin(Tensor x, Tensor E, Tensor(a!) idx, Tensor(b!)? margin) -> ()", _round_argmin)
_define("logits_argmax(Tensor x, Tensor E, Tensor bias, Tensor(a!) tok, Tensor(b!)? margin) -> ()", _logits_argmax)
_define("split_bf16(Tensor x, Tensor(a!) out, int copies) -> ()", _split_bf16)
_define("embed_split(Tensor E, Tensor(a!) E2, Tensor(b!) sqnorm, Tensor(c!)? E_clamped) -> ()", _embed_split)
_define("dist_scores(Tensor x, Tensor dot, Tensor esq, Tensor(a!) out) -> ()", _dist_scores)
_define("round_argmin_tc(Tensor? x, Tensor E2, Tensor cst, Tensor(a!) ws, Tensor(b!) idx, Tensor(c!)? margin, int V, int mode) -> ()",
        _round_argmin_tc)
_define("embed_split_padded(Tensor E, Tensor(a!) E2, Tensor(b!) sqnorm, Tensor(c!)? E_clamped) -> ()", _embed_split_padded)
_define("round_argmin_tc_padded(Tensor? x, Tensor E2, Tensor cst, Tensor(a!) ws, Tensor(b!) idx, Tensor(c!)? margin, int V, int D, "
        "int mode) -> ()", _round_argmin_tc_padded)
_define("posterior_step(Tensor x_t, Tensor? idx, Tensor? pred, Tensor? E, Tensor? noise, int seed, int step_counter, int seq_offset, "
        "Tensor t, int t_stride, Tensor? mask, int mask_tok_stride, int mask_d_stride, Tensor? x_start, Tensor(a!) out, "
        "Tensor(b!)? out_bf16, Tensor(c!)? pred_out, Tensor(d!)? mean_out, int mode, float eta, int clip, float top_p, "
        "Tensor? step_counter_dev) -> ()", _posterior_step)
_define("posterior_step_ld(Tensor x_t, Tensor? idx, Tensor? pred, Tensor? E, Tensor? noise, int seed, int step_counter, "
        "int seq_offset, Tensor t, int t_stride, Tensor? mask, int mask_tok_stride, int mask_d_stride, Tensor? x_start, Tensor(a!) out, "
        "Tensor(b!)? out_bf16, Tensor(c!)? pred_out, Tensor(d!)? mean_out, int mode, float eta, int clip, float top_p, "
        "Tensor? step_counter_dev) -> ()", _posterior_step_ld)
_define("xstart_from_eps(Tensor x_t, Tensor eps, Tensor t, int t_stride, Tensor(a!) out) -> ()", _xstart_from_eps)
_define("q_sample(Tensor x0, Tensor? noise, int seed, int step_counter, int seq_offset, Tensor? t, int t_stride, Tensor? mask, "
        "int mask_tok_stride, int mask_d_stride, Tensor(a!) out, Tensor(b!)? out_bf16) -> ()", _q_sample)
_define("q_sample_ld(Tensor x0, Tensor? noise, int seed, int step_counter, int seq_offset, Tensor? t, int t_stride, Tensor? mask, "
        "int mask_tok_stride, int mask_d_stride, Tensor(a!) out, Tensor(b!)? out_bf16) -> ()", _q_sample_ld)
_define("fill_normal(Tensor(a!) out, int seed, int step_counter, int elem_offset, float top_p) -> ()", _fill_normal)
_define("step_advance(Tensor(a!) cursor, Tensor t_idx, Tensor t_model, Tensor(b!) t_cur, Tensor(c!) tm_cur, Tensor(d!) ctr_cur, "
        "int ctr_base) -> ()", _step_advance)
_define("dpm_solver_step(Tensor x_t, Tensor? idx, Tensor? pred, Tensor? E, Tensor(a!) pred_hist, Tensor coef, Tensor? cursor, "
        "Tensor? mask, int mask_tok_stride, int mask_d_stride, Tensor? x_start, Tensor(b!) out, Tensor(c!)? out_bf16, int clip) -> ()",
        _dpm_solver_step)
_define("decode_prepare(Tensor tokens, Tensor mask, bool strict, Tensor(a!) status, Tensor(b!) note_len, Tensor(c!) notes, "
        "Tensor(d!) meta) -> ()", _decode_prepare)
_define("merge_and_mask(Tensor? src, Tensor src_len, Tensor trg, Tensor trg_len, int seq_len, int end_token, Tensor(a!) input_ids, "
        "Tensor(b!) input_mask, Tensor(c!) length) -> ()", _merge_and_mask)
_define("sequence_metrics(Tensor notes, Tensor note_len, Tensor meta, Tensor(a!) vectors, Tensor(b!) status, Tensor(c!) stats) -> ()",
        _sequence_metrics)
_define("onnc(Tensor vectors, Tensor(a!)? msim, Tensor(b!) most_sim) -> ()", _onnc)

OP_NAMES = ["cast_f32_bf16", "cast_f32_bf16_ld", "cast_bf16_f32", "add_pos_time", "embed_gather", "timestep_mlp", "layernorm_bf16",
            "linear_bf16", "linear_bf16_cols", "attention_bf16", "round_argmin", "logits_argmax", "split_bf16", "dist_scores",
            "embed_split", "embed_split_padded", "round_argmin_tc", "round_argmin_tc_padded", "posterior_step", "posterior_step_ld",
            "xstart_from_eps", "q_sample", "q_sample_ld", "fill_normal", "step_advance", "dpm_solver_step", "decode_prepare",
            "merge_and_mask", "sequence_metrics", "onnc"]
ops = getattr(torch.ops, NAMESPACE)
