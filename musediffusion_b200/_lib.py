"""ctypes binding of the C-ABI library (include/musediff_b200.h).

The library is the product: if it is missing or fails to load, importing this module raises — there is no CPU or
eager-PyTorch fallback anywhere in the package."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmusediff_b200.so")

c_p = ctypes.c_void_p
c_i = ctypes.c_int
c_i64 = ctypes.c_int64
c_u64 = ctypes.c_uint64
c_f = ctypes.c_float

# name -> argtypes, mirrors include/musediff_b200.h exactly (tests check every symbol is exported)
SIGNATURES = {
    "md_set_schedule": [c_p, c_i, c_p],
    "md_cast_f32_bf16": [c_p, c_p, c_i64, c_p],
    "md_cast_f32_bf16_ld": [c_p, c_p, c_i64, c_i, c_i, c_p],
    "md_cast_bf16_f32": [c_p, c_p, c_i64, c_p],
    "md_add_pos_time": [c_p, c_p, c_p, c_i, c_i, c_i, c_p, c_i64, c_p],
    "md_embed_gather": [c_p, c_p, c_i, c_p, c_i64, c_i, c_i, c_p],
    "md_timestep_mlp": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_p],
    "md_layernorm_bf16": [c_p, c_p, c_p, c_p, c_f, c_p, c_i64, c_i, c_p],
    "md_linear_bf16": [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_i, c_i, c_p],
    "md_linear_bf16_cols": [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_i, c_i, c_p],
    "md_attention_bf16": [c_p, c_p, c_i, c_i, c_i, c_i, c_p],
    "md_round_argmin": [c_p, c_p, c_p, c_p, c_i64, c_i, c_i, c_p],
    "md_logits_argmax": [c_p, c_p, c_p, c_p, c_p, c_i64, c_i, c_i, c_p],
    "md_split_bf16": [c_p, c_p, c_i64, c_i, c_i, c_p],
    "md_dist_scores": [c_p, c_p, c_p, c_p, c_i64, c_i, c_i, c_i, c_p],
    "md_round_tc_padded_vocab": [c_i],
    "md_embed_split": [c_p, c_i, c_i, c_p, c_p, c_p, c_p],
    "md_round_argmin_tc": [c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_i, c_i, c_i, c_p],
    "md_embed_split_padded": [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_p],
    "md_round_argmin_tc_padded": [c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_i, c_i, c_i, c_i, c_p],
    "md_posterior_step": [c_p, c_p, c_p, c_p, c_p, c_u64, c_u64, c_i64, c_p, c_i, c_p, c_i64, c_i64, c_p, c_p, c_p,
                          c_p, c_p, c_i, c_i, c_i, c_i, c_f, c_i, c_f, c_p, c_p],
    "md_posterior_step_ld": [c_p, c_p, c_p, c_p, c_p, c_u64, c_u64, c_i64, c_p, c_i, c_p, c_i64, c_i64, c_p, c_p, c_p,
                             c_i, c_p, c_p, c_i, c_i, c_i, c_i, c_f, c_i, c_f, c_p, c_p],
    "md_step_advance": [c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_u64, c_p],
    "md_dpm_solver_step": [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_i64, c_i64, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i,
                           c_p],
    "md_xstart_from_eps": [c_p, c_p, c_p, c_i, c_p, c_i, c_i, c_i, c_p],
    "md_q_sample": [c_p, c_p, c_u64, c_u64, c_i64, c_p, c_i, c_p, c_i64, c_i64, c_p, c_p, c_i, c_i, c_i, c_p],
    "md_q_sample_ld": [c_p, c_p, c_u64, c_u64, c_i64, c_p, c_i, c_p, c_i64, c_i64, c_p, c_p, c_i, c_i, c_i, c_i, c_p],
    "md_fill_normal": [c_p, c_i64, c_u64, c_u64, c_i64, c_f, c_p],
    "md_decode_prepare": [c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p],
    "md_merge_and_mask": [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p],
    "md_sequence_metrics": [c_p, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p],
    "md_onnc": [c_p, c_i, c_p, c_p, c_p],
}

EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_TANH, EPI_BIAS_POS_TIME, EPI_BIAS_SPLIT = 0, 1, 2, 4, 5
STEP_DDPM, STEP_DDIM = 0, 1
MAX_CONST_T = 2048


class MuseDiffLibraryError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise MuseDiffLibraryError(
            "musediffusion_b200: %s not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C musediffusion_b200/csrc`). There is no fallback path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.md_last_error.restype = ctypes.c_char_p
    lib.md_last_error.argtypes = []
    lib.md_abi_version.restype = c_i
    lib.md_abi_version.argtypes = []
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = c_i
        fn.argtypes = argtypes
    return lib


lib = _load()


def check(rc, name):
    if rc != 0:
        raise MuseDiffLibraryError("%s failed (%d): %s" % (name, rc, lib.md_last_error().decode("utf-8", "replace")))


def call(name, *args):
    check(getattr(lib, name)(*args), name)
