"""TransformerNetModel — host-side mirror of MuseDiffusion/models/network.py:20-158 whose forward runs on the
hand-written sm_100a kernels (tcgen05 GEMMs + fused attention + vectorised residual-LayerNorm) through the C-ABI library.

The module tree reproduces the reference's parameter names exactly (211 state-dict keys at the base config,
SURVEY.md section 5), so `load_state_dict` of a reference checkpoint works unchanged.  The encoder the reference
borrows from HF `transformers` (`BertEncoder`, network.py:10,74,151) is restated here as plain parameter holders —
12 post-LN layers {query,key,value,attention.output.dense+LayerNorm, intermediate.dense, output.dense+LayerNorm} —
with bert-base-uncased sizes by default (`AutoConfig.from_pretrained('bert-base-uncased')`, network.py:44).

Inference only: dropout (network.py:76,149) is the identity in eval mode, which is the only mode the sampling path
uses (run/sample.py:88)."""
import math
from types import SimpleNamespace

import torch
import torch.nn as nn

from . import _lib, ops

BERT_BASE = dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                 layer_norm_eps=1e-12)


class _SelfAttention(nn.Module):
    def __init__(self, h):
        super().__init__()
        self.query = nn.Linear(h, h)
        self.key = nn.Linear(h, h)
        self.value = nn.Linear(h, h)


class _DenseLN(nn.Module):
    def __init__(self, fan_in, h, eps):
        super().__init__()
        self.dense = nn.Linear(fan_in, h)
        self.LayerNorm = nn.LayerNorm(h, eps=eps)


class _Attention(nn.Module):
    def __init__(self, h, eps):
        super().__init__()
        self.self = _SelfAttention(h)
        self.output = _DenseLN(h, h, eps)


class _Intermediate(nn.Module):
    def __init__(self, h, f):
        super().__init__()
        self.dense = nn.Linear(h, f)


class _Layer(nn.Module):
    def __init__(self, h, f, eps):
        super().__init__()
        self.attention = _Attention(h, eps)
        self.intermediate = _Intermediate(h, f)
        self.output = _DenseLN(f, h, eps)


class _Encoder(nn.Module):
    """Parameter holder with HF BertEncoder's key layout (`layer.{i}.…`)."""

    def __init__(self, cfg):
        super().__init__()
        self.layer = nn.ModuleList([_Layer(cfg.hidden_size, cfg.intermediate_size, cfg.layer_norm_eps)
                                    for _ in range(cfg.num_hidden_layers)])


def _zero_pad(t, rows, cols):
    """t [r, c] (or [r]) zero-extended to [rows, cols] (or [rows])."""
    if t.shape[0] == rows and (t.dim() == 1 or t.shape[1] == cols):
        return t
    out = torch.zeros((rows,) if t.dim() == 1 else (rows, cols), dtype=t.dtype, device=t.device)
    out[tuple(slice(0, n) for n in t.shape)] = t
    return out


class WeightPack:
    """Device-resident bf16 / fp32 weights in the layout the kernels consume: built from the parameters once per parameter
    version (`checkpoint.pack_tensors`), or served straight from a packed weight file (`checkpoint.load_pack`).

    A width D that is not a multiple of 64 is zero-padded to Dp = ops.padded_width(D) here, at load time: up1_w
    [H, Dp] (zero columns: the pad columns of the input contribute nothing), dn2_w [Dp, H] and dn2_b [Dp] (zero rows: the
    pad columns of the output, and so of its [hi | lo] split, are exactly 0).  The embedding E stays [V, D]."""

    def __init__(self, model, tensors=None):
        dev = model.word_embedding.weight.device if tensors is None else tensors["E"].device
        if dev.type != "cuda":
            raise _lib.MuseDiffLibraryError("TransformerNetModel.forward needs the model on a CUDA device "
                                            "(there is no CPU path); call model.to('cuda') first")
        if tensors is None:
            from .checkpoint import pack_tensors
            tensors = pack_tensors({k: v for k, v in model.state_dict().items()}, model.num_heads)
        self.device = dev
        self.H = model.hidden_size
        self.NH = model.num_heads
        self.eps = model.layer_norm_eps
        for name in ("E", "lm_bias", "t0_w", "t0_b", "t2_w", "t2_b", "pos", "ln_g", "ln_b"):
            setattr(self, name, tensors[name])
        for name in ("up1_w", "up1_b", "up2_w", "up2_b", "dn1_w", "dn1_b", "dn2_w", "dn2_b"):
            setattr(self, name, tensors.get(name))          # None: hidden_dim == hidden size, no up / down projection
        self.has_up, self.has_down = self.up1_w is not None, self.dn1_w is not None
        if self.has_up != (model.input_dims != model.hidden_size) or self.has_down != (model.output_dims != model.hidden_size):
            raise ValueError("weight pack and model disagree about input_up_proj / output_down_proj")
        self.D = self.E.shape[1]
        self.Dp = ops.padded_width(self.D) if self.has_up else self.D         # no projections: D == H, a multiple of 64
        if self.has_up:
            self.up1_w = _zero_pad(self.up1_w, self.H, self.Dp)
        if self.has_down:
            self.dn2_w, self.dn2_b = _zero_pad(self.dn2_w, self.Dp, self.H), _zero_pad(self.dn2_b, self.Dp, 0)
        self.layers = []
        i = 0
        while "l%d.wqkv" % i in tensors:
            self.layers.append(SimpleNamespace(**{k: tensors["l%d.%s" % (i, k)] for k in
                                                  ("wqkv", "bqkv", "wo", "bo", "g1", "b1", "w1", "bi", "w2", "b2", "g2", "b2n")}))
            i += 1
        if i != len(model.input_transformers.layer):
            raise ValueError("weight pack holds %d encoder layers, the model has %d" % (i, len(model.input_transformers.layer)))
        # split-bf16 operands for fp32-grade logits on the tensor cores (get_logits):
        #   x.E^T = [xh|xl|xh|xl] . [Eh|Eh|El|El]^T   (all four partial products, K = 4 D, fp32 accumulation)
        V, D = self.E.shape
        Vp = (V + 7) // 8 * 8
        e2 = ops.split_bf16(self.E, copies=1)                       # [V, 2D] = [Eh | El]
        self.E_split = torch.zeros((Vp, 4 * D), dtype=torch.bfloat16, device=dev)
        self.E_split[:V, 0 * D:1 * D] = e2[:, :D]
        self.E_split[:V, 1 * D:2 * D] = e2[:, :D]
        self.E_split[:V, 2 * D:3 * D] = e2[:, D:]
        self.E_split[:V, 3 * D:4 * D] = e2[:, D:]
        self.lm_bias_pad = torch.zeros((Vp,), dtype=torch.float32, device=dev)
        self.lm_bias_pad[:V] = self.lm_bias
        self.split = None          # SplitEmbedding for the tensor-core decode, built on first use
        self.logit_cst = None


class Workspace:
    """Activation buffers for one token count M (reused across steps: nothing is allocated inside the loop)."""

    def __init__(self, M, Dp, H, F, dev):
        bf = lambda *s: torch.empty(s, dtype=torch.bfloat16, device=dev)
        self.M = M
        self.xb = bf(M, Dp)
        self.a = bf(M, H)
        self.b = bf(M, H)
        self.c = bf(M, H)
        self.qkv = bf(M, 3 * H)
        self.mid = bf(M, F)


class TransformerNetModel(nn.Module):
    """Same constructor, attributes and methods as the reference class (network.py:20-158).

    Extra keyword `encoder_config` overrides the bert-base sizes (used for the scaled-up benchmark config)."""

    def __init__(self, input_dims, output_dims, hidden_t_dim, vocab_size, seq_len, dropout=0.1, logits_mode=1,
                 encoder_config=None):
        super().__init__()
        for name, d in (("input_dims", input_dims), ("output_dims", output_dims)):
            if int(d) <= 0 or int(d) % 4:
                raise ValueError("%s (hidden_dim) = %d is not supported: the embedding width must be a positive multiple of 4 "
                                 "(the kernels move rows in float4 groups)" % (name, d))
        cfg = SimpleNamespace(**{**BERT_BASE, **(encoder_config or {})})
        cfg.max_position_embeddings = seq_len
        cfg.vocab_size = vocab_size
        self.config = cfg
        self.input_dims = input_dims
        self.hidden_t_dim = hidden_t_dim
        self.output_dims = output_dims
        self.logits_mode = logits_mode
        self.hidden_size = cfg.hidden_size
        self.num_heads = cfg.num_attention_heads
        self.layer_norm_eps = cfg.layer_norm_eps
        if cfg.hidden_size % cfg.num_attention_heads or cfg.hidden_size // cfg.num_attention_heads != 64:
            raise NotImplementedError("the fused attention kernel is specialised for head dim 64")

        self.word_embedding = nn.Embedding(vocab_size, input_dims)
        self.lm_head = nn.Linear(input_dims, vocab_size)
        with torch.no_grad():
            self.lm_head.weight = self.word_embedding.weight          # tied, network.py:55-58
        time_embed_dim = hidden_t_dim * 4
        self.time_embed = nn.Sequential(nn.Linear(hidden_t_dim, time_embed_dim), nn.SiLU(),
                                        nn.Linear(time_embed_dim, cfg.hidden_size))
        if input_dims != cfg.hidden_size:                                # network.py:67-72
            self.input_up_proj = nn.Sequential(nn.Linear(input_dims, cfg.hidden_size), nn.Tanh(),
                                               nn.Linear(cfg.hidden_size, cfg.hidden_size))
        self.input_transformers = _Encoder(cfg)
        self.dropout = nn.Dropout(dropout)
        self.register_buffer("position_ids", torch.arange(cfg.max_position_embeddings).expand((1, -1)))
        self.position_embeddings = nn.Embedding(cfg.max_position_embeddings, cfg.hidden_size)
        self.LayerNorm = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)
        if output_dims != cfg.hidden_size:                               # network.py:81-86
            self.output_down_proj = nn.Sequential(nn.Linear(cfg.hidden_size, cfg.hidden_size), nn.Tanh(),
                                                  nn.Linear(cfg.hidden_size, output_dims))
        self._pack = None
        self._pack_key = None
        self._pack_refs = None
        self._ws = {}

    # ------------------------------------------------------------------------------------------ packing
    def _params_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def load_weight_pack(self, path, device=None):
        """Serve the kernels from a packed weight file (checkpoint.write_pack) instead of the nn.Parameters: one read of the
        file into one device buffer, no fp32 state dict, no per-tensor packing kernels.  The parameters the rest of the
        sampling path touches directly (word_embedding / lm_head.bias, run/sample.py:92-101 clones the embedding) are
        filled from the pack and the module is moved to `device`; the encoder's nn.Parameters keep their construction-
        time values and are NOT what forward() computes with until `load_state_dict` / `weight_pack(force=True)` is called."""
        from .checkpoint import load_pack
        device = torch.device(device if device is not None else "cuda")
        config, tensors = load_pack(path, device)
        for k, mine in (("hidden_size", self.hidden_size), ("num_attention_heads", self.num_heads),
                        ("num_hidden_layers", len(self.input_transformers.layer)), ("hidden_dim", self.input_dims),
                        ("seq_len", self.config.max_position_embeddings), ("vocab_size", self.config.vocab_size)):
            if k in config and int(config[k]) != int(mine):
                raise ValueError("weight pack %s was written for %s=%s, this model has %s" % (path, k, config[k], mine))
        self.to(device)
        with torch.no_grad():
            self.word_embedding.weight.copy_(tensors["E"])
            self.lm_head.bias.copy_(tensors["lm_bias"])
            self.position_embeddings.weight.copy_(tensors["pos"])
        self._pack = WeightPack(self, tensors=tensors)
        self._pack_key = self._params_key()
        self._pack_refs = [p.data for p in self.parameters()]
        self._ws = {}
        return self

    def weight_pack(self, force=False):
        key = self._params_key()
        if force or self._pack is None or key != self._pack_key:
            self._pack = WeightPack(self)
            self._pack_key = key
            # keep the storages the key was taken from alive for as long as the pack is: `.to()` / `load_state_dict` on
            # another device replace them, and the caching allocator hands a freed block to the next tensor of the same
            # size — an equal (address, version) key must always mean the same weights
            self._pack_refs = [p.data for p in self.parameters()]
            self._ws = {}
        return self._pack

    def workspace(self, M):
        ws = self._ws.get(M)
        if ws is None:
            pk = self.weight_pack()
            self._ws = {M: Workspace(M, pk.Dp, pk.H, self.config.intermediate_size, pk.device)}
            ws = self._ws[M]
        return ws

    # ------------------------------------------------------------------------------------------ reference API
    def get_embeds(self, input_ids):
        """network.py:88-89."""
        return ops.embed_gather(self.weight_pack().E, input_ids)

    def get_logits(self, hidden_repr):
        """network.py:91-93 (logits_mode 1): lm_head(x) = x E^T + b as ONE tcgen05 GEMM over split-bf16 operands
        (all four partial products of x = xh + xl, E = Eh + El with fp32 accumulation: fp32-grade logits)."""
        if self.logits_mode not in (1, 2):
            raise NotImplementedError                                  # network.py:105-106
        pk = self.weight_pack()
        V, D = pk.E.shape
        A = ops.split_bf16(hidden_repr.reshape(-1, D), copies=2)     # [M, 4D] = [xh|xl|xh|xl]
        if self.logits_mode == 1:
            out = ops.linear(A, pk.E_split, pk.lm_bias_pad, _lib.EPI_BIAS, out_dtype=torch.float32)
            return out[:, :V].reshape(*hidden_repr.shape[:-1], V).to(hidden_repr.dtype)
        # logits_mode 2 (network.py:94-104): minus the Euclidean distance to every embedding row, [B, L, V]
        dot = ops.linear(A, pk.E_split, None, _lib.EPI_BIAS, out_dtype=torch.float32)
        esq = ops.split_embedding(pk.E).sqnorm
        out = ops.dist_scores(hidden_repr.reshape(-1, D), dot, esq, V)
        return out.reshape(*hidden_repr.shape[:-1], V).to(hidden_repr.dtype)

    def decode_tokens(self, hidden_repr, want_margin=False):
        """get_logits + argmax(-1) (run/sample.py:219-220) fused into one kernel; logits never reach HBM."""
        pk = self.weight_pack()
        if pk.split is None:
            pk.split = ops.SplitEmbedding(pk.E)
            pk.logit_cst = pk.split.logit_cst(pk.lm_bias)
        r = ops.round_argmin_tc(hidden_repr, pk.split, cst=pk.logit_cst, mode=1, want_margin=want_margin)
        if want_margin:
            return r[0].view(hidden_repr.shape[:-1]).long(), r[1].view(hidden_repr.shape[:-1])
        return r.view(hidden_repr.shape[:-1]).long()

    @staticmethod
    def timestep_embedding(timesteps, dim, max_period=10000):
        """network.py:108-129 (kept for API parity; the forward path computes it inside md_timestep_mlp)."""
        half = dim // 2
        freqs = torch.exp(-math.log(max_period) * torch.arange(0, half, dtype=torch.float32, device=timesteps.device) / half)
        args = timesteps[:, None].float() * freqs[None]
        emb = torch.cat([torch.cos(args), torch.sin(args)], dim=-1)
        if dim % 2:
            emb = torch.cat([emb, torch.zeros_like(emb[:, :1])], dim=-1)
        return emb

    def forward(self, x, timesteps, **_):
        """network.py:131-158.  x: [B, L, D] float, timesteps: [B] (int or float).  Returns [B, L, D] in x.dtype."""
        return self.denoise(x, timesteps).type(x.dtype)

    # ------------------------------------------------------------------------------------------ engine
    # sequences are independent, so a large batch runs through the encoder in passes of at most `max_tokens_per_pass` tokens
    # that share ONE activation workspace (SURVEY.md section 8a: FFN-mid alone is 35 GB at 1024 sequences of the scaled
    # config).  The default is the bench operating point (256 x 2096 tokens): a 512-sequence batch in one pass measured
    # 5.8 % slower per sequence than two passes of 256 (round 1 step sweep).
    max_tokens_per_pass = 256 * 2096

    def pass_size(self, B, L):
        """sequences per encoder pass: equal-sized passes, each within the token cap (at least one sequence)."""
        cap = max(1, int(self.max_tokens_per_pass) // L) if self.max_tokens_per_pass else B
        n_pass = -(-B // cap)
        return -(-B // n_pass)

    def denoise(self, x, timesteps, x_bf16=None, uniform_t=False, out=None, split_out=None):
        """The CUDA forward.  `x_bf16`: optional bf16 copy of x already produced by the posterior-step kernel, [B, L, Dp]
        (Dp = ops.padded_width(D), zero columns D..Dp-1); `uniform_t`: all rows share timesteps[0] (true inside the sampling
        loops) -> one time-embedding row; `split_out`: bf16 [B, L, 2Dp] — the last Linear then writes the [hi | 0 | lo | 0]
        split of the output (operand of the tensor-core rounding) INSTEAD of the fp32 tensor, and `split_out` is returned."""
        pk = self.weight_pack()
        if not x.is_cuda:
            raise _lib.MuseDiffLibraryError("TransformerNetModel.forward needs CUDA tensors (no CPU path)")
        B, L, D = x.shape
        if L > self.config.max_position_embeddings:
            raise ValueError("sequence length %d exceeds seq_len %d" % (L, self.config.max_position_embeddings))
        t = timesteps.reshape(-1).float()
        if not uniform_t:
            if t.numel() == 1:
                uniform_t = True                  # one timestep for the whole batch (GaussianDiffusion._step allows it)
            elif t.numel() != B:                  # the reference asserts t.shape == (B,) (network.py:137 via timestep_embedding)
                raise ValueError("timesteps has %d entries for a batch of %d sequences" % (t.numel(), B))
        if split_out is not None and not pk.has_down:
            raise ValueError("split_out needs the output_down_proj GEMM (hidden_dim != hidden size)")
        Dp = pk.Dp
        if split_out is not None:
            out = split_out.view(B, L, 2 * Dp)
        else:
            if out is None:
                out = torch.empty((B, L, D), dtype=torch.float32, device=x.device)
            out = out.view(B, L, D)
        if pk.has_up:
            xb = (x_bf16.view(B, L, Dp) if x_bf16 is not None
                  else ops.cast_bf16(x.reshape(B * L, D).float(), width=Dp).view(B, L, Dp))
        else:
            xb = x.float().contiguous()                   # emb_x = x (network.py:143-144): the fp32 state feeds the pre-LN sum
        temb = ops.timestep_mlp(t[:1] if uniform_t else t, pk.t0_w, pk.t0_b, pk.t2_w, pk.t2_b)
        mb = self.pass_size(B, L)
        ws = self.workspace(mb * L)
        for s in range(0, B, mb):
            e = min(B, s + mb)
            self._encoder_pass(pk, ws, xb[s:e], temb if uniform_t else temb[s:e], uniform_t, out[s:e], split_out is not None)
        return out

    def _encoder_pass(self, pk, ws, xb, temb, uniform_t, out, split=False):
        """network.py:141-157 for a contiguous slice of sequences: xb bf16 [b, L, Dp] -> out fp32 [b, L, D]
        (split: bf16 [b, L, 2Dp] = [hi | 0 | lo | 0])."""
        b, L, Dp = xb.shape
        M, H = b * L, pk.H
        E = _lib
        a, bb, c, qkv, mid = ws.a[:M], ws.b[:M], ws.c[:M], ws.qkv[:M], ws.mid[:M]
        if pk.has_up:
            ops.linear(xb.view(M, Dp), pk.up1_w, pk.up1_b, E.EPI_BIAS_TANH, out=a)
            ops.linear(a, pk.up2_w, pk.up2_b, E.EPI_BIAS_POS_TIME, pos=pk.pos, temb=temb,
                       temb_stride=0 if uniform_t else H, L=L, out=bb)
        else:
            ops.add_pos_time(xb.view(M, Dp), pk.pos, temb, 0 if uniform_t else H, L, bb)
        h, h1, pre = a, c, bb
        ops.layernorm(pre, pk.ln_g, pk.ln_b, pk.eps, out=h)
        for ly in pk.layers:
            ops.linear(h, ly.wqkv, ly.bqkv, E.EPI_BIAS, out=qkv)
            ops.attention(qkv, b, L, pk.NH, out=h1)                          # ctx -> h1 buffer
            ops.linear(h1, ly.wo, ly.bo, E.EPI_BIAS, out=pre)
            ops.layernorm(pre, ly.g1, ly.b1, pk.eps, resid=h, out=h1)        # LN(dense(ctx) + h)
            ops.linear(h1, ly.w1, ly.bi, E.EPI_BIAS_GELU, out=mid)
            ops.linear(mid, ly.w2, ly.b2, E.EPI_BIAS, out=pre)
            ops.layernorm(pre, ly.g2, ly.b2n, pk.eps, resid=h1, out=h)       # LN(dense(mid) + h1)
        if not pk.has_down:
            ops.cast_f32(h, out=out.view(M, -1))          # h.type(x.dtype) of the last hidden state (network.py:155-157)
            return
        ops.linear(h, pk.dn1_w, pk.dn1_b, E.EPI_BIAS_TANH, out=h1)
        if split:
            ops.linear(h1, pk.dn2_w, pk.dn2_b, E.EPI_BIAS_SPLIT, out=out.view(M, 2 * Dp))
        else:                                             # N = Dp, the D real columns are stored
            ops.linear(h1, pk.dn2_w, pk.dn2_b, E.EPI_BIAS, out=out.view(M, -1))
