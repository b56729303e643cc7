"""On-disk formats of the sampling path (SURVEY.md section 8(f) row 3).

1. What the reference's trainer leaves in a model directory and `run/sample.py:76-85` reads back:
     model_*.pt            `torch.save(state_dict)`, read through blobfile (utils/dist_util.py:118-124)
     training_args.json    `TrainSettings(...).json()` — pydantic v1 (config/sample.py:114-134, config/train.py)
   `load_training_args` / `load_state_dict` read both with plain json / torch.load (no blobfile, no pydantic).

2. A packed weight file (`*.mdpack`) for instant start-up: the denoiser's weights exactly as the kernels consume them
   (`pack_tensors`: bf16 [N, K] GEMM operands with W_q|W_k|W_v fused and 1/sqrt(64) folded into W_q, fp32 biases /
   LayerNorm / position / time-MLP / embedding), written ONCE from a checkpoint.  Loading is one read of the file into a
   single device buffer (memory-mapped source, no fp32 state dict, no per-tensor cast / cat kernels): every packed tensor
   is a view into that buffer at a 256-byte aligned offset.

   layout:  b"MDPACK01" | u64 header_len | header JSON (utf-8) | padding to 256 | tensor bytes (each 256-aligned)
   header:  {"format": 1, "config": {...model hyper-parameters...}, "tensors": [{"name", "dtype", "shape", "offset", "nbytes"}]}
   Tensors keep the reference's shapes at every hidden_dim D: a D that is not a multiple of 64 is zero-padded to the
   tensor-core width when the pack is loaded (`network.WeightPack`), not in the file, so packs of every width share one format.
"""
import json
import math
import os
from types import SimpleNamespace

import numpy as np
import torch

MAGIC = b"MDPACK01"
ALIGN = 256
_DTYPES = {"bfloat16": torch.bfloat16, "float32": torch.float32}

# the fields of TrainSettings that create_model_and_diffusion reads (utils/initialization.py:108-136) and their defaults
# (config/train.py:35-68); everything else in training_args.json is carried along untouched
MODEL_FIELDS = {"seq_len": 2096, "vocab_size": 729, "hidden_t_dim": 128, "hidden_dim": 128, "dropout": 0.1,
                "diffusion_steps": 2000, "noise_schedule": "sqrt", "predict_xstart": True, "rescale_timesteps": True,
                "timestep_respacing": ""}


def training_args_path(model_path):
    """config/sample.py:123-134: `training_args.json` sits next to the checkpoint unless given explicitly."""
    return os.path.join(os.path.split(os.path.abspath(model_path))[0], "training_args.json")


def load_training_args(path):
    """`TrainSettings.parse_file(model_config_json)` (run/sample.py:77) without pydantic: the file is the flat JSON object
    `TrainSettings(...).json()` wrote.  `path` may be the json itself, a checkpoint next to it, or the directory."""
    if os.path.isdir(path):
        path = os.path.join(path, "training_args.json")
    elif not path.endswith(".json"):
        path = training_args_path(path)
    with open(path) as f:
        raw = json.load(f)
    if not isinstance(raw, dict):
        raise ValueError("%s does not hold a TrainSettings object" % path)
    args = dict(MODEL_FIELDS)
    args.update(raw)
    for k in ("predict_xstart", "rescale_timesteps"):             # pydantic's bool_validator accepts these spellings too
        if isinstance(args[k], str):
            args[k] = args[k].strip().lower() in ("1", "true", "yes", "on", "y", "t")
    return SimpleNamespace(**args)


def load_state_dict(path, map_location="cpu"):
    """utils/dist_util.py:118-124 (`bf.BlobFile(path, "rb")` + torch.load) for local paths."""
    with open(path, "rb") as f:
        return torch.load(f, map_location=map_location)


# ------------------------------------------------------------------------------------------------ packing
def pack_tensors(sd, num_heads):
    """state dict (reference key names, any device / float dtype) -> ordered dict name -> packed tensor, the layout
    `network.WeightPack` serves to the kernels.  Pure tensor bookkeeping (cast / cat / scale by a power of two)."""
    bf = lambda t: t.detach().to(torch.bfloat16).contiguous()
    f32 = lambda t: t.detach().to(torch.float32).contiguous()
    out = {}
    out["E"] = f32(sd["word_embedding.weight"])
    out["lm_bias"] = f32(sd["lm_head.bias"])
    out["t0_w"], out["t0_b"] = f32(sd["time_embed.0.weight"]), f32(sd["time_embed.0.bias"])
    out["t2_w"], out["t2_b"] = f32(sd["time_embed.2.weight"]), f32(sd["time_embed.2.bias"])
    if "input_up_proj.0.weight" in sd:               # absent when hidden_dim == encoder hidden size (network.py:67-72)
        out["up1_w"], out["up1_b"] = bf(sd["input_up_proj.0.weight"]), f32(sd["input_up_proj.0.bias"])
        out["up2_w"], out["up2_b"] = bf(sd["input_up_proj.2.weight"]), f32(sd["input_up_proj.2.bias"])
    out["pos"] = f32(sd["position_embeddings.weight"])
    out["ln_g"], out["ln_b"] = f32(sd["LayerNorm.weight"]), f32(sd["LayerNorm.bias"])
    if "output_down_proj.0.weight" in sd:            # absent when hidden_dim == encoder hidden size (network.py:81-86)
        out["dn1_w"], out["dn1_b"] = bf(sd["output_down_proj.0.weight"]), f32(sd["output_down_proj.0.bias"])
        out["dn2_w"], out["dn2_b"] = bf(sd["output_down_proj.2.weight"]), f32(sd["output_down_proj.2.bias"])
    H = sd["LayerNorm.weight"].shape[0]
    scale = 1.0 / math.sqrt(H // num_heads)          # exact power of two for head dim 64: folding it into W_q is lossless
    i = 0
    while "input_transformers.layer.%d.attention.self.query.weight" % i in sd:
        p = "input_transformers.layer.%d." % i
        g = lambda k: sd[p + k].detach().float()
        out["l%d.wqkv" % i] = bf(torch.cat([g("attention.self.query.weight") * scale, g("attention.self.key.weight"),
                                            g("attention.self.value.weight")], dim=0))
        out["l%d.bqkv" % i] = f32(torch.cat([g("attention.self.query.bias") * scale, g("attention.self.key.bias"),
                                             g("attention.self.value.bias")], dim=0))
        out["l%d.wo" % i], out["l%d.bo" % i] = bf(g("attention.output.dense.weight")), f32(g("attention.output.dense.bias"))
        out["l%d.g1" % i], out["l%d.b1" % i] = f32(g("attention.output.LayerNorm.weight")), f32(g("attention.output.LayerNorm.bias"))
        out["l%d.w1" % i], out["l%d.bi" % i] = bf(g("intermediate.dense.weight")), f32(g("intermediate.dense.bias"))
        out["l%d.w2" % i], out["l%d.b2" % i] = bf(g("output.dense.weight")), f32(g("output.dense.bias"))
        out["l%d.g2" % i], out["l%d.b2n" % i] = f32(g("output.LayerNorm.weight")), f32(g("output.LayerNorm.bias"))
        i += 1
    return out


def write_pack(path, sd, config):
    """Pack `sd` (reference state dict) and write `path`.  `config`: dict with hidden_dim, hidden_t_dim, vocab_size, seq_len
    and the encoder sizes (hidden_size, num_hidden_layers, num_attention_heads, intermediate_size, layer_norm_eps)."""
    tensors = pack_tensors(sd, int(config["num_attention_heads"]))
    table, offset = [], 0
    for name, t in tensors.items():
        nbytes = t.numel() * t.element_size()
        table.append({"name": name, "dtype": str(t.dtype).replace("torch.", ""), "shape": list(t.shape), "offset": offset,
                      "nbytes": nbytes})
        offset += (nbytes + ALIGN - 1) // ALIGN * ALIGN
    header = json.dumps({"format": 1, "config": config, "tensors": table, "data_bytes": offset}).encode("utf-8")
    data_start = (len(MAGIC) + 8 + len(header) + ALIGN - 1) // ALIGN * ALIGN
    with open(path, "wb") as f:
        f.write(MAGIC)
        f.write(np.uint64(len(header)).tobytes())
        f.write(header)
        f.write(b"\0" * (data_start - f.tell()))
        for ent, t in zip(table, tensors.values()):
            raw = t.detach().cpu().contiguous().view(torch.uint8).numpy() if t.numel() else np.zeros(0, np.uint8)
            f.write(raw.tobytes())
            f.write(b"\0" * ((ent["nbytes"] + ALIGN - 1) // ALIGN * ALIGN - ent["nbytes"]))
    return path


def read_pack_header(path):
    with open(path, "rb") as f:
        if f.read(len(MAGIC)) != MAGIC:
            raise ValueError("%s is not a musediffusion_b200 weight pack" % path)
        n = int(np.frombuffer(f.read(8), dtype=np.uint64)[0])
        header = json.loads(f.read(n).decode("utf-8"))
    data_start = (len(MAGIC) + 8 + n + ALIGN - 1) // ALIGN * ALIGN
    return header, data_start


def load_pack(path, device):
    """-> (config dict, dict name -> tensor on `device`).  The tensor bytes are memory-mapped and copied to the device in
    ONE transfer; the returned tensors are views into that single buffer (256-byte aligned: TMA / vector-load safe)."""
    header, data_start = read_pack_header(path)
    mm = np.memmap(path, dtype=np.uint8, mode="r", offset=data_start, shape=(int(header["data_bytes"]),))
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)              # the mapping is read-only on purpose: it is only copied from
        buf = torch.from_numpy(np.asarray(mm)).to(device)          # one H2D copy straight from the page cache
    out = {}
    for ent in header["tensors"]:
        dt = _DTYPES[ent["dtype"]]
        flat = buf[ent["offset"]:ent["offset"] + ent["nbytes"]]
        out[ent["name"]] = flat.view(dt).view(ent["shape"])
    return header["config"], out


def model_config_of(args, model):
    """what `write_pack` records so that a pack can rebuild its model without training_args.json"""
    cfg = model.config
    return {"hidden_dim": model.input_dims, "hidden_t_dim": model.hidden_t_dim, "vocab_size": cfg.vocab_size,
            "seq_len": cfg.max_position_embeddings, "hidden_size": cfg.hidden_size, "num_hidden_layers": cfg.num_hidden_layers,
            "num_attention_heads": cfg.num_attention_heads, "intermediate_size": cfg.intermediate_size,
            "layer_norm_eps": cfg.layer_norm_eps,
            **{k: getattr(args, k) for k in ("diffusion_steps", "noise_schedule", "predict_xstart", "rescale_timesteps",
                                             "timestep_respacing", "dropout") if args is not None and hasattr(args, k)}}
