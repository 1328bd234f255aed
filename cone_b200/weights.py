"""State-dict layout of the reference `CONE` module and a deterministic random initialiser.

The key names and shapes are exactly those of `checkpoint["model"]` as saved by
`cone/train.py:184-223` and loaded by `cone/inference.py:525-528` (SURVEY.md §8b), so a
reference checkpoint loads into this package unchanged and a state dict made here loads into
the reference `CONE` (`oracle/ref_harness.py` does exactly that to make the golden vectors).
"""
from __future__ import annotations

import math
from collections import OrderedDict

import torch

from .config import ConeConfig


def state_dict_shapes(cfg: ConeConfig) -> "OrderedDict[str, tuple]":
    """name -> shape for every tensor in the reference model's state dict."""
    d, ff = cfg.hidden_dim, cfg.dim_feedforward
    dv, dt = cfg.v_feat_dim, cfg.t_feat_dim
    s: "OrderedDict[str, tuple]" = OrderedDict()

    def attn(prefix):
        s[prefix + ".in_proj_weight"] = (3 * d, d)
        s[prefix + ".in_proj_bias"] = (3 * d,)
        s[prefix + ".out_proj.weight"] = (d, d)
        s[prefix + ".out_proj.bias"] = (d,)

    def ffn_norms(prefix, n_norm):
        s[prefix + ".linear1.weight"] = (ff, d)
        s[prefix + ".linear1.bias"] = (ff,)
        s[prefix + ".linear2.weight"] = (d, ff)
        s[prefix + ".linear2.bias"] = (d,)
        for i in range(1, n_norm + 1):
            s[f"{prefix}.norm{i}.weight"] = (d,)
            s[f"{prefix}.norm{i}.bias"] = (d,)

    for i in range(cfg.enc_layers):  # cone/transformer.py:213-228
        p = f"transformer.encoder.layers.{i}"
        attn(p + ".self_attn")
        ffn_norms(p, 2)
    for i in range(cfg.dec_layers):  # cone/transformer.py:272-292
        p = f"transformer.decoder.layers.{i}"
        attn(p + ".self_attn")
        attn(p + ".multihead_attn")
        ffn_norms(p, 3)
    s["transformer.decoder.norm.weight"] = (d,)  # cone/transformer.py:35
    s["transformer.decoder.norm.bias"] = (d,)
    # cone/position_encoding.py:14-16 (constructed, unused unless --use_txt_pos)
    s["txt_position_embed.position_embeddings.weight"] = (cfg.max_q_l, d)
    s["txt_position_embed.LayerNorm.weight"] = (d,)
    s["txt_position_embed.LayerNorm.bias"] = (d,)
    for i, (a, b) in enumerate([(d, d), (d, d), (d, 2)]):  # span_embed = MLP(d,d,2,3) model.py:49
        s[f"span_embed.layers.{i}.weight"] = (b, a)
        s[f"span_embed.layers.{i}.bias"] = (b,)
    s["class_embed.weight"] = (2, d)  # model.py:50
    s["class_embed.bias"] = (2,)
    s["query_embed.weight"] = (cfg.num_queries, d)  # model.py:54
    # model.py:57-72; input_vid_proj reads the motion features (`--v_motion_feat_dim`), the adapter the appearance ones
    for name, din in (("input_txt_proj", dt), ("input_vid_proj", cfg.motion_dim)):
        for i in range(cfg.n_input_proj):
            k = din if i == 0 else d
            s[f"{name}.{i}.LayerNorm.weight"] = (k,)
            s[f"{name}.{i}.LayerNorm.bias"] = (k,)
            s[f"{name}.{i}.net.1.weight"] = (d, k)
            s[f"{name}.{i}.net.1.bias"] = (d,)
    s["saliency_proj.weight"] = (1, d)  # model.py:74
    s["saliency_proj.bias"] = (1,)
    s["adapter_layer.layers.0.weight"] = (d, dv)  # MLP(dv, d, dv, 2) model.py:80
    s["adapter_layer.layers.0.bias"] = (d,)
    s["adapter_layer.layers.1.weight"] = (dv, d)
    s["adapter_layer.layers.1.bias"] = (dv,)
    return s


def init_state_dict(cfg: ConeConfig, seed: int = 0, perturb: bool = True,
                    head_gain: float = 12.0, attn_gain: float = 2.0) -> "OrderedDict[str, torch.Tensor]":
    """Random fp32 state dict, deterministic in (cfg, seed).

    Matrices follow the reference's initial distributions (xavier-uniform inside
    `transformer.*`, `cone/transformer.py:44-47`; U(±1/sqrt(fan_in)) for other Linear layers;
    N(0,1) embeddings).  With `perturb=True` LayerNorm gains/offsets and attention biases are
    also randomised (the reference initialises them to 1/0/0) so that a kernel that drops a
    gain, an offset or a bias cannot pass parity by accident; the q/k projections are scaled by
    `attn_gain`, the slot embeddings by 2 and the last span-head matrix by `head_gain` (with a
    negative width offset) — a freshly initialised model emits (0.5, 0.5) for every proposal,
    which would make pooling, fusion and NMS degenerate.  The result is shaped like a trained
    checkpoint rather than a fresh one; `perturb=False` gives the reference's own fresh init.
    """
    g = torch.Generator(device="cpu")
    g.manual_seed(1_000_003 * (seed + 1))
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    for name, shape in state_dict_shapes(cfg).items():
        is_norm = ".norm" in name or "LayerNorm" in name
        if is_norm:
            if name.endswith("weight"):
                t = torch.ones(shape)
                if perturb:
                    t = t + 0.1 * torch.randn(shape, generator=g)
            else:
                t = torch.zeros(shape)
                if perturb:
                    t = 0.1 * torch.randn(shape, generator=g)
        elif name in ("query_embed.weight", "txt_position_embed.position_embeddings.weight"):
            t = torch.randn(shape, generator=g)  # nn.Embedding default
            if perturb and name == "query_embed.weight":
                t = t * 2.0
        elif len(shape) == 2:
            fan_out, fan_in = shape
            if name.startswith("transformer."):
                # xavier-uniform; torch applies it to the packed (3d, d) in_proj as one matrix
                bound = math.sqrt(6.0 / (fan_in + fan_out))
            else:
                bound = 1.0 / math.sqrt(fan_in)
            t = (torch.rand(shape, generator=g) * 2 - 1) * bound
            if perturb and name == "span_embed.layers.2.weight":
                t = t * head_gain  # spread the sigmoid outputs so the 5 proposals differ
            if perturb and name.endswith("in_proj_weight"):
                t[: 2 * fan_in] *= attn_gain  # sharper attention: slots attend to different frames
        else:  # biases
            if name.endswith("in_proj_bias") or name.endswith("out_proj.bias"):
                t = torch.zeros(shape)
                if perturb:
                    t = 0.05 * torch.randn(shape, generator=g)
            else:
                # fan_in of the matching weight
                wname = name[: -len("bias")] + "weight"
                fan_in = state_dict_shapes(cfg)[wname][1]
                t = (torch.rand(shape, generator=g) * 2 - 1) / math.sqrt(fan_in)
                if perturb and name == "span_embed.layers.2.bias":
                    t[1] -= 1.5  # narrower proposals, as a trained head gives
        sd[name] = t.to(torch.float32).contiguous()
    return sd


def check_state_dict(cfg: ConeConfig, sd) -> None:
    """Raise if `sd` is not a reference-shaped CONE state dict for `cfg`."""
    want = state_dict_shapes(cfg)
    missing = [k for k in want if k not in sd]
    if missing:
        raise KeyError(f"state dict lacks {len(missing)} tensors, e.g. {missing[:3]}")
    for k, shp in want.items():
        if tuple(sd[k].shape) != tuple(shp):
            raise ValueError(f"{k}: shape {tuple(sd[k].shape)} != expected {shp}")
