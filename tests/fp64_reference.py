"""The oracle's Moment-DETR forward and fine matching evaluated in float64.

TEST INFRASTRUCTURE ONLY.  A thin restatement, like tests/motion_oracle.py: the state dict and the inputs are cast to
float64 and handed to `oracle.cone_oracle.cone_forward` / `clip_matching` unchanged, with the layer counts of the
config (the oracle's own defaults are 2 / 2).  Two pieces stay fp32, as in torch's reference
(oracle/cone_oracle.py:156, 184): `position_embedding_sine` builds its table with `cumsum(dtype=float32)`, and the
key-padding mask is an fp32 -inf tensor.  Both are exact or are added to float64 values, so type promotion makes
everything after them float64: the only fp32 rounding left is that of the sine table itself.

With float32 inputs the functions return exactly the oracle's fp32 values (tests/test_config_matrix.py checks it).
"""
from __future__ import annotations

from typing import Dict

import torch

from oracle import cone_oracle as O


def cast_state_dict(sd: Dict[str, torch.Tensor], dtype=torch.float64) -> Dict[str, torch.Tensor]:
    return {k: v.detach().to("cpu", dtype) for k, v in sd.items()}


def cone_forward(sd, cfg, txt, tmask, vid, vmask, dtype=torch.float64) -> Dict[str, torch.Tensor]:
    """`O.cone_forward` on padded batches (masks 1 = valid) in `dtype`, with the config's layer counts."""
    c = lambda x: torch.as_tensor(x).to("cpu", dtype)
    with torch.no_grad():
        return O.cone_forward(cast_state_dict(sd, dtype), c(txt), c(tmask), c(vid), c(vmask), cfg.nheads,
                              cfg.enc_layers, cfg.dec_layers, cfg.n_input_proj)


def clip_matching(sd, cls, vid, vmask, spans, dtype=torch.float64) -> torch.Tensor:
    """`O.clip_matching` in `dtype` on the given proposals."""
    c = lambda x: torch.as_tensor(x).to("cpu", dtype)
    with torch.no_grad():
        return O.clip_matching(cast_state_dict(sd, dtype), c(cls), c(vid), c(vmask), c(spans))


def pool_slices(vid, start, end) -> torch.Tensor:
    """[B * nq, Dv] means of `vid[b][start[b, j]:end[b, j]]`, Python slices of the padded rows (a negative end counts back
    from the padded length; an empty slice gives NaN), in the dtype of `vid`: the pooling lines of `O.clip_matching`."""
    return torch.vstack([feat[s:e].mean(axis=0) for feat, ss, ee in zip(vid, start, end) for s, e in zip(ss, ee)])


def clip_matching_exact_bounds(sd, cls, vid, vmask, spans, dtype=torch.float64) -> torch.Tensor:
    """`O.clip_matching` with the [start, end) bounds computed as the fp32 reference computes them (`O.proposal_bounds` on
    the fp32 spans and mask), and the pooling, adapter, normalisation and dot product in `dtype`.  `clip_matching` above
    casts the spans first, so at a floor/ceil boundary it can pool other rows than the fp32 reference; this one pools the
    same rows.  In float32 it returns exactly `O.clip_matching`'s bits."""
    c = lambda x: torch.as_tensor(x).to("cpu", dtype)
    f32 = lambda x: torch.as_tensor(x).to("cpu", torch.float32)
    with torch.no_grad():
        start, end = O.proposal_bounds(f32(spans), f32(vmask))
        cls = c(cls)
        t = cls / cls.norm(dim=1, keepdim=True)
        p = O.adapter(cast_state_dict(sd, dtype), pool_slices(c(vid), start, end)).reshape(*start.shape, -1)
        p = p / p.norm(dim=2, keepdim=True)
        return torch.einsum("bld,bd->bl", p, t)
