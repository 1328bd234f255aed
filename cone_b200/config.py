"""Hot-path knobs of CONE's coarse-to-fine inference, as plain function arguments.

The reference carries these in an argparse namespace (`cone/config.py:56-125`,
values fixed per dataset in `cone/scripts/train_{ego4d,mad}.sh`).  Only the
fields the inference path reads are kept (SURVEY.md §8c lists them).
"""
from __future__ import annotations

import dataclasses
import math


@dataclasses.dataclass(frozen=True)
class ConeConfig:
    # feature dims (cone/config.py `--v_appear_feat_dim`, `--t_feat_dim`, `--v_motion_feat_dim`); a motion dim of 0
    # means one feature source serves both roles (the reference's released configs)
    v_feat_dim: int = 256
    t_feat_dim: int = 768
    v_motion_feat_dim: int = 0
    # model (cone/config.py:101-125)
    hidden_dim: int = 256
    nheads: int = 8
    dim_feedforward: int = 1024
    enc_layers: int = 2
    dec_layers: int = 2
    num_queries: int = 5
    n_input_proj: int = 2
    # data / windows (cone/config.py:73-75, :56, :59)
    max_v_l: int = 90
    max_q_l: int = 20
    clip_length: float = 0.53333
    topk_window: int = 20
    eval_bsz: int = 32
    # post-processing (cone/config.py:157-159)
    nms_thd: float = 0.5
    max_before_nms: int = 200
    max_after_nms: int = 5
    name: str = "ego4d"

    @property
    def motion_dim(self) -> int:
        """Input width of `input_vid_proj`: the motion feature dim, `v_feat_dim` when no separate stream is set."""
        return self.v_motion_feat_dim or self.v_feat_dim

    @property
    def stride(self) -> int:
        """window stride = half a window (`cone/inference.py:272`)."""
        return int(self.max_v_l / 2)

    def num_window(self, ctx_l: int) -> int:
        """`cone/inference.py:286`."""
        return math.ceil(ctx_l / self.stride) + 1

    def window_bounds(self, i: int, ctx_l: int) -> tuple[int, int]:
        """[start, end) frame range of window `i` (`cone/inference.py:291-292`)."""
        s = max((i - 1) * self.stride, 0)
        e = min((i - 1) * self.stride + self.max_v_l, ctx_l)
        return s, e

    def replace(self, **kw) -> "ConeConfig":
        return dataclasses.replace(self, **kw)


# BASELINE.json configs[0]/[1]: Ego4D-NLQ shape (train_ego4d.sh:12-14,22-32)
EGO4D = ConeConfig(v_feat_dim=256, t_feat_dim=768, max_v_l=90, max_q_l=20, clip_length=0.53333,
                   topk_window=20, eval_bsz=32, name="ego4d")
# reference scripts' MAD shape (train_mad.sh:12-14,23-25,36; README.md:149)
MAD512 = ConeConfig(v_feat_dim=512, t_feat_dim=512, max_v_l=125, max_q_l=25, clip_length=0.2,
                    topk_window=30, eval_bsz=16, name="mad512")
# BASELINE.json configs[2]: "CLIP 768-d video at 5 fps ... topk_window=30"
MAD768 = ConeConfig(v_feat_dim=768, t_feat_dim=768, max_v_l=125, max_q_l=25, clip_length=0.2,
                    topk_window=30, eval_bsz=16, name="mad768")

PRESETS = {"ego4d": EGO4D, "mad512": MAD512, "mad768": MAD768}
