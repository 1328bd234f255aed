"""Seeded synthetic inputs of the shapes the reference path consumes (SURVEY.md §8d).

What the reference reads from LMDB (`cone/ego4d_mad_dataloader.py:258-302, 453-473`):
per video a raw frame-feature matrix `features [L, Dv]`; per query `token_features
[n_tok, Dt]` and a holistic `cls_features [Dv]`.  Annotations are the jsonl rows of
`StartEndDataset` (`ego4d_mad_dataloader.py:19-29`): query_id, clip_id, timestamps, duration.
"""
from __future__ import annotations

import dataclasses
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np

from .config import ConeConfig


@dataclasses.dataclass
class SynthQuery:
    query_id: str
    video_idx: int
    tokens: np.ndarray  # [n_tok, Dt] float32, raw (not truncated, not normalised)
    cls: np.ndarray  # [Dv] float32, raw
    timestamps: Tuple[float, float]  # ground-truth span in seconds


@dataclasses.dataclass
class SynthDataset:
    cfg: ConeConfig
    videos: List[np.ndarray]  # each [L_v, Dv] float32, raw
    queries: List[SynthQuery]  # grouped by video, in video order
    motion: Optional[List[np.ndarray]] = None  # each [L_v, Dm] float32, raw: a separate motion stream

    @property
    def video_ids(self) -> List[str]:
        return [f"video{v:05d}" for v in range(len(self.videos))]

    def annotations(self) -> List[dict]:
        """jsonl rows in the reference's annotation format."""
        vids = self.video_ids
        return [dict(query_id=q.query_id, query=f"synthetic query {i}", video_id=vids[q.video_idx],
                     clip_id=vids[q.video_idx], timestamps=[float(q.timestamps[0]), float(q.timestamps[1])],
                     duration=float(len(self.videos[q.video_idx]) * self.cfg.clip_length))
                for i, q in enumerate(self.queries)]


def make_dataset(cfg: ConeConfig, n_videos: int, frames: Union[int, Sequence[int], None],
                 queries_per_video: Union[int, Sequence[int]], seed: int = 0, plant: float = 0.5,
                 id_offset: int = 0, frames_range: Union[Tuple[int, int], None] = None,
                 motion_dim: Optional[int] = None) -> SynthDataset:
    """`frames`: one L for every video or an explicit per-video list; or `frames_range=(lo, hi)`
    to draw each video's length uniformly.  `motion_dim`: also draw a separate motion stream of that width, same
    lengths, from its own generator (the appearance features and queries do not change)."""
    rng = np.random.default_rng(seed)
    if frames_range is not None:
        lens = [int(x) for x in rng.integers(frames_range[0], frames_range[1] + 1, size=n_videos)]
    elif isinstance(frames, int):
        lens = [frames] * n_videos
    else:
        lens = [int(x) for x in frames]
        assert len(lens) == n_videos
    if isinstance(queries_per_video, int):
        nq = [queries_per_video] * n_videos
    else:
        nq = [int(x) for x in queries_per_video]
        assert len(nq) == n_videos
    videos: List[np.ndarray] = []
    queries: List[SynthQuery] = []
    for v in range(n_videos):
        L = lens[v]
        x = rng.standard_normal((L, cfg.v_feat_dim), dtype=np.float32)
        for j in range(nq[v]):
            n_tok = int(rng.integers(4, cfg.max_q_l + 6))  # > max_q_l exercises truncation
            tok = rng.standard_normal((n_tok, cfg.t_feat_dim), dtype=np.float32)
            cls = rng.standard_normal((cfg.v_feat_dim,), dtype=np.float32)
            dur_s = L * cfg.clip_length
            span_s = float(rng.uniform(2.0, 30.0))
            span_s = min(span_s, dur_s)
            st = float(rng.uniform(0.0, max(dur_s - span_s, 0.0)))
            ed = st + span_s
            if plant:
                f0 = int(st / cfg.clip_length)
                f1 = max(int(np.ceil(ed / cfg.clip_length)), f0 + 1)
                x[f0:f1] += np.float32(plant) * cls[None, :]
            queries.append(SynthQuery(f"v{v + id_offset:05d}_{j}", v, tok, cls, (st, ed)))
        videos.append(x)
    motion = None
    if motion_dim:
        mrng = np.random.default_rng([seed, 1])
        # a per-video offset and scale: the motion rows are not centred like the appearance rows
        motion = [(mrng.standard_normal((len(x), motion_dim), dtype=np.float32) * np.float32(mrng.uniform(0.5, 3.0))
                   + np.float32(mrng.uniform(-0.5, 0.5))) for x in videos]
    return SynthDataset(cfg, videos, queries, motion)
