"""The reference's `eval_epoch` stages 0-3 (`cone/inference.py:227-322`) over in-memory features, driven through
`ConeEngine`: host features -> pinned staging -> HBM -> kernels -> per-query predictions in the reference's
submission format (`postprocessing_format_mad`, inference.py:169-202)."""
from __future__ import annotations

import dataclasses
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from .config import ConeConfig
from .engine import ConeEngine, GroundingOutput, QueryBatch, host_feature_dtype, pack_queries

MODES = ("fusion", "proposal", "matching")  # order of GroundingOutput.nms[:, m]


@dataclasses.dataclass
class HostStep:
    """One step's inputs staged in pinned host memory."""
    frames: torch.Tensor  # [n_frames, Dv] fp32 or fp16 pinned
    qb: QueryBatch  # pinned
    video_ids: List[int]
    motion: Optional[torch.Tensor] = None  # [n_frames, Dm] fp32 or fp16 pinned: separate motion stream, None = `frames`

    def h2d_bytes(self) -> int:
        return (self.frames.numel() * self.frames.element_size() + self.qb.h2d_bytes() +
                (self.motion.numel() * self.motion.element_size() if self.motion is not None else 0))


def plan_steps(video_lengths: Sequence[int], queries, max_frames_per_step: int) -> List[List[int]]:
    """Group consecutive videos into steps of at most `max_frames_per_step` frames (>= 1 video each)."""
    steps, cur, tot = [], [], 0
    for v, L in enumerate(video_lengths):
        if cur and tot + L > max_frames_per_step:
            steps.append(cur)
            cur, tot = [], 0
        cur.append(v)
        tot += L
    if cur:
        steps.append(cur)
    return steps


def stage_step(cfg: ConeConfig, videos: Sequence[np.ndarray], queries, video_ids: Sequence[int], pin: bool = True,
               motion_videos: Optional[Sequence[np.ndarray]] = None) -> HostStep:
    """Concatenate the step's videos (and their motion features, when a separate motion stream is given) and pack
    its queries (dataset order preserved within the step).  float16 features stay float16, each stream on its own;
    a stream that mixes float16 with other types raises ValueError."""
    host_feature_dtype([videos[v] for v in video_ids], "videos")
    if motion_videos is not None:
        host_feature_dtype([motion_videos[v] for v in video_ids], "motion features")
    vid_set = {v: i for i, v in enumerate(video_ids)}
    sel = [(i, q) for i, q in enumerate(queries) if q.video_idx in vid_set]
    local = [dataclasses.replace(q, video_idx=vid_set[q.video_idx]) for _, q in sel]
    lens = [len(videos[v]) for v in video_ids]
    frames = torch.from_numpy(np.concatenate([videos[v] for v in video_ids], axis=0))
    motion = None
    if motion_videos is not None:
        for v in video_ids:  # both streams are sliced with the same window bounds: no silent truncation
            if len(motion_videos[v]) != len(videos[v]):
                raise ValueError(f"video {v}: {len(motion_videos[v])} motion rows for {len(videos[v])} appearance rows")
        motion = torch.from_numpy(np.concatenate([motion_videos[v] for v in video_ids], axis=0))
    qb = pack_queries(cfg, lens, local, dataset_indices=[i for i, _ in sel])
    if pin and torch.cuda.is_available():
        frames = frames.pin_memory()
        motion = motion.pin_memory() if motion is not None else None
        qb = qb.pin()
    return HostStep(frames, qb, list(video_ids), motion)


def run_step(engine: ConeEngine, step: HostStep, want_rows: bool = False) -> GroundingOutput:
    """H2D of the step's inputs (async from pinned memory) + the whole device path."""
    dev = engine.device
    with torch.cuda.device(dev):
        frames = step.frames.to(dev, non_blocking=True)
        motion = step.motion.to(dev, non_blocking=True) if step.motion is not None else None
        qb = step.qb.to(dev)
        return engine.ground(frames, qb, want_rows=want_rows, motion=motion)


def output_to_host(cfg: ConeConfig, step: HostStep, out: GroundingOutput, full: bool = True) -> Dict[str, dict]:
    """D2H + conversion to per-query Python structures (same layout as the oracle's `eval_pipeline`)."""
    nms = out.nms.cpu().numpy()
    cnt = out.nms_count.cpu().numpy()
    res: Dict[str, dict] = {}
    if full:
        rl = out.ranklist.cpu().numpy()
        ws, wl = out.win_start.cpu().numpy(), out.win_len.cpu().numpy()
        sp, pr, mt = out.pred_spans.cpu().numpy(), out.prob_fg.cpu().numpy(), out.match.cpu().numpy()
        rows = out.rows.cpu().numpy() if out.rows is not None else None
        rcnt = out.rows_count.cpu().numpy() if out.rows_count is not None else None
    for j, qid in enumerate(step.qb.query_ids):
        r = {m: nms[j, i, : cnt[j, i]].tolist() for i, m in enumerate(MODES)}
        if full:
            n_win = int((wl[j] > 0).sum())
            r["ranklist"] = [int(x) for x in rl[j] if x >= 0]
            r["windows"] = [(int(ws[j, t]), int(wl[j, t])) for t in range(n_win)]
            r["pred_spans"] = sp[j, :n_win]
            r["prob_fg"] = pr[j, :n_win]
            r["match"] = mt[j, :n_win]
            if rows is not None:
                r["rows"] = rows[j, : rcnt[j]].tolist()
        res[qid] = r
    return res


def ground_dataset(engine: ConeEngine, videos: Sequence[np.ndarray], queries, max_frames_per_step: int = 1 << 20,
                   full: bool = True, want_rows: bool = True,
                   motion_videos: Optional[Sequence[np.ndarray]] = None) -> Dict[str, dict]:
    """Stages 0-3 over a whole in-memory dataset.  Videos are processed in steps of consecutive videos; the
    reference pools proposals over windows padded to the longest window of each `eval_bsz` batch of queries
    (SURVEY.md §8 A9), which is reproduced exactly when a step holds whole eval batches (always true for a
    single step).  `motion_videos[v]` [L_v, Dm]: raw features of a separate motion stream (`--motion_feat_dir`), the
    input of Moment-DETR; None = the appearance features serve both roles.  Videos, motion features and queries may
    each be float32 or float16 (one type per stream): float16 is staged, copied and read as such, and the results are
    bitwise those of the float32 upcast."""
    _check_streams(videos, motion_videos, queries)
    res: Dict[str, dict] = {}
    lens = [len(v) for v in videos]
    for ids in plan_steps(lens, queries, max_frames_per_step):
        step = stage_step(engine.cfg, videos, queries, ids, motion_videos=motion_videos)
        if step.qb.tok_len.numel() == 0:
            continue
        out = run_step(engine, step, want_rows=want_rows)
        res.update(output_to_host(engine.cfg, step, out, full=full))
    return res


def _check_streams(videos, motion_videos, queries) -> None:
    if motion_videos is not None and len(motion_videos) != len(videos):
        raise ValueError(f"{len(motion_videos)} motion feature tensors for {len(videos)} videos")
    host_feature_dtype(videos, "videos")  # before any step runs
    if motion_videos is not None:
        host_feature_dtype(motion_videos, "motion features")
    host_feature_dtype([q.tokens for q in queries] + [q.cls for q in queries], "queries")


def to_submission(results: Dict[str, dict], annotations: Sequence[dict], mode: str = "fusion") -> List[dict]:
    """The reference's MAD submission rows (inference.py:169-202): one dict per query, dataset order."""
    return [dict(query_id=a["query_id"], video_id=a["video_id"], predicted_times=results[a["query_id"]][mode])
            for a in annotations]


def recall_at_k(results: Dict[str, dict], gt: Dict[str, Sequence[float]], mode: str = "fusion",
                thresholds=(0.3, 0.5), topk=(1, 5)) -> np.ndarray:
    """R@K at IoU thresholds over the NMS'd predictions — the metric of standalone_eval/evaluate_mad.py:60-104
    (hull IoU in fp32, strict `>`), computed from the kernel outputs on the host."""
    rec = np.zeros((len(topk), len(thresholds)))
    thr = np.asarray(thresholds, dtype=np.float32)
    for qid, r in results.items():
        rows = np.asarray(r[mode], dtype=np.float64)
        if rows.size == 0:
            continue
        st, ed = rows[: max(topk), 0].astype(np.float32), rows[: max(topk), 1].astype(np.float32)
        g0, g1 = np.float32(gt[qid][0]), np.float32(gt[qid][1])
        inter = np.maximum(np.minimum(ed, g1) - np.maximum(st, g0), np.float32(0))
        hull = np.maximum(ed, g1) - np.minimum(st, g0)
        hit = (inter / hull)[:, None] > thr[None, :]
        for i, k in enumerate(topk):
            rec[i] += hit[:k].any(axis=0)
    return rec / max(len(results), 1)


@dataclasses.dataclass
class MetricCounters:
    """Device-side metric state accumulated over steps (and summed over ranks by `sharding.reduce_counters`)."""
    topk: Sequence[int]
    thresholds: Sequence[float]
    window_topk: Sequence[int]
    hits: torch.Tensor  # [3, len(topk), len(thresholds)] int64, rankings in MODES order
    window_hits: torch.Tensor  # [len(window_topk)] int64
    n_queries: torch.Tensor  # [1] int64
    top1_iou: List[torch.Tensor] = dataclasses.field(default_factory=list)  # per step [Nq, 3] fp64 (Ego4D mIoU)

    def recall_mad(self, mode: str = "fusion") -> np.ndarray:
        """`evaluate_mad.evaluate_nlq_performance`'s table [len(topk), len(thresholds)]: float32 counters divided
        by the number of queries in float32, as `recall_x_iou /= len(submission)` does."""
        h = self.hits[MODES.index(mode)].cpu().numpy().astype(np.float32)
        return h / np.float32(max(int(self.n_queries.item()), 1))

    def recall_ego4d(self, mode: str = "fusion"):
        """`evaluate_ego4d_nlq.evaluate_nlq_performance`: (recall [len(thresholds), len(topk)] float64, mIoU)."""
        m = MODES.index(mode)
        n = max(int(self.n_queries.item()), 1)
        rec = self.hits[m].cpu().numpy().astype(np.float64).T / n
        iou = torch.cat([t[:, m] for t in self.top1_iou]).cpu().numpy() if self.top1_iou else np.zeros(0)
        with np.errstate(invalid="ignore"):
            return rec, float(np.mean(iou)) if iou.size else float("nan")

    def window_recall(self) -> np.ndarray:
        return self.window_hits.cpu().numpy().astype(np.float32) / np.float32(max(int(self.n_queries.item()), 1))


def new_counters(device, topk=(1, 5), thresholds=(0.3, 0.5), window_topk=(1, 5, 10, 30, 50)) -> MetricCounters:
    return MetricCounters(tuple(topk), tuple(thresholds), tuple(window_topk),
                          torch.zeros((3, len(topk), len(thresholds)), dtype=torch.int64, device=device),
                          torch.zeros((len(window_topk),), dtype=torch.int64, device=device),
                          torch.zeros((1,), dtype=torch.int64, device=device))


def accumulate_metrics(engine: ConeEngine, counters: MetricCounters, step: HostStep, out: GroundingOutput,
                       gt: Dict[str, Sequence[float]], flavour: str = "mad") -> None:
    """Adds one step's hits to `counters` on the device: no prediction leaves the GPU (SURVEY.md §8(f)1)."""
    g = torch.tensor([[float(gt[q][0]), float(gt[q][1])] for q in step.qb.query_ids], dtype=torch.float64)
    g = g.reshape(-1, 2).to(engine.device, non_blocking=True)
    _, top1 = engine.eval_recall(out.nms, out.nms_count, g, counters.topk, counters.thresholds, flavour,
                                 hits=counters.hits, want_top1=(flavour == "ego4d"))
    if top1 is not None:
        counters.top1_iou.append(top1)
    engine.eval_window_recall(out.ranklist, g, counters.window_topk, hits=counters.window_hits)
    counters.n_queries += g.shape[0]


def evaluate_dataset(engine: ConeEngine, videos: Sequence[np.ndarray], queries, gt: Dict[str, Sequence[float]],
                     flavour: str = "mad", topk=(1, 5), thresholds=(0.3, 0.5), window_topk=(1, 5, 10, 30, 50),
                     max_frames_per_step: int = 1 << 20, video_ids: Optional[Sequence[int]] = None,
                     motion_videos: Optional[Sequence[np.ndarray]] = None) -> MetricCounters:
    """Stages 0-3 + metric counters over (this rank's share of) a dataset; only the counters are read back.
    `motion_videos` as in `ground_dataset`."""
    _check_streams(videos, motion_videos, queries)
    counters = new_counters(engine.device, topk, thresholds, window_topk)
    lens = [len(v) for v in videos]
    mine = None if video_ids is None else set(video_ids)
    for ids in plan_steps(lens, queries, max_frames_per_step):
        ids = [v for v in ids if mine is None or v in mine]
        if not ids:
            continue
        step = stage_step(engine.cfg, videos, queries, ids, motion_videos=motion_videos)
        if step.qb.tok_len.numel() == 0:
            continue
        out = run_step(engine, step)
        accumulate_metrics(engine, counters, step, out, gt, flavour)
    return counters
