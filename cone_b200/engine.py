"""Host-side runtime over the C ABI: owns the weights handle and the workspace, exposes each stage of the
reference path (`cone/inference.py:227-322`) as a method on device tensors, and the whole path as
`ground()`.  PyTorch is used for device memory and streams only."""
from __future__ import annotations

import ctypes as C
import dataclasses
import math
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from .config import ConeConfig
from .weights import check_state_dict, state_dict_shapes


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


# storage types a raw feature tensor (frames, motion rows, tokens, CLS) may have; results are those of `t.float()`
FEATURE_DTYPES = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16, torch.bfloat16: _lib.DTYPE_BF16}


def _need_feature(t: torch.Tensor, name: str):
    """(contiguous t, its CONE_DTYPE_* code) for a raw feature tensor."""
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if t.dtype not in FEATURE_DTYPES:
        raise TypeError(f"{name} must be float32, float16 or bfloat16, got {t.dtype}")
    return t.contiguous(), FEATURE_DTYPES[t.dtype]


def host_feature_dtype(arrays, what: str) -> np.dtype:
    """Storage type of a set of host feature arrays that are staged together: float16 when every array is float16,
    else float32 (other float types are converted as before).  A mix of float16 and other types raises ValueError:
    concatenating them would silently promote the float16 ones."""
    kinds = {np.asarray(a).dtype == np.float16 for a in arrays}
    if len(kinds) > 1:
        raise ValueError(f"{what} mix float16 and float32 features: cast them to one dtype")
    return np.dtype(np.float16 if kinds == {True} else np.float32)


@dataclasses.dataclass
class QueryBatch:
    """Queries of a set of videos, grouped by video (the order the kernels run in).  `order[i]` is the
    dataset index of the i-th packed query, so results can be scattered back."""
    video_offsets: torch.Tensor  # [Nv+1] int64, frame offset of each video in the concatenated frame tensor
    q_first: torch.Tensor  # [Nv+1] int32, first packed query of each video
    q_video_start: torch.Tensor  # [Nq] int64
    q_video_len: torch.Tensor  # [Nq] int32
    tokens: torch.Tensor  # [Nq, max_q_l, Dt] raw (fp32, fp16 or bf16), zero padded (truncated to max_q_l)
    tok_len: torch.Tensor  # [Nq] int32
    cls: torch.Tensor  # [Nq, Dv] raw (fp32, fp16 or bf16)
    q_batch: torch.Tensor  # [Nq] int32 reference eval-batch id (dataset index // eval_bsz)
    n_batches: int
    max_video_frames: int
    max_video_queries: int
    total_scores: int  # sum over videos of (#queries x #frames): size of the ragged frame-score buffer
    order: np.ndarray  # [Nq] dataset index of each packed query
    query_ids: List[str]  # packed order

    def to(self, device, non_blocking=True) -> "QueryBatch":
        kw = {f.name: (getattr(self, f.name).to(device, non_blocking=non_blocking)
                       if isinstance(getattr(self, f.name), torch.Tensor) else getattr(self, f.name))
              for f in dataclasses.fields(self)}
        return QueryBatch(**kw)

    def pin(self) -> "QueryBatch":
        kw = {f.name: (getattr(self, f.name).pin_memory() if isinstance(getattr(self, f.name), torch.Tensor)
                       else getattr(self, f.name)) for f in dataclasses.fields(self)}
        return QueryBatch(**kw)

    def record_stream(self, stream) -> None:
        """Tell the caching allocator that `stream` uses these tensors (they were copied on a side stream)."""
        for f in dataclasses.fields(self):
            t = getattr(self, f.name)
            if isinstance(t, torch.Tensor) and t.is_cuda:
                t.record_stream(stream)

    def h2d_bytes(self) -> int:
        return sum(getattr(self, f.name).numel() * getattr(self, f.name).element_size()
                   for f in dataclasses.fields(self) if isinstance(getattr(self, f.name), torch.Tensor))


def pack_queries(cfg: ConeConfig, video_lengths: Sequence[int], queries, first_dataset_index: int = 0,
                 dataset_indices: Optional[Sequence[int]] = None) -> QueryBatch:
    """Host tensors for a list of queries (objects with query_id, video_idx, tokens, cls) in DATASET order.

    `dataset_indices[i]` is the position of `queries[i]` in the whole dataset: the reference's DataLoader forms its
    eval batches from consecutive DATASET indices (`cone/inference.py:306-315`), and a proposal is pooled over
    windows padded to the longest window of its eval batch (SURVEY.md §8 A9), so the batch id of a query must come
    from its true index even when a step holds a non-contiguous selection (annotations not grouped by video, or a
    rank's share of a multi-video step).  Default: the queries are consecutive from `first_dataset_index`."""
    nq = len(queries)
    if dataset_indices is None:
        ds_idx = np.arange(nq, dtype=np.int64) + int(first_dataset_index)
    else:
        ds_idx = np.asarray(dataset_indices, dtype=np.int64)
        if ds_idx.shape != (nq,):
            raise ValueError(f"dataset_indices must have one entry per query ({nq}), got shape {ds_idx.shape}")
    batch_of, dense = np.unique(ds_idx // cfg.eval_bsz, return_inverse=True) if nq else (np.zeros(0), np.zeros(0, np.int64))
    order = np.argsort(np.asarray([q.video_idx for q in queries], dtype=np.int64), kind="stable")
    offs = np.zeros(len(video_lengths) + 1, dtype=np.int64)
    offs[1:] = np.cumsum(np.asarray(video_lengths, dtype=np.int64))
    vid = np.asarray([queries[i].video_idx for i in order], dtype=np.int64)
    q_first = np.searchsorted(vid, np.arange(len(video_lengths) + 1)).astype(np.int32)
    # float16 queries stay float16 (zero padded in float16): the device converts them on load
    fdt = host_feature_dtype([q.tokens for q in queries] + [q.cls for q in queries], "queries")
    tokens = np.zeros((nq, cfg.max_q_l, cfg.t_feat_dim), dtype=fdt)
    tok_len = np.zeros(nq, dtype=np.int32)
    cls = np.zeros((nq, cfg.v_feat_dim), dtype=fdt)
    for j, i in enumerate(order):
        q = queries[i]
        t = q.tokens[: cfg.max_q_l]  # `q_feat[:self.max_q_l]` (dataloader:272)
        tokens[j, : len(t)] = t
        tok_len[j] = len(t)
        cls[j] = q.cls
    per_video = np.diff(q_first)
    return QueryBatch(
        video_offsets=torch.from_numpy(offs), q_first=torch.from_numpy(q_first),
        q_video_start=torch.from_numpy(offs[vid]), q_video_len=torch.from_numpy(np.diff(offs)[vid].astype(np.int32)),
        tokens=torch.from_numpy(tokens), tok_len=torch.from_numpy(tok_len), cls=torch.from_numpy(cls),
        q_batch=torch.from_numpy(np.asarray(dense, dtype=np.int64).reshape(-1)[order].astype(np.int32)),
        n_batches=max(int(len(batch_of)), 1),
        max_video_frames=int(max(video_lengths)) if len(video_lengths) else 0,
        max_video_queries=int(per_video.max()) if nq else 0,
        total_scores=int((per_video.astype(np.int64) * np.diff(offs)).sum()), order=order,
        query_ids=[queries[i].query_id for i in order])


@dataclasses.dataclass
class GroundingOutput:
    """Device results of `ConeEngine.ground`, packed-query order."""
    ranklist: torch.Tensor  # [Nq, stride] int32, -1 padded
    win_start: torch.Tensor  # [Nq, k] int32 (frame index inside the video)
    win_len: torch.Tensor  # [Nq, k] int32, 0 = absent
    pred_spans: torch.Tensor  # [Nq, k, nq, 2]
    prob_fg: torch.Tensor  # [Nq, k, nq]
    match: torch.Tensor  # [Nq, k, nq]
    nms: torch.Tensor  # [Nq, 3, max_after, 5] fp64 rows [st, ed, score, match, fusion]; 0 fusion 1 proposal 2 matching
    nms_count: torch.Tensor  # [Nq, 3] int32
    rows: Optional[torch.Tensor] = None  # [Nq, k*nq, 4] fp64
    rows_count: Optional[torch.Tensor] = None

    def d2h_bytes(self) -> int:
        return self.nms.numel() * 8 + self.nms_count.numel() * 4


class ConeEngine:
    """Weights + workspace + the kernels of the coarse-to-fine path on one GPU."""

    def __init__(self, cfg: ConeConfig, state_dict: Dict[str, torch.Tensor], device="cuda:0", precision: str = "fp32",
                 workspace_bytes: int = 4 << 30):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.ConeError("cone_b200 needs a CUDA device (there is no CPU path)")
        self.cfg = cfg
        self.device = torch.device(device)
        self.precision = {"fp32": _lib.PREC_FP32, "tc": _lib.PREC_TC, "bf16": _lib.PREC_TC}[precision]
        self.dims = _lib.ConeDims(cfg.v_feat_dim, cfg.t_feat_dim, cfg.hidden_dim, cfg.nheads, cfg.dim_feedforward,
                                  cfg.enc_layers, cfg.dec_layers, cfg.num_queries, cfg.max_v_l, cfg.max_q_l,
                                  cfg.v_motion_feat_dim)
        self._handle = C.c_void_p(0)
        self._ws = None
        with torch.cuda.device(self.device):
            self.load_state_dict(state_dict)
            self.reserve(workspace_bytes)

    # ---- weights ------------------------------------------------------------------------------
    def load_state_dict(self, state_dict) -> None:
        check_state_dict(self.cfg, state_dict)
        blob = torch.cat([state_dict[k].detach().to("cpu", torch.float32).reshape(-1)
                          for k in state_dict_shapes(self.cfg)]).contiguous()
        want = self.lib.cone_weights_expected_floats(C.byref(self.dims))
        if want == 0:
            _lib.check(-1, "cone_weights_expected_floats")
        assert blob.numel() == want, (blob.numel(), want)
        if self._handle:  # live weights: rewrite the existing handle in place (pointers and captured graphs stay valid)
            with torch.cuda.device(self.device):
                _lib.check(self.lib.cone_weights_update(self._handle, C.c_void_p(blob.data_ptr()), blob.numel(), _stream()),
                           "cone_weights_update")
            return
        new = C.c_void_p(0)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.cone_weights_create(C.c_void_p(blob.data_ptr()), blob.numel(), C.byref(self.dims),
                                                    _stream(), C.byref(new)), "cone_weights_create")
        self._handle = new

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                self.lib.cone_weights_destroy(self._handle)
                self._handle = C.c_void_p(0)
        except Exception:
            pass

    def reserve(self, nbytes: int) -> None:
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = None
            self._ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)

    def _wsargs(self, need: int = 0):
        if need:
            self.reserve(need)
        return _ptr(self._ws), self._ws.numel()

    # ---- stage kernels ------------------------------------------------------------------------
    def l2_normalize(self, x: torch.Tensor, eps: float) -> torch.Tensor:
        """x / (||x|| + eps) per row (eps < 0: x / max(||x||, -eps)); x fp32, fp16 or bf16, the result fp32."""
        x, xt = _need_feature(x, "x")
        out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
        rows = x.numel() // x.shape[-1]
        _lib.check(self.lib.cone_l2_normalize_ex(_ptr(x), xt, _ptr(out), rows, x.shape[-1], eps, _stream()),
                   "cone_l2_normalize_ex")
        return out

    def encoder_tail(self, layer: int, att: torch.Tensor, res: torch.Tensor, cta_group: int = 0) -> torch.Tensor:
        """norm2(x + FFN(x)), x = norm1(res + out_proj(att)) of encoder layer `layer` (cone/transformer.py:239-245) on
        [M, 256] fp32 rows through the fused tensor-core kernel."""
        att, res = _need(att, torch.float32, "att"), _need(res, torch.float32, "res")
        out = torch.empty_like(res)
        M = att.shape[0]
        ws, n = self._wsargs(10 * M * att.shape[1] + (1 << 20))
        _lib.check(self.lib.cone_encoder_tail(self._handle, layer, _ptr(att), _ptr(res), M, _ptr(out), cta_group, ws, n,
                                              _stream()), "cone_encoder_tail")
        return out

    def adapter(self, x: torch.Tensor, residual: bool = False, precision: Optional[str] = None) -> torch.Tensor:
        """`model.adapter_layer(x)` (cone/model.py:80); `residual=True` gives `adapter_layer(x) + x`."""
        x = _need(x, torch.float32, "x")
        out = torch.empty_like(x)
        rows = x.numel() // x.shape[-1]
        prec = self.precision if precision is None else {"fp32": _lib.PREC_FP32, "tc": _lib.PREC_TC}[precision]
        ws, n = self._wsargs(rows * self.cfg.hidden_dim * 4 + rows * max(self.cfg.v_feat_dim, 1024) * 2 + (1 << 20))
        _lib.check(self.lib.cone_adapter(self._handle, _ptr(x), _ptr(out), rows, int(residual), ws, n, prec,
                                         _stream()), "cone_adapter")
        return out

    def linear(self, x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, relu: bool = False,
               residual: Optional[torch.Tensor] = None, precision: Optional[str] = None) -> torch.Tensor:
        """`F.linear` (+ residual, + ReLU) on rows through the library's GEMM path of the given precision."""
        x = _need(x, torch.float32, "x")
        weight = _need(weight, torch.float32, "weight")
        M, K = x.shape
        N = weight.shape[0]
        y = torch.empty((M, N), dtype=torch.float32, device=x.device)
        prec = self.precision if precision is None else {"fp32": _lib.PREC_FP32, "tc": _lib.PREC_TC,
                                                          "split": _lib.PREC_TC_SPLIT}[precision]
        ws, nb = self._wsargs(M * K * 6 + 4096)
        _lib.check(self.lib.cone_linear(self._handle, _ptr(x), _ptr(weight), _ptr(bias), M, N, K, int(relu),
                                        _ptr(residual), _ptr(y), ws, nb, prec, _stream()), "cone_linear")
        return y

    def video_prepare(self, frames: torch.Tensor, want_ctx=True, want_vidproj=True, motion: Optional[torch.Tensor] = None):
        """Stage 0 + per-frame `input_vid_proj` over concatenated frames [n, Dv] (raw appearance features).
        `motion` [n, Dm]: raw features of a separate motion stream, one row per appearance row; `input_vid_proj` then
        reads them L2-normalised (ego4d_mad_dataloader.py:284-292).  Without it the appearance rows are projected
        raw, which is only valid when the model's motion dim is Dv.  `frames` and `motion` may each be stored as fp32,
        fp16 or bf16; the results (fp32) are those of the fp32 upcast."""
        frames, ft = _need_feature(frames, "frames")
        n = frames.shape[0]
        if motion is not None:
            motion, mt = self._check_motion(motion, n)
        elif want_vidproj and self.cfg.motion_dim != self.cfg.v_feat_dim:
            raise ValueError(f"the model reads {self.cfg.motion_dim}-d motion features: pass `motion` [n_frames, "
                             f"{self.cfg.motion_dim}] (appearance rows are {self.cfg.v_feat_dim}-d)")
        ctx = torch.empty(frames.shape, dtype=torch.float32, device=frames.device) if want_ctx else None
        vp = torch.empty((n, self.cfg.hidden_dim), dtype=torch.float32, device=frames.device) if want_vidproj else None
        ws, nb = self._wsargs()
        _lib.check(self.lib.cone_video_prepare_ex(self._handle, _ptr(frames), ft, n, _ptr(ctx),
                                                  _ptr(vp if motion is None else None), ws, nb, self.precision, _stream()),
                   "cone_video_prepare_ex")
        if motion is not None and want_vidproj:
            _lib.check(self.lib.cone_video_prepare_motion_ex(self._handle, _ptr(motion), mt, n, _ptr(vp), ws, nb,
                                                             self.precision, _stream()), "cone_video_prepare_motion_ex")
        return ctx, vp

    def _check_motion(self, motion: torch.Tensor, n_frames: int):
        """Both streams are sliced with the same window bounds (ego4d_mad_dataloader.py:144-159): a motion tensor of
        another length is refused rather than truncated.  Returns (motion, its dtype code)."""
        motion, mt = _need_feature(motion, "motion")
        if motion.dim() != 2 or motion.shape != (n_frames, self.cfg.motion_dim):
            raise ValueError(f"motion must be [{n_frames}, {self.cfg.motion_dim}] (one row per appearance frame), "
                             f"got {tuple(motion.shape)}")
        return motion, mt

    def frame_scores(self, ctx: torch.Tensor, qb: QueryBatch, cls_norm: torch.Tensor):
        """`einsum('db,b->d')` of every query against its own video (cone/inference.py:284) as one grouped
        GEMM; returns (ragged scores, offsets[Nq])."""
        lens64 = qb.q_video_len.to(torch.int64)
        score_offsets = torch.cumsum(lens64, 0) - lens64
        scores = torch.empty((max(qb.total_scores, 1),), dtype=torch.float32, device=ctx.device)
        n_videos = qb.video_offsets.numel() - 1
        _lib.check(self.lib.cone_frame_scores(_ptr(ctx), self.cfg.v_feat_dim, _ptr(qb.video_offsets), _ptr(qb.q_first),
                                              n_videos, qb.max_video_frames, qb.max_video_queries, _ptr(cls_norm),
                                              _ptr(scores), _ptr(score_offsets), self.precision, _stream()),
                   "cone_frame_scores")
        return scores, score_offsets

    def window_ranklist(self, frame_score: torch.Tensor, score_offsets: torch.Tensor, frame_count: torch.Tensor,
                        ranklist_stride: Optional[int] = None, want_scores: bool = False, max_v_l: Optional[int] = None):
        """Full window rank-list per query from (ragged) frame scores (cone/inference.py:286-299)."""
        frame_score = _need(frame_score, torch.float32, "frame_score")
        score_offsets = _need(score_offsets, torch.int64, "score_offsets")
        frame_count = _need(frame_count, torch.int32, "frame_count")
        max_v_l = max_v_l or self.cfg.max_v_l
        nq = frame_count.numel()
        if ranklist_stride is None:
            ranklist_stride = math.ceil(int(frame_count.max().item()) / int(max_v_l / 2)) + 1
        rl = torch.empty((nq, ranklist_stride), dtype=torch.int32, device=frame_score.device)
        ws = torch.empty((nq, ranklist_stride), dtype=torch.float32, device=frame_score.device) if want_scores else None
        _lib.check(self.lib.cone_window_ranklist(_ptr(frame_score), _ptr(score_offsets), _ptr(frame_count), nq, max_v_l,
                                                 _ptr(rl), _ptr(ws), ranklist_stride, _stream()), "cone_window_ranklist")
        return (rl, ws) if want_scores else rl

    def prefilter(self, frames_raw: torch.Tensor, cls_raw: torch.Tensor, topk: Optional[int] = None, want_scores: bool = False):
        """Stages 0 + 1 for ONE video in one call (`cone_prefilter`): raw frames [L, Dv] and raw CLS [Nq, Dv] -> the first
        `topk` window ids of every query's rank-list (-1 where the video has fewer windows) and their window scores.
        The same pre-filter `compute_window_ranklist` runs (run_on_video/cone_localizator.py:83-100) and the 2D-TAN
        variant reuses (cone_2dtan/moment_localization/test.py:173-239).  Frames and CLS may each be fp32, fp16 or bf16."""
        frames_raw, ft = _need_feature(frames_raw, "frames_raw")
        cls_raw, ct = _need_feature(cls_raw, "cls_raw")
        L, nq = frames_raw.shape[0], cls_raw.shape[0]
        topk = topk or self.cfg.topk_window
        idx = torch.empty((nq, topk), dtype=torch.int32, device=frames_raw.device)
        sc = torch.empty((nq, topk), dtype=torch.float32, device=frames_raw.device) if want_scores else None
        need = self.lib.cone_prefilter_workspace_bytes(C.byref(self.dims), L, nq)
        ws, nb = self._wsargs(need)
        _lib.check(self.lib.cone_prefilter_ex(self._handle, _ptr(frames_raw), ft, L, _ptr(cls_raw), ct, nq, topk, _ptr(idx),
                                              _ptr(sc), ws, nb, _stream()), "cone_prefilter_ex")
        return (idx, sc) if want_scores else idx

    def forward(self, src_txt, txt_len, src_vid, vid_len, want_saliency=False, want_aux=False):
        """`CONE.forward` on a dense padded batch (cone/model.py:82-128); lengths instead of masks."""
        src_txt = _need(src_txt, torch.float32, "src_txt")
        src_vid = _need(src_vid, torch.float32, "src_vid")
        txt_len = _need(txt_len, torch.int32, "txt_len")
        vid_len = _need(vid_len, torch.int32, "vid_len")
        B, Lt, _ = src_txt.shape
        _, Lv, _ = src_vid.shape
        nq = self.cfg.num_queries
        dev = src_vid.device
        logits = torch.empty((B, nq, 2), dtype=torch.float32, device=dev)
        spans = torch.empty((B, nq, 2), dtype=torch.float32, device=dev)
        sal = torch.empty((B, Lv), dtype=torch.float32, device=dev) if want_saliency else None
        n_aux = self.cfg.dec_layers - 1
        aux_l = torch.empty((n_aux, B, nq, 2), dtype=torch.float32, device=dev) if want_aux and n_aux else None
        aux_s = torch.empty((n_aux, B, nq, 2), dtype=torch.float32, device=dev) if want_aux and n_aux else None
        need = self.lib.cone_workspace_bytes(C.byref(self.dims), B, Lv, Lt)
        ws, nb = self._wsargs(need)
        _lib.check(self.lib.cone_forward(self._handle, _ptr(src_txt), _ptr(txt_len), _ptr(src_vid), _ptr(vid_len), B, Lt,
                                         Lv, _ptr(logits), _ptr(spans), _ptr(sal), _ptr(aux_l), _ptr(aux_s), ws, nb,
                                         self.precision, _stream()), "cone_forward")
        return logits, spans, sal, aux_l, aux_s

    def clip_matching(self, src_cls_txt, src_vid_appear, vid_len, spans):
        """`CONE.forward_clip_matching` (cone/model.py:130-152) on a dense padded batch."""
        cls = _need(src_cls_txt, torch.float32, "src_cls_txt")
        vid = _need(src_vid_appear, torch.float32, "src_vid_appear")
        vid_len = _need(vid_len, torch.int32, "vid_len")
        spans = _need(spans, torch.float32, "proposal")
        B, Lv, _ = vid.shape
        nq = spans.shape[1]
        out = torch.empty((B, nq), dtype=torch.float32, device=vid.device)
        need = B * nq * (2 * self.cfg.v_feat_dim + self.cfg.hidden_dim) * 4 + B * self.cfg.v_feat_dim * 4 + (4 << 20)
        ws, nb = self._wsargs(need * 2)
        _lib.check(self.lib.cone_clip_matching(self._handle, _ptr(cls), _ptr(vid), _ptr(vid_len), _ptr(spans), B, Lv, nq,
                                               _ptr(out), ws, nb, self.precision, _stream()), "cone_clip_matching")
        return out

    def fuse_nms(self, pred_spans, prob_fg, match, win_start, win_len, want_rows=False, cfg: Optional[ConeConfig] = None,
                 fixed_duration: int = 0, sort_within_window: bool = True):
        """Stage 3.  `fixed_duration` / `sort_within_window` select the single-video front end's variant
        (run_on_video/cone_localizator.py:183-219); the defaults are eval_epoch's."""
        cfg = cfg or self.cfg
        nq_, k, nslot = prob_fg.shape
        dev = prob_fg.device
        out = torch.zeros((nq_, 3, cfg.max_after_nms, 5), dtype=torch.float64, device=dev)
        cnt = torch.zeros((nq_, 3), dtype=torch.int32, device=dev)
        rows = torch.zeros((nq_, k * nslot, 4), dtype=torch.float64, device=dev) if want_rows else None
        rcnt = torch.zeros((nq_,), dtype=torch.int32, device=dev) if want_rows else None
        _lib.check(self.lib.cone_fuse_nms_ex(_ptr(_need(pred_spans, torch.float32, "pred_spans")),
                                             _ptr(_need(prob_fg, torch.float32, "prob_fg")),
                                             _ptr(_need(match, torch.float32, "match")),
                                             _ptr(_need(win_start, torch.int32, "win_start")),
                                             _ptr(_need(win_len, torch.int32, "win_len")), nq_, k, nslot,
                                             float(np.float32(cfg.clip_length)), float(cfg.nms_thd), cfg.max_before_nms,
                                             cfg.max_after_nms, int(fixed_duration), int(bool(sort_within_window)),
                                             _ptr(out), _ptr(cnt), _ptr(rows), _ptr(rcnt), _stream()),
                   "cone_fuse_nms_ex")
        return out, cnt, rows, rcnt

    # ---- metric counters (SURVEY.md §8(f)1) ---------------------------------------------------
    def eval_recall(self, nms: torch.Tensor, nms_count: torch.Tensor, gt: torch.Tensor, topk=(1, 5),
                    thresholds=(0.3, 0.5), flavour: str = "mad", hits: Optional[torch.Tensor] = None,
                    want_top1: bool = False):
        """R@K / IoU hit counters of `evaluate_mad.py:60-104` (flavour "mad") or `evaluate_ego4d_nlq.py:65-117`
        ("ego4d") from the stage-3 output.  gt [Nq, 2] fp64 seconds, packed-query order.  Returns
        (hits [3, len(topk), len(thresholds)] int64 on the device — accumulated into when passed in —, top-1 IoU
        [Nq, 3] fp64 or None)."""
        nms = _need(nms, torch.float64, "nms")
        nms_count = _need(nms_count, torch.int32, "nms_count")
        gt = _need(gt, torch.float64, "gt")
        nq_ = nms.shape[0]
        if gt.shape != (nq_, 2):
            raise ValueError(f"gt must be [{nq_}, 2], got {tuple(gt.shape)}")
        if hits is None:
            hits = torch.zeros((3, len(topk), len(thresholds)), dtype=torch.int64, device=nms.device)
        hits = _need(hits, torch.int64, "hits")
        if hits.shape != (3, len(topk), len(thresholds)):
            raise ValueError("hits must be [3, len(topk), len(thresholds)]")
        top1 = torch.empty((nq_, 3), dtype=torch.float64, device=nms.device) if want_top1 else None
        tk = (C.c_int32 * len(topk))(*[int(k) for k in topk])
        th = (C.c_double * len(thresholds))(*[float(t) for t in thresholds])
        _lib.check(self.lib.cone_eval_recall(_ptr(nms), _ptr(nms_count), _ptr(gt), nq_, nms.shape[2], tk, len(topk), th,
                                             len(thresholds), {"mad": 0, "ego4d": 1}[flavour], _ptr(hits), _ptr(top1),
                                             _stream()), "cone_eval_recall")
        return hits, top1

    def eval_window_recall(self, ranklist: torch.Tensor, gt: torch.Tensor, topk=(1, 5, 10, 30, 50),
                           hits: Optional[torch.Tensor] = None, cfg: Optional[ConeConfig] = None) -> torch.Tensor:
        """Window pre-filtering recall counters (`evaluate_pre_filtered_window.py:30-72`) from the rank-lists."""
        cfg = cfg or self.cfg
        ranklist = _need(ranklist, torch.int32, "ranklist")
        gt = _need(gt, torch.float64, "gt")
        if hits is None:
            hits = torch.zeros((len(topk),), dtype=torch.int64, device=ranklist.device)
        hits = _need(hits, torch.int64, "hits")
        tk = (C.c_int32 * len(topk))(*[int(k) for k in topk])
        _lib.check(self.lib.cone_eval_window_recall(_ptr(ranklist), ranklist.shape[1], _ptr(gt), ranklist.shape[0],
                                                    float(cfg.clip_length), cfg.max_v_l, tk, len(topk), _ptr(hits),
                                                    _stream()), "cone_eval_window_recall")
        return hits

    # ---- the whole path -------------------------------------------------------------------------
    def ground(self, frames: torch.Tensor, qb: QueryBatch, want_rows: bool = False, prepared=None,
               motion: Optional[torch.Tensor] = None) -> GroundingOutput:
        """Stages 0-3 for concatenated raw `frames` [n_frames, Dv] and the packed queries `qb` (both on the
        device).  No host synchronisation inside: sizes come from host metadata in `qb`.
        `motion` [n_frames, Dm]: raw features of a separate motion stream (`--motion_feat_dir`), concatenated like
        `frames`; stages 0/1 and the matching pool keep reading `frames`, Moment-DETR reads the motion rows.
        `prepared` = (ctx, vidproj) from an earlier `video_prepare(frames, motion=motion)`: stage 0 is per VIDEO
        (cone/inference.py:241-260 runs it once per video before any query), so a long video whose queries are
        processed in several calls (BASELINE.json configs[4]) pays for it once; `motion` is then not read.
        `frames`, `motion`, `qb.tokens` and `qb.cls` may each be stored as fp32, fp16 or bf16: the output is bitwise
        the one of the same call on their fp32 upcasts (the library converts on load and keeps the fp32 order)."""
        cfg = self.cfg
        frames, ft = _need_feature(frames, "frames")
        dev = frames.device
        nq = qb.tok_len.numel()
        k = cfg.topk_window
        ns = cfg.num_queries
        # stage 0: context features and per-frame video projection
        ctx, vidproj = prepared if prepared is not None else self.video_prepare(frames, motion=motion)
        # host-side normalisations of the reference's dataset code, on the device
        cls_norm = self.l2_normalize(qb.cls, 1e-5)  # dataloader:472 / :280
        tok_norm = self.l2_normalize(qb.tokens, 1e-5)  # dataloader:274-276 (zero pad rows stay zero)
        # stage 1: frame scores -> window rank-list
        scores, score_offsets = self.frame_scores(ctx, qb, cls_norm)
        stride = cfg.num_window(qb.max_video_frames)
        ranklist = self.window_ranklist(scores, score_offsets, qb.q_video_len, ranklist_stride=stride)
        del scores
        # stage 2
        spans = torch.empty((nq, k, ns, 2), dtype=torch.float32, device=dev)
        prob = torch.empty((nq, k, ns), dtype=torch.float32, device=dev)
        match = torch.empty((nq, k, ns), dtype=torch.float32, device=dev)
        wstart = torch.empty((nq, k), dtype=torch.int32, device=dev)
        wlen = torch.empty((nq, k), dtype=torch.int32, device=dev)
        ws, nb = self._wsargs()
        _lib.check(self.lib.cone_ground_windows_ex(
            self._handle, _ptr(frames), ft, frames.shape[0], _ptr(vidproj), _ptr(qb.q_video_start), _ptr(qb.q_video_len),
            _ptr(ranklist), stride, _ptr(tok_norm), _ptr(qb.tok_len), _ptr(cls_norm), _ptr(qb.q_batch), qb.n_batches,
            nq, k, _ptr(spans), _ptr(prob), _ptr(match), _ptr(wstart), _ptr(wlen), ws, nb, self.precision, _stream()),
            "cone_ground_windows_ex")
        # stage 3
        nms, cnt, rows, rcnt = self.fuse_nms(spans, prob, match, wstart, wlen, want_rows=want_rows)
        return GroundingOutput(ranklist, wstart, wlen, spans, prob, match, nms, cnt, rows, rcnt)

    # ---- the single-video front end (SURVEY.md §8(f)3) ------------------------------------------
    def prepare_video(self, frames: torch.Tensor):
        """Per-video part of `CONELocalizator.predict_moment` (run_on_video/cone_localizator.py:127-136):
        F.normalize of the frames, adapter + residual WITHOUT re-normalisation (the ranking features), and the
        per-frame `input_vid_proj` of the NORMALISED frames (what the demo slices into windows).
        Returns (xn, ctx, vidproj), all on the device."""
        frames = _need(frames, torch.float32, "frames")
        xn = self.l2_normalize(frames, -1e-5)
        ctx = self.adapter(xn, residual=True, precision="fp32")  # the window ranking stays fp32 in every mode
        _, vidproj = self.video_prepare(xn, want_ctx=False)
        return xn, ctx, vidproj

    def ground_video(self, xn: torch.Tensor, ctx: torch.Tensor, vidproj: torch.Tensor, qb: QueryBatch,
                     cfg: Optional[ConeConfig] = None, want_rows: bool = False) -> GroundingOutput:
        """Per-query part of `predict_moment` (:131-221) for queries of ONE video prepared by `prepare_video`:
        tokens F.normalize'd, CLS used raw, windows zero-padded to max_v_l for pooling, spans scaled by max_v_l,
        slots in slot order, fusion ranking with the demo's NMS constants (pass them in `cfg`).  No host sync.
        fp32 only, like `prepare_video`."""
        cfg = cfg or self.cfg
        xn = _need(xn, torch.float32, "xn")
        _need(qb.tokens, torch.float32, "qb.tokens")
        _need(qb.cls, torch.float32, "qb.cls")
        dev = xn.device
        nq, k, ns = qb.tok_len.numel(), cfg.topk_window, cfg.num_queries
        tok_norm = self.l2_normalize(qb.tokens, -1e-5)
        scores, score_offsets = self.frame_scores(ctx, qb, qb.cls)
        stride = cfg.num_window(qb.max_video_frames)
        ranklist = self.window_ranklist(scores, score_offsets, qb.q_video_len, ranklist_stride=stride)
        spans = torch.empty((nq, k, ns, 2), dtype=torch.float32, device=dev)
        prob = torch.empty((nq, k, ns), dtype=torch.float32, device=dev)
        match = torch.empty((nq, k, ns), dtype=torch.float32, device=dev)
        wstart = torch.empty((nq, k), dtype=torch.int32, device=dev)
        wlen = torch.empty((nq, k), dtype=torch.int32, device=dev)
        ws, nb = self._wsargs()
        _lib.check(self.lib.cone_ground_windows(
            self._handle, _ptr(xn), xn.shape[0], _ptr(vidproj), _ptr(qb.q_video_start), _ptr(qb.q_video_len),
            _ptr(ranklist), stride, _ptr(tok_norm), _ptr(qb.tok_len), _ptr(qb.cls), None, 1,
            nq, k, _ptr(spans), _ptr(prob), _ptr(match), _ptr(wstart), _ptr(wlen), ws, nb, self.precision, _stream()),
            "cone_ground_windows")
        nms, cnt, rows, rcnt = self.fuse_nms(spans, prob, match, wstart, wlen, want_rows=want_rows, cfg=cfg,
                                             fixed_duration=cfg.max_v_l, sort_within_window=False)
        return GroundingOutput(ranklist, wstart, wlen, spans, prob, match, nms, cnt, rows, rcnt)


def read_profile() -> Dict[str, dict]:
    """Per-category kernel time since profiling was enabled: {name: {ms, launches, flops, bytes}}."""
    lib = _lib.load()
    n = lib.cone_profile_categories()
    ms, fl, by = (C.c_double * n)(), (C.c_double * n)(), (C.c_double * n)()
    la = (C.c_int64 * n)()
    _lib.check(lib.cone_profile_read(ms, la, fl, by, n), "cone_profile_read")
    return {lib.cone_profile_name(i).decode(): {"ms": ms[i], "launches": int(la[i]), "flops": fl[i], "bytes": by[i]}
            for i in range(n)}
