"""Single-video, single-query front end over the same kernels: the B200 counterpart of
`run_on_video/cone_localizator.py` (`CONELocalizator`, SURVEY.md §8(f)3).

Same method names and argument meaning as the reference class:

    loc = CONELocalizator(state_dict_or_ckpt_path, cfg=EGO4D_DEMO, device="cuda:0")
    ranklist = loc.compute_window_ranklist(adapter_video_feats, text_cls_feat)      # cone_localizator.py:84-100
    moments  = loc.predict_moment(video_feats, (text_token_feats, text_cls_feat))   # cone_localizator.py:121-221

What is different underneath: the per-video work (normalisation, adapter, per-frame input projection) is done
once per video and cached on the device (`set_video`), and the per-query work is captured in a CUDA graph on
first use, so a query costs one H2D of its features, one graph launch and one D2H of <= 5 moments.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import List, Optional, Tuple, Union

import torch

from .config import EGO4D, ConeConfig
from .engine import ConeEngine, GroundingOutput, QueryBatch, pack_queries

# the demo's own constants (run_on_video/cone_localizator.py:12-37, 213-217): clip_length 0.5333 (not 0.53333),
# predicted_moments[:100], nms_thd 0.5, max_after_nms 5
EGO4D_DEMO = EGO4D.replace(clip_length=0.5333, max_before_nms=100, nms_thd=0.5, max_after_nms=5, name="ego4d_demo")


def _as_f32(x) -> torch.Tensor:
    t = torch.as_tensor(x)
    return t.detach().to(torch.float32)


def _video_key(obj, v: torch.Tensor):
    """Identity of a video for the per-video cache.  NOT `id(obj)` alone: CPython reuses the ids of freed objects,
    and the reference driver builds `video_feats` as a function-local that dies after every call
    (run_on_video/run.py:54-57), so a second video could silently hit the first one's cache.  The cache therefore
    keeps a strong reference to the object it was filled from (its id cannot be recycled while cached) and the key
    also carries the storage address, the shape, the tensor version counter (every in-place edit of a torch tensor)
    and a fingerprint of 16 evenly spaced rows (numpy arrays have no version counter: an in-place edit that misses
    all sampled rows is not seen — call `set_video` after editing a numpy array in place)."""
    ver = getattr(obj, "_version", None)
    n = v.shape[0]
    rows = sorted({(i * (n - 1)) // 15 for i in range(16)}) if n else []
    sample = v[rows].contiguous().cpu().numpy().tobytes() if rows else b""
    return (id(obj), int(v.data_ptr()), tuple(v.shape), ver, hash(sample))


class CONELocalizator:
    def __init__(self, load_checkpoint_path: Union[str, dict] = "ckpt/model_best.ckpt", device: str = "cuda",
                 cfg: ConeConfig = EGO4D_DEMO, precision: str = "fp32", workspace_bytes: int = 1 << 30,
                 use_cuda_graph: bool = True):
        """`load_checkpoint_path`: a checkpoint file holding {"model": state_dict} as the reference loads it
        (cone_localizator.py:75-76), or the state dict itself."""
        if cfg.motion_dim != cfg.v_feat_dim:
            raise NotImplementedError("the single-video front end reads one feature stream for every role "
                                      "(run_on_video/cone_localizator.py:127-165); a model with a separate motion "
                                      "stream runs through ConeEngine.ground / inference.ground_dataset")
        if isinstance(load_checkpoint_path, str):
            sd = torch.load(load_checkpoint_path, map_location="cpu")["model"]
        else:
            sd = load_checkpoint_path
        self.cfg = cfg
        self.device = torch.device("cuda:0" if device == "cuda" else device)
        self.localizator = ConeEngine(cfg, sd, device=self.device, precision=precision, workspace_bytes=workspace_bytes)
        self.slide_window_size = int(cfg.max_v_l / 2)
        self.max_v_l = cfg.max_v_l
        self.use_cuda_graph = use_cuda_graph
        self._video = None  # (key, xn, ctx, vidproj)
        self._video_obj = None  # strong reference to the object the cache was filled from (see _video_key)
        self._graph = None
        self._static: Optional[SimpleNamespace] = None

    # ---- reference API ---------------------------------------------------------------------------
    @torch.no_grad()
    def compute_window_ranklist(self, video_feats, text_cls_feat) -> List[int]:
        """(L, Dv) adapted features x (Dv,) CLS -> window ids by descending max frame score, ties by lower id."""
        eng = self.localizator
        with torch.cuda.device(self.device):
            v = _as_f32(video_feats).to(self.device).contiguous()
            qb = self._query_batch(v.shape[0], torch.zeros((1, self.cfg.t_feat_dim)), _as_f32(text_cls_feat).cpu().reshape(-1))
            qb = qb.to(self.device)
            fs, offs = eng.frame_scores(v, qb, qb.cls)
            rl = eng.window_ranklist(fs, offs, qb.q_video_len, max_v_l=self.max_v_l)
            return [int(x) for x in rl[0].cpu().tolist() if x >= 0]

    @torch.no_grad()
    def set_video(self, video_feats) -> None:
        """Upload one video's raw features and run the per-video stage; queries then reuse it."""
        v = _as_f32(video_feats)
        if v.dim() != 2 or v.shape[1] != self.cfg.v_feat_dim:
            raise ValueError(f"video_feats must be [L, {self.cfg.v_feat_dim}], got {tuple(v.shape)}")
        with torch.cuda.device(self.device):
            xn, ctx, vidproj = self.localizator.prepare_video(v.to(self.device, non_blocking=True).contiguous())
            if self._graph is not None and self._video is not None and self._video[1].shape == xn.shape:
                # same length (or the same video after a weight update): refill the tensors the captured graph reads —
                # its launch geometry depends on the number of frames only, so it stays valid
                for dst, src in zip(self._video[1:], (xn, ctx, vidproj)):
                    dst.copy_(src)
                self._video = (_video_key(video_feats, v),) + tuple(self._video[1:])
                self._video_obj = video_feats
                return
        self._video = (_video_key(video_feats, v), xn, ctx, vidproj)
        self._video_obj = video_feats
        self._graph = None
        self._static = None

    def _query_batch(self, n_frames: int, tokens: torch.Tensor, cls: torch.Tensor) -> QueryBatch:
        cfg = self.cfg
        if tokens.shape[0] > cfg.max_q_l:  # pad_feature would raise in the reference (cone_localizator.py:114)
            raise ValueError(f"{tokens.shape[0]} text tokens exceed max_q_l={cfg.max_q_l}")
        q = SimpleNamespace(query_id="q", video_idx=0, tokens=tokens.numpy(), cls=cls.numpy())
        return pack_queries(cfg, [n_frames], [q])

    def _run(self, qb: QueryBatch) -> GroundingOutput:
        _, xn, ctx, vidproj = self._video
        return self.localizator.ground_video(xn, ctx, vidproj, qb, cfg=self.cfg)

    @torch.no_grad()
    def predict_moment(self, video_feats, text_feats: Tuple) -> List[List[float]]:
        """-> [[st, ed, fusion_score], ...] (<= max_after_nms rows), as the reference returns."""
        if self._video is None or self._video_obj is not video_feats or \
                self._video[0] != _video_key(video_feats, _as_f32(video_feats)):
            self.set_video(video_feats)
        tokens, cls = _as_f32(text_feats[0]).cpu(), _as_f32(text_feats[1]).cpu().reshape(-1)
        n_frames = self._video[1].shape[0]
        host_qb = self._query_batch(n_frames, tokens, cls)
        with torch.cuda.device(self.device):
            if not self.use_cuda_graph:
                out = self._run(host_qb.to(self.device))
            else:
                out = self._replay(host_qb)
            cnt = int(out.nms_count[0, 0].item())
            rows = out.nms[0, 0, :cnt].cpu().numpy()
        return [[float(r[0]), float(r[1]), float(r[4])] for r in rows]

    # ---- CUDA graph of the per-query part --------------------------------------------------------
    def _replay(self, host_qb: QueryBatch) -> GroundingOutput:
        st = self._static
        if st is None:
            st = SimpleNamespace(qb=host_qb.to(self.device, non_blocking=False), out=None)
            self._run(st.qb)  # warm-up: lazy weight caches, kernel attributes
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                st.out = self._run(st.qb)
            self._graph, self._static = g, st
        else:  # only the query's own tensors change between replays
            st.qb.tokens.copy_(host_qb.tokens, non_blocking=True)
            st.qb.tok_len.copy_(host_qb.tok_len, non_blocking=True)
            st.qb.cls.copy_(host_qb.cls, non_blocking=True)
        self._graph.replay()
        return st.out
