"""Feature ingest (SURVEY.md §8(f)2): the reference's feature records -> pinned host memory -> HBM, overlapped with
the kernels of the previous step.

Record format (what `feature_extraction/misc/convert_h5_to_lmdb.py:20-40` writes and
`cone/ego4d_mad_dataloader.py:258-302, 453-473` reads): one LMDB value per video id / query id, each the bytes of
`np.savez_compressed(...)` holding `features [L, Dv]` for a video, or `token_features [n_tok, Dt]` plus
`cls_features` (Ego4D) / `eot_features` (MAD CLIP) `[Dv]` or `[1, Dv]` for a query.

Only the decoding, staging and overlap are built here; the normalisations the reference applies on the host after
decoding (`l2_normalize_np_array`) run on the device inside `ConeEngine.ground`.  `lmdb` itself is an optional
import: `LmdbStore` raises if the package is missing, `DirStore` / `DictStore` read the same records from a
directory of `<key>.npz` files or a dict.
"""
from __future__ import annotations

import io
import os
import queue
import threading
from typing import Dict, Iterator, List, Optional, Sequence, Tuple

import numpy as np

from .config import ConeConfig
from .inference import HostStep, plan_steps, stage_step
from .synth import SynthQuery


# ------------------------------------------------------------------------------------------------ records
def encode_record(compress: bool = True, **arrays) -> bytes:
    """`dumps_npz` of the reference's converter (convert_h5_to_lmdb.py:20-27)."""
    with io.BytesIO() as w:
        (np.savez_compressed if compress else np.savez)(w, **arrays)
        return w.getvalue()


def _as_feature(a: np.ndarray, dtype, key: str) -> np.ndarray:
    """`a` as a contiguous array of `dtype` (float32 or float16).  float16 records pass through unchanged; wider
    records are rounded once, and a finite value beyond the float16 range raises instead of becoming inf."""
    dtype = np.dtype(dtype)
    if dtype not in (np.dtype(np.float32), np.dtype(np.float16)):
        raise ValueError(f"feature dtype must be float32 or float16, got {dtype}")
    with np.errstate(over="ignore"):
        out = np.ascontiguousarray(a, dtype=dtype)
    if dtype == np.float16 and a.dtype != np.float16:
        bad = np.isinf(out) & np.isfinite(a)
        if bad.any():
            raise ValueError(f"{key}: {int(bad.sum())} finite values exceed the float16 range "
                             f"(largest magnitude {float(np.abs(a[bad]).max()):.6g})")
    return out


def decode_video_record(buf, dtype=np.float32, key: str = "video record") -> np.ndarray:
    """bytes -> raw features [L, Dv] (ego4d_mad_dataloader.py:294-302 returns them un-normalised) as `dtype`:
    float32 (the reference's type) or float16 (half the host, pinned and HBM footprint; see `_as_feature`).
    `key` names the record in errors."""
    with io.BytesIO(bytes(buf)) as r:
        dump = np.load(r, allow_pickle=False)
        if "features" not in dump:
            raise KeyError("video record has no 'features' array")
        return _as_feature(dump["features"], dtype, key)


def decode_query_record(buf, dtype=np.float32, key: str = "query record") -> Tuple[np.ndarray, np.ndarray]:
    """bytes -> (token_features [n_tok, Dt], holistic feature [Dv]) as `dtype` (float32 or float16), raw
    (ego4d_mad_dataloader.py:258-282): `cls_features` if present, else `eot_features`; a [1, Dv] holistic feature is
    squeezed."""
    with io.BytesIO(bytes(buf)) as r:
        dump = np.load(r, allow_pickle=False)
        tok = _as_feature(dump["token_features"], dtype, key)
        cls = np.asarray(dump["cls_features"] if "cls_features" in dump else dump["eot_features"])
        if cls.ndim == 2:
            cls = cls[0]
    return tok, _as_feature(cls, dtype, key)


# ------------------------------------------------------------------------------------------------ stores
class DictStore:
    """key -> record bytes, in memory."""

    def __init__(self, records: Dict[str, bytes]):
        self.records = records

    def get(self, key: str) -> bytes:
        return self.records[key]


class DirStore:
    """A directory of `<key>.npz` files, each one record."""

    def __init__(self, root: str):
        self.root = root

    def get(self, key: str) -> bytes:
        with open(os.path.join(self.root, key + ".npz"), "rb") as f:
            return f.read()


class LmdbStore:
    """The reference's LMDB environments (ego4d_mad_dataloader.py:73-86: readonly, no readahead, buffers=True)."""

    def __init__(self, path: str):
        try:
            import lmdb
        except ImportError as e:  # no silent fallback: the caller asked for LMDB
            raise ImportError("LmdbStore needs the `lmdb` package; use DirStore / DictStore for exported records") from e
        self.env = lmdb.open(path, readonly=True, create=False, max_readers=4096 * 8, readahead=False)
        self.txn = self.env.begin(buffers=True)

    def get(self, key: str) -> bytes:
        v = self.txn.get(key.encode())
        if v is None:
            raise KeyError(key)
        return bytes(v)


# ------------------------------------------------------------------------------------------------ staging
def load_queries(query_store, annotations: Sequence[dict], video_index: Dict[str, int],
                 feature_dtype=np.float32) -> List[SynthQuery]:
    """Annotation rows (query_id, clip_id, timestamps — ego4d_mad_dataloader.py:19-29) -> query objects in DATASET
    order, features decoded from `query_store` as `feature_dtype` (float32 or float16, see `decode_query_record`)."""
    out = []
    for a in annotations:
        tok, cls = decode_query_record(query_store.get(a["query_id"]), feature_dtype, key=a["query_id"])
        ts = a.get("timestamps", (0.0, 0.0))
        out.append(SynthQuery(a["query_id"], video_index[a["clip_id"]], tok, cls, (float(ts[0]), float(ts[1]))))
    return out


class StagedSteps:
    """Iterator of `HostStep`s whose decoding (npz inflate) and pinned staging run on a background thread, `depth`
    steps ahead of the consumer: while the GPU works on step i the host decompresses and pins step i+1 — the part of
    the reference's DataLoader workers that is on the path (the LMDB read + inflate is the dominant host cost,
    SURVEY.md §8 A1)."""

    def __init__(self, cfg: ConeConfig, video_store, video_ids: Sequence[str], video_lengths: Sequence[int], queries,
                 max_frames_per_step: int = 1 << 20, depth: int = 2, pin: bool = True, motion_store=None,
                 feature_dtype=np.float32):
        """`motion_store`: records of a separate motion stream under the same keys (`--motion_feat_dir`); None = the
        appearance records serve both roles.  `feature_dtype` (float32 or float16): the type video and motion records
        are decoded to and staged in (see `decode_video_record`)."""
        self.cfg, self.store, self.video_ids, self.queries, self.pin = cfg, video_store, list(video_ids), queries, pin
        self.motion_store = motion_store
        self.feature_dtype = feature_dtype
        self.plan = plan_steps(video_lengths, queries, max_frames_per_step)
        self._q: "queue.Queue" = queue.Queue(maxsize=max(1, depth))
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._produce, daemon=True)
        self._thread.start()

    def _put(self, item) -> bool:
        """Blocking put that gives up when the consumer has closed the iterator."""
        while not self._stop.is_set():
            try:
                self._q.put(item, timeout=0.1)
                return True
            except queue.Full:
                continue
        return False

    def _produce(self) -> None:
        try:
            for ids in self.plan:
                if self._stop.is_set():
                    return
                # stage_step only indexes videos[v] for v in ids: a dict of this step's decoded arrays is enough
                dt = self.feature_dtype
                vids: Dict[int, np.ndarray] = {v: decode_video_record(self.store.get(self.video_ids[v]), dt,
                                                                      key=self.video_ids[v]) for v in ids}
                mot = None if self.motion_store is None else \
                    {v: decode_video_record(self.motion_store.get(self.video_ids[v]), dt, key=self.video_ids[v])
                     for v in ids}
                step = stage_step(self.cfg, vids, self.queries, ids, pin=self.pin, motion_videos=mot)
                if not self._put(step):
                    return
            self._put(None)
        except BaseException as e:  # surface decoding errors in the consumer thread
            self._put(e)

    def close(self) -> None:
        """Stop the producer (the consumer abandoned the iterator): staged pinned steps are dropped."""
        self._stop.set()
        while True:
            try:
                self._q.get_nowait()
            except queue.Empty:
                break
        self._thread.join(timeout=5.0)

    def __enter__(self) -> "StagedSteps":
        return self

    def __exit__(self, *exc) -> None:
        self.close()

    def __iter__(self) -> Iterator[HostStep]:
        try:
            while True:
                item = self._q.get()
                if item is None:
                    return
                if isinstance(item, BaseException):
                    raise item
                yield item
        finally:  # also runs when the consumer breaks out of its loop (generator close)
            self.close()


def ground_store(engine, video_store, query_store, annotations: Sequence[dict], video_lengths: Optional[Dict[str, int]] = None,
                 max_frames_per_step: int = 1 << 20, full: bool = False, motion_store=None,
                 feature_dtype=np.float32) -> Dict[str, dict]:
    """`eval_epoch` stages 0-3 straight from feature stores: decode -> pinned -> HBM -> kernels, the decoding of the
    next step overlapping the kernels of the current one.  `video_lengths` (frames per clip_id) avoids a first pass
    over the video records when the annotations do not carry it.  `motion_store` holds the records of a separate
    motion stream (`--motion_feat_dir`) under the same clip ids, `features [L, Dm]`; None = the reference's
    same-directory case.  `feature_dtype=np.float16` keeps every feature in float16 from the decoded record to HBM
    (float16 records pass through, wider ones are rounded once on the host); the results are bitwise those of
    `ground_dataset` on the same float16 arrays.  numpy has no bfloat16: bf16 features are reachable only through
    `ConeEngine` with torch tensors."""
    from .inference import output_to_host, run_step
    clip_ids = list(dict.fromkeys(a["clip_id"] for a in annotations))
    index = {c: i for i, c in enumerate(clip_ids)}
    if video_lengths is None:
        video_lengths = {c: int(decode_video_record(video_store.get(c)).shape[0]) for c in clip_ids}
    queries = load_queries(query_store, annotations, index, feature_dtype)
    res: Dict[str, dict] = {}
    steps = StagedSteps(engine.cfg, video_store, clip_ids, [video_lengths[c] for c in clip_ids], queries,
                        max_frames_per_step, motion_store=motion_store, feature_dtype=feature_dtype)
    for step in steps:
        if step.qb.tok_len.numel() == 0:
            continue
        out = run_step(engine, step, want_rows=full)
        res.update(output_to_host(engine.cfg, step, out, full=full))
    return res
