"""Half-precision feature storage on the host (no GPU): query packing and step staging keep float16, mixed types are
refused before they could be promoted, the H2D byte count follows the element size, and the record decoders round
float32 records to float16 once and refuse values that would overflow."""
import dataclasses

import numpy as np
import pytest

from cone_b200 import ingest
from cone_b200.config import EGO4D
from cone_b200.engine import pack_queries
from cone_b200.inference import evaluate_dataset, ground_dataset, stage_step
from cone_b200.synth import make_dataset


def _half(ds):
    videos = [v.astype(np.float16) for v in ds.videos]
    motion = None if ds.motion is None else [m.astype(np.float16) for m in ds.motion]
    queries = [dataclasses.replace(q, tokens=q.tokens.astype(np.float16), cls=q.cls.astype(np.float16)) for q in ds.queries]
    return videos, motion, queries


def _ds(motion_dim=None):
    cfg = EGO4D.replace(eval_bsz=2, v_motion_feat_dim=motion_dim or 0)
    return cfg, make_dataset(cfg, 3, [120, 40, 75], [2, 1, 2], seed=4, motion_dim=motion_dim)


def test_pack_queries_keeps_float16():
    cfg, ds = _ds()
    _, _, queries = _half(ds)
    qb = pack_queries(cfg, [len(v) for v in ds.videos], queries)
    assert qb.tokens.numpy().dtype == np.float16 and qb.cls.numpy().dtype == np.float16
    ref = pack_queries(cfg, [len(v) for v in ds.videos], ds.queries)
    assert ref.tokens.numpy().dtype == np.float32 and ref.cls.numpy().dtype == np.float32
    # same layout, zero padding in float16: the float16 batch is the rounded float32 batch
    assert np.array_equal(qb.tokens.numpy(), ref.tokens.numpy().astype(np.float16))
    assert np.array_equal(qb.cls.numpy(), ref.cls.numpy().astype(np.float16))
    assert np.array_equal(qb.tok_len.numpy(), ref.tok_len.numpy())


def test_stage_step_keeps_float16_per_stream_and_counts_bytes():
    cfg, ds = _ds(motion_dim=1024)
    videos, motion, queries = _half(ds)
    ids = [0, 1, 2]
    n = sum(len(v) for v in ds.videos)
    ref = stage_step(cfg, ds.videos, ds.queries, ids, pin=False, motion_videos=ds.motion)
    half = stage_step(cfg, videos, queries, ids, pin=False, motion_videos=motion)
    assert half.frames.numpy().dtype == np.float16 and half.motion.numpy().dtype == np.float16
    assert np.array_equal(half.frames.numpy(), ref.frames.numpy().astype(np.float16))
    feat16 = n * 256 * 2 + n * 1024 * 2 + half.qb.tokens.numel() * 2 + half.qb.cls.numel() * 2
    feat32 = 2 * feat16
    assert ref.h2d_bytes() - half.h2d_bytes() == feat32 - feat16
    # the motion stream's type is independent of the appearance type
    mixed = stage_step(cfg, ds.videos, ds.queries, ids, pin=False, motion_videos=motion)
    assert mixed.frames.numpy().dtype == np.float32 and mixed.motion.numpy().dtype == np.float16
    assert mixed.h2d_bytes() == ref.h2d_bytes() - n * 1024 * 2


def test_mixed_dtypes_are_refused():
    cfg, ds = _ds(motion_dim=1024)
    videos, motion, queries = _half(ds)
    mixed_v = [videos[0]] + list(ds.videos[1:])
    with pytest.raises(ValueError, match="videos mix float16 and float32"):
        stage_step(cfg, mixed_v, ds.queries, [0, 1], pin=False)
    with pytest.raises(ValueError, match="motion features mix"):
        stage_step(cfg, ds.videos, ds.queries, [0, 1], pin=False, motion_videos=[motion[0]] + list(ds.motion[1:]))
    with pytest.raises(ValueError, match="queries mix"):
        pack_queries(cfg, [len(v) for v in ds.videos], [queries[0]] + list(ds.queries[1:]))
    # the dataset drivers check every video, motion tensor and query before any work: the engine is never touched
    # (one video per step would otherwise stage uniform steps)
    for fn in (ground_dataset, lambda *a, **k: evaluate_dataset(a[0], a[1], a[2], {}, **k)):
        with pytest.raises(ValueError, match="videos mix"):
            fn(None, [ds.videos[0], videos[1], ds.videos[2]], ds.queries, max_frames_per_step=1)
        with pytest.raises(ValueError, match="motion features mix"):
            fn(None, ds.videos, ds.queries, max_frames_per_step=1, motion_videos=[ds.motion[0], motion[1], ds.motion[2]])
        with pytest.raises(ValueError, match="queries mix"):
            fn(None, ds.videos, list(ds.queries[:-1]) + [queries[-1]], max_frames_per_step=1)


def test_decode_records_as_float16():
    rng = np.random.default_rng(0)
    f32 = rng.standard_normal((17, 256), dtype=np.float32) * 30
    f16 = f32.astype(np.float16)
    got = ingest.decode_video_record(ingest.encode_record(features=f16), dtype=np.float16)
    assert got.dtype == np.float16 and np.array_equal(got, f16)  # passes through
    got = ingest.decode_video_record(ingest.encode_record(features=f32), dtype=np.float16)
    assert got.dtype == np.float16 and np.array_equal(got, f16)  # rounded once
    assert ingest.decode_video_record(ingest.encode_record(features=f16)).dtype == np.float32  # default unchanged
    tok, cls = ingest.decode_query_record(ingest.encode_record(token_features=f32[:5], cls_features=f32[5:6]),
                                          dtype=np.float16)
    assert tok.dtype == cls.dtype == np.float16 and cls.shape == (256,)
    assert np.array_equal(tok, f16[:5]) and np.array_equal(cls, f16[5])
    tok, cls = ingest.decode_query_record(ingest.encode_record(token_features=f16[:5], eot_features=f16[5]),
                                          dtype=np.float16)
    assert np.array_equal(tok, f16[:5]) and np.array_equal(cls, f16[5])
    # a finite value beyond the float16 range (65504) would become inf: refused, naming the record
    big = f32.copy()
    big[3, 7] = 1e5
    with pytest.raises(ValueError, match="clip_7.*float16 range"):
        ingest.decode_video_record(ingest.encode_record(features=big), dtype=np.float16, key="clip_7")
    with pytest.raises(ValueError, match="float16 range"):
        ingest.decode_query_record(ingest.encode_record(token_features=f32[:2], cls_features=big[3]), dtype=np.float16)
    # an inf already in the record is passed on as it is, as in float32
    inf = f32.copy()
    inf[0, 0] = np.inf
    assert np.isinf(ingest.decode_video_record(ingest.encode_record(features=inf), dtype=np.float16)[0, 0])
    with pytest.raises(ValueError, match="float32 or float16"):
        ingest.decode_video_record(ingest.encode_record(features=f32), dtype=np.float64)


def test_staged_steps_yield_float16():
    cfg, ds = _ds(motion_dim=1024)
    vs = ingest.DictStore({k: ingest.encode_record(features=v) for k, v in zip(ds.video_ids, ds.videos)})
    ms = ingest.DictStore({k: ingest.encode_record(features=m.astype(np.float16)) for k, m in zip(ds.video_ids, ds.motion)})
    qs = ingest.DictStore({q.query_id: ingest.encode_record(token_features=q.tokens, cls_features=q.cls)
                           for q in ds.queries})
    queries = ingest.load_queries(qs, ds.annotations(), {c: i for i, c in enumerate(ds.video_ids)},
                                  feature_dtype=np.float16)
    assert all(q.tokens.dtype == q.cls.dtype == np.float16 for q in queries)
    videos, motion, _ = _half(ds)
    steps = list(ingest.StagedSteps(cfg, vs, ds.video_ids, [len(v) for v in ds.videos], queries, max_frames_per_step=150,
                                    pin=False, motion_store=ms, feature_dtype=np.float16))
    assert len(steps) == 2
    for s in steps:
        assert s.frames.numpy().dtype == s.motion.numpy().dtype == np.float16
        assert s.qb.tokens.numpy().dtype == s.qb.cls.numpy().dtype == np.float16
        want = stage_step(cfg, videos, queries, s.video_ids, pin=False, motion_videos=motion)
        assert np.array_equal(s.frames.numpy(), want.frames.numpy())
        assert np.array_equal(s.motion.numpy(), want.motion.numpy())
        assert np.array_equal(s.qb.tokens.numpy(), want.qb.tokens.numpy())
        assert s.h2d_bytes() == want.h2d_bytes()
