"""Separate motion and appearance feature streams (`--v_motion_feat_dim` != `--v_appear_feat_dim`), host side: state-dict
layout, blob sizing in the library, configuration, staging, and the two-stream oracle.  No compute calls."""
import ctypes as C
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from cone_b200 import _lib, build, ingest
from cone_b200.config import EGO4D, MAD512
from cone_b200.inference import stage_step
from cone_b200.model import build_model, config_from_opt
from cone_b200.synth import make_dataset
from cone_b200.weights import check_state_dict, init_state_dict, state_dict_shapes
from oracle import cone_oracle as O
import motion_oracle as MO

EGO4D_SF = EGO4D.replace(v_motion_feat_dim=2304)  # Ego4D CLIP appearance + SlowFast motion


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _dims(cfg):
    return _lib.ConeDims(cfg.v_feat_dim, cfg.t_feat_dim, cfg.hidden_dim, cfg.nheads, cfg.dim_feedforward, cfg.enc_layers,
                         cfg.dec_layers, cfg.num_queries, cfg.max_v_l, cfg.max_q_l, cfg.v_motion_feat_dim)


def test_state_dict_sizes_input_vid_proj_by_the_motion_dim():
    s, base = state_dict_shapes(EGO4D_SF), state_dict_shapes(EGO4D)
    assert list(s) == list(base)
    assert s["input_vid_proj.0.LayerNorm.weight"] == (2304,) and s["input_vid_proj.0.LayerNorm.bias"] == (2304,)
    assert s["input_vid_proj.0.net.1.weight"] == (256, 2304)
    # everything else, the adapter (appearance, Dv) and the second projection layer included, is unchanged
    changed = {k for k in s if s[k] != base[k]}
    assert changed == {"input_vid_proj.0.LayerNorm.weight", "input_vid_proj.0.LayerNorm.bias", "input_vid_proj.0.net.1.weight"}
    assert s["adapter_layer.layers.0.weight"] == (256, 256) and s["adapter_layer.layers.1.weight"] == (256, 256)
    # a motion dim equal to Dv is the single-stream layout
    assert state_dict_shapes(EGO4D.replace(v_motion_feat_dim=256)) == base


@pytest.mark.parametrize("cfg", [EGO4D, MAD512])
@pytest.mark.parametrize("dm", [1024, 2304])
def test_blob_size_and_workspaces_cover_the_motion_dim(lib, cfg, dm):
    two = cfg.replace(v_motion_feat_dim=dm)
    d2 = _dims(two)
    assert lib.cone_weights_expected_floats(C.byref(d2)) == sum(math.prod(x) for x in state_dict_shapes(two).values())
    # m_dim 0 and m_dim = Dv describe the same single-stream model
    d0, dv = _dims(cfg), _dims(cfg.replace(v_motion_feat_dim=cfg.v_feat_dim))
    for f in (lambda d: lib.cone_weights_expected_floats(C.byref(d)),
              lambda d: lib.cone_prepare_workspace_bytes(C.byref(d), 5000),
              lambda d: lib.cone_workspace_bytes(C.byref(d), 64, cfg.max_v_l, cfg.max_q_l)):
        assert f(d0) == f(dv) > 0
    # the frame stage and the dense forward stage Dm-wide rows: their workspace grows with Dm
    n = 5000
    assert lib.cone_prepare_workspace_bytes(C.byref(d2), n) >= lib.cone_prepare_workspace_bytes(C.byref(d0), n) + n * 4 * (dm - cfg.v_feat_dim)
    assert lib.cone_workspace_bytes(C.byref(d2), 64, cfg.max_v_l, cfg.max_q_l) > lib.cone_workspace_bytes(C.byref(d0), 64, cfg.max_v_l, cfg.max_q_l)


def test_motion_dim_must_be_a_multiple_of_16(lib):
    bad = _dims(EGO4D.replace(v_motion_feat_dim=2300))
    assert lib.cone_weights_expected_floats(C.byref(bad)) == 0
    assert b"motion feature dim" in lib.cone_last_error()
    # refused at handle creation too, before any device work
    blob = np.zeros(16, dtype=np.float32)
    h = C.c_void_p(0)
    rc = lib.cone_weights_create(blob.ctypes.data_as(C.c_void_p), blob.size, C.byref(bad), None, C.byref(h))
    assert rc == -1 and not h.value
    assert b"motion feature dim" in lib.cone_last_error()


def test_check_state_dict_refuses_a_single_stream_dict_for_a_two_stream_config():
    sd = init_state_dict(EGO4D, 0)
    check_state_dict(EGO4D, sd)
    with pytest.raises(ValueError, match="input_vid_proj.0"):
        check_state_dict(EGO4D_SF, sd)
    check_state_dict(EGO4D_SF, init_state_dict(EGO4D_SF, 0))


def _opt(**kw):
    o = dict(v_appear_feat_dim=256, v_motion_feat_dim=2304, t_feat_dim=768, max_v_l=90, max_q_l=20)
    o.update(kw)
    return SimpleNamespace(**o)


def test_config_from_opt_and_build_model_accept_distinct_dims():
    cfg = config_from_opt(_opt())
    assert (cfg.v_feat_dim, cfg.v_motion_feat_dim, cfg.motion_dim) == (256, 2304, 2304)
    assert config_from_opt(_opt(v_motion_feat_dim=256)).motion_dim == 256
    model, _ = build_model(_opt())
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    assert shapes["input_vid_proj.0.net.1.weight"] == (256, 2304)
    assert shapes["adapter_layer.layers.0.weight"] == (256, 256)
    model.load_state_dict(init_state_dict(cfg, 1))  # a two-stream checkpoint loads into it
    # the training-side variants still raise
    with pytest.raises(NotImplementedError):
        build_model(_opt(use_txt_pos=True))


def test_synthetic_motion_stream_keeps_the_appearance_data():
    a = make_dataset(EGO4D, 3, [120, 75, 200], 2, seed=4)
    b = make_dataset(EGO4D, 3, [120, 75, 200], 2, seed=4, motion_dim=2304)
    assert a.motion is None
    assert all(np.array_equal(x, y) for x, y in zip(a.videos, b.videos))
    assert all(np.array_equal(p.tokens, q.tokens) and np.array_equal(p.cls, q.cls) for p, q in zip(a.queries, b.queries))
    assert [m.shape for m in b.motion] == [(120, 2304), (75, 2304), (200, 2304)]
    assert all(m.dtype == np.float32 for m in b.motion)
    c = make_dataset(EGO4D, 3, [120, 75, 200], 2, seed=4, motion_dim=2304)
    assert all(np.array_equal(x, y) for x, y in zip(b.motion, c.motion))


def test_oracle_without_motion_equals_the_single_stream_oracle_exactly():
    cfg = EGO4D.replace(eval_bsz=4)
    sd = init_state_dict(cfg, 7)
    ds = make_dataset(cfg, 3, [300, 91, 455], [3, 2, 3], seed=12)
    want = O.eval_pipeline(sd, cfg, ds.videos, ds.queries)
    got = MO.eval_pipeline(sd, cfg, ds.videos, ds.queries)
    assert got.keys() == want.keys()
    for k in want:
        assert got[k].keys() == want[k].keys()
        for f in want[k]:
            if f in ("pred_spans", "prob_fg", "match"):
                assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(got[k][f], want[k][f])), (k, f)
            else:
                assert got[k][f] == want[k][f], (k, f)


def test_oracle_two_streams_rank_on_appearance_and_ground_on_motion():
    cfg = EGO4D.replace(eval_bsz=4, v_motion_feat_dim=512)
    sd = init_state_dict(cfg, 7)
    ds = make_dataset(cfg, 2, [300, 120], [2, 2], seed=3, motion_dim=512)
    got = MO.eval_pipeline(sd, cfg, ds.videos, ds.queries, motion_videos=ds.motion)
    # stage 1 reads the appearance stream only
    for q in ds.queries:
        with torch.no_grad():
            ctx = O.stage0_video_context(sd, torch.from_numpy(O.l2_normalize_np(ds.videos[q.video_idx])))
            rl, _ = O.stage1_ranklist(ctx, torch.from_numpy(O.l2_normalize_np(q.cls)), cfg.max_v_l)
        assert got[q.query_id]["ranklist"] == rl
    # stage 2 of one window by hand: normalised motion rows into Moment-DETR, raw appearance rows into the pooling
    q = ds.queries[0]
    s, n = got[q.query_id]["windows"][0]
    tok, cls_n = O.prepare_query_text(q.tokens, q.cls, cfg.max_q_l)
    mot = torch.from_numpy(O.l2_normalize_np(ds.motion[q.video_idx][s: s + n]))[None]
    app = torch.from_numpy(ds.videos[q.video_idx][s: s + n])[None]
    with torch.no_grad():
        out = O.cone_forward(sd, tok[None], torch.ones(1, len(tok)), mot, torch.ones(1, n))
        match = O.clip_matching(sd, torch.from_numpy(cls_n)[None], app, torch.ones(1, n), out["pred_spans"])
    assert np.allclose(got[q.query_id]["pred_spans"][0], out["pred_spans"][0].numpy(), atol=1e-6)
    assert np.allclose(got[q.query_id]["match"][0], match[0].numpy(), atol=1e-6)


def test_stream_length_mismatch_raises():
    cfg = EGO4D_SF.replace(eval_bsz=2)
    ds = make_dataset(cfg, 2, [120, 75], [2, 1], seed=4, motion_dim=2304)
    short = [ds.motion[0], ds.motion[1][:-1]]
    with pytest.raises(ValueError, match="motion rows"):
        stage_step(cfg, ds.videos, ds.queries, [0, 1], pin=False, motion_videos=short)
    with pytest.raises(ValueError, match="motion rows"):
        MO.eval_pipeline(init_state_dict(cfg, 0), cfg, ds.videos, ds.queries, motion_videos=short)
    with pytest.raises(ValueError, match="motion feature tensors"):
        MO.eval_pipeline(init_state_dict(cfg, 0), cfg, ds.videos, ds.queries, motion_videos=ds.motion[:1])


def test_staging_carries_the_motion_stream():
    cfg = EGO4D_SF.replace(eval_bsz=2)
    ds = make_dataset(cfg, 3, [200, 90, 310], [2, 1, 3], seed=6, motion_dim=2304)
    one = stage_step(cfg, ds.videos, ds.queries, [0, 2], pin=False)
    two = stage_step(cfg, ds.videos, ds.queries, [0, 2], pin=False, motion_videos=ds.motion)
    assert one.motion is None and torch.equal(one.frames, two.frames)
    assert torch.equal(two.motion, torch.from_numpy(np.concatenate([ds.motion[0], ds.motion[2]])))
    assert two.h2d_bytes() == one.h2d_bytes() + 510 * 2304 * 4
    # from feature stores: the motion records use the same keys and the same `features` array
    vs = ingest.DictStore({k: ingest.encode_record(features=v) for k, v in zip(ds.video_ids, ds.videos)})
    ms = ingest.DictStore({k: ingest.encode_record(features=m) for k, m in zip(ds.video_ids, ds.motion)})
    lens = [len(v) for v in ds.videos]
    steps = list(ingest.StagedSteps(cfg, vs, ds.video_ids, lens, ds.queries, max_frames_per_step=300, pin=False,
                                    motion_store=ms))
    assert [s.video_ids for s in steps] == [[0, 1], [2]]
    for s in steps:
        want = stage_step(cfg, ds.videos, ds.queries, s.video_ids, pin=False, motion_videos=ds.motion)
        assert torch.equal(s.frames, want.frames) and torch.equal(s.motion, want.motion)
    bad = ingest.DictStore({k: ingest.encode_record(features=m[:-3]) for k, m in zip(ds.video_ids, ds.motion)})
    with pytest.raises(ValueError, match="motion rows"):
        list(ingest.StagedSteps(cfg, vs, ds.video_ids, lens, ds.queries, max_frames_per_step=300, pin=False,
                                motion_store=bad))


def test_single_video_front_end_refuses_two_streams():
    from cone_b200.localizer import CONELocalizator
    with pytest.raises(NotImplementedError, match="one feature stream"):
        CONELocalizator(init_state_dict(EGO4D_SF, 0), cfg=EGO4D_SF)
