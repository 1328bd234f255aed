"""Separate motion and appearance feature streams on the GPU: the whole path against the two-stream oracle
(tests/motion_oracle.py) in fp32 and tensor-core mode, the drop-in module, the motion projection's slabbing, the
store-driven path and the refusals."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from cone_b200 import _lib, ingest
from cone_b200.config import EGO4D, MAD512
from cone_b200.engine import ConeEngine
from cone_b200.inference import ground_dataset, recall_at_k
from cone_b200.model import build_model
from cone_b200.synth import make_dataset
from cone_b200.weights import init_state_dict
from oracle import cone_oracle as O
import motion_oracle as MO
from helpers import FP32_TOL, ROUND_TOL, TC_TOL, assert_close, assert_match_close, dense_case, pooled_bounds, rows_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Ego4D: 256-d appearance + 2304-d SlowFast motion; MAD-512: 512-d CLIP appearance + 1024-d motion
CASES = {
    "ego4d_2304": (EGO4D.replace(eval_bsz=8, v_motion_feat_dim=2304), 21, dict(n_videos=4, frames=[900, 455, 91, 1300],
                                                                                queries_per_video=4, seed=33)),
    "mad512_1024": (MAD512.replace(eval_bsz=4, v_motion_feat_dim=1024), 4, dict(n_videos=2, frames=[2000, 700],
                                                                                 queries_per_video=[4, 3], seed=9)),
}
_cache = {}


def _case(name):
    if name not in _cache:
        cfg, wseed, dkw = CASES[name]
        sd = init_state_dict(cfg, wseed)
        ds = make_dataset(cfg, motion_dim=cfg.v_motion_feat_dim, **dkw)
        _cache[name] = (cfg, sd, ds, MO.eval_pipeline(sd, cfg, ds.videos, ds.queries, motion_videos=ds.motion))
    return _cache[name]


@pytest.mark.parametrize("name", list(CASES))
def test_two_streams_fp32_vs_oracle(name):
    cfg, sd, ds, ora = _case(name)
    eng = ConeEngine(cfg, sd, device=DEV, precision="fp32", workspace_bytes=3 << 30)
    res = ground_dataset(eng, ds.videos, ds.queries, motion_videos=ds.motion)
    span_tol = ROUND_TOL + 2e-5 * max(len(v) for v in ds.videos) * cfg.clip_length
    flips = 0
    n_same = 0
    for q in ds.queries:
        r, o = res[q.query_id], ora[q.query_id]
        assert sorted(r["ranklist"]) == sorted(o["ranklist"])
        assert r["ranklist"][: cfg.topk_window] == o["ranklist"][: cfg.topk_window], q.query_id
        assert r["windows"] == o["windows"], q.query_id
        assert_close(r["pred_spans"], np.stack(o["pred_spans"]), FP32_TOL, "pred_spans")
        assert_close(r["prob_fg"], np.stack(o["prob_fg"]), FP32_TOL, "prob_fg")
        f = assert_match_close(r["match"], np.stack(o["match"]), np.stack(o["pred_spans"]), [n for _, n in r["windows"]],
                               FP32_TOL)
        flips += f
        n_same += all(rows_close(r[m], o[m], span_tol) for m in ("fusion", "proposal", "matching"))
    # NMS keep-lists: the same rows in the same order, up to the 4-decimal rounding; only a query whose matching score
    # crossed a floor/ceil pooling boundary may differ
    assert n_same >= len(ds.queries) - flips, (n_same, len(ds.queries), flips)
    gt = {q.query_id: list(q.timestamps) for q in ds.queries}
    for mode in ("fusion", "proposal", "matching"):
        want = O.recall_at_k_iou({q.query_id: ora[q.query_id][mode] for q in ds.queries}, gt)
        assert np.array_equal(np.round(recall_at_k(res, gt, mode=mode) * len(ds.queries)),
                              np.round(want * len(ds.queries))), mode
    # the motion stream is what Moment-DETR reads: without it the same handle refuses, and projecting the
    # appearance rows instead would give other proposals
    with pytest.raises(ValueError, match="motion"):
        ground_dataset(eng, ds.videos, ds.queries)


@pytest.mark.parametrize("name", list(CASES))
def test_two_streams_tc_vs_oracle(name):
    cfg, sd, ds, ora = _case(name)
    eng = ConeEngine(cfg, sd, device=DEV, precision="tc", workspace_bytes=3 << 30)
    res = ground_dataset(eng, ds.videos, ds.queries, motion_videos=ds.motion)
    errs, n_prop, n_flip = [], 0, 0
    for q in ds.queries:
        r, o = res[q.query_id], ora[q.query_id]
        assert r["ranklist"][: cfg.topk_window] == o["ranklist"][: cfg.topk_window], q.query_id  # fp32 in every mode
        assert r["windows"] == o["windows"]
        osp = np.stack(o["pred_spans"])
        errs.append(np.abs(r["pred_spans"] - osp).ravel())
        errs.append(np.abs(r["prob_fg"] - np.stack(o["prob_fg"])).ravel())
        # matching scores where both sides pool the same rows; proposals whose floor/ceil bounds moved are counted
        dur = np.asarray([n for _, n in r["windows"]], dtype=np.float32)[:, None]
        same = np.all(pooled_bounds(r["pred_spans"], dur) == pooled_bounds(osp, dur), axis=0)
        dm = np.abs(r["match"] - np.stack(o["match"]))
        assert dm[same].max() <= TC_TOL, f"{q.query_id}: match differs by {dm[same].max():.3e} on identical pooled rows"
        n_prop += same.size
        n_flip += int((~same).sum())
    err = np.concatenate(errs)
    print(f"[tc-two-streams] {name}: n {err.size} max {err.max():.3e} rms {np.sqrt(np.mean(err ** 2)):.3e}; "
          f"pooled-row bounds differ for {n_flip} of {n_prop} proposals")
    assert err.max() <= TC_TOL, f"{name}: max error {err.max():.3e} > {TC_TOL}"
    assert n_flip <= 0.08 * n_prop


@pytest.mark.parametrize("precision,tol", [("fp32", FP32_TOL), ("tc", TC_TOL)])
def test_drop_in_module_with_a_motion_feature_dim(precision, tol):
    opt = SimpleNamespace(v_appear_feat_dim=256, v_motion_feat_dim=2304, t_feat_dim=768, max_v_l=90, max_q_l=20,
                          precision=precision, aux_loss=True)
    model, _ = build_model(opt)
    cfg = model.cfg
    sd = init_state_dict(cfg, 3)
    model.load_state_dict(sd)
    model = model.to(DEV).eval()
    app, vm, txt, tm, cls = dense_case(EGO4D, 103)  # appearance rows [B, 90, 256], text, CLS
    g = torch.Generator().manual_seed(17)
    mot = torch.randn(app.shape[0], app.shape[1], 2304, generator=g) * vm[..., None]
    mot = mot / (mot.norm(dim=-1, keepdim=True) + 1e-5)  # what the dataloader hands the model
    with torch.no_grad():
        want = O.cone_forward(sd, txt, tm, mot, vm)
        wmatch = O.clip_matching(sd, cls, app, vm, want["pred_spans"])
    out = model(src_txt=txt.to(DEV), src_txt_mask=tm.to(DEV), src_vid_motion=mot.to(DEV), src_vid_motion_mask=vm.to(DEV))
    assert_close(out["pred_spans"].cpu(), want["pred_spans"], tol, "pred_spans")
    assert_close(torch.softmax(out["pred_logits"], -1).cpu(), torch.softmax(want["pred_logits"], -1), tol, "class probabilities")
    assert_close(out["aux_outputs"][0]["pred_spans"].cpu(), want["aux_outputs"][0]["pred_spans"], tol, "aux_spans")
    if precision == "fp32":
        assert_close(out["saliency_scores"].cpu(), want["saliency_scores"], tol, "saliency")
    match = model.forward_clip_matching(src_cls_txt=cls.to(DEV), src_vid_appear=app.to(DEV), src_vid_appear_mask=vm.to(DEV),
                                        proposal=want["pred_spans"].to(DEV))
    assert_close(match.cpu(), wmatch, tol, "match")


def _prepare_motion(eng, motion, ws_bytes):
    n = motion.shape[0]
    out = torch.empty((n, eng.cfg.hidden_dim), dtype=torch.float32, device=DEV)
    ws = torch.empty(int(ws_bytes), dtype=torch.uint8, device=DEV)
    rc = eng.lib.cone_video_prepare_motion(eng._handle, C.c_void_p(motion.data_ptr()), n, C.c_void_p(out.data_ptr()),
                                           C.c_void_p(ws.data_ptr()), ws.numel(), eng.precision,
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, "cone_video_prepare_motion")
    return out


@pytest.mark.parametrize("precision", ["fp32", "tc"])
@pytest.mark.parametrize("dm", [1024, 2304, 4096])
def test_motion_projection_widths_and_slabs(precision, dm):
    """l2norm_rows, the LayerNorm rows kernel, split3 and tc_gemm (K = Dm, 3 Dm) on Dm-wide rows against the oracle's
    projection of the normalised rows; a workspace that forces several slabs gives the same bits as one slab."""
    cfg = EGO4D.replace(v_motion_feat_dim=dm)
    sd = init_state_dict(cfg, 5)
    eng = ConeEngine(cfg, sd, device=DEV, precision=precision, workspace_bytes=1 << 30)
    g = torch.Generator().manual_seed(dm)
    motion = torch.randn(1000, dm, generator=g) * 2.0 + 0.3
    with torch.no_grad():
        want = O.input_proj(sd, "input_vid_proj", torch.from_numpy(O.l2_normalize_np(motion.numpy())))
    m = motion.to(DEV)
    dims = eng.dims
    one = _prepare_motion(eng, m, eng.lib.cone_prepare_workspace_bytes(C.byref(dims), 1000))
    small = eng.lib.cone_prepare_workspace_bytes(C.byref(dims), 300)
    many = _prepare_motion(eng, m, small)  # slabs of at most 300 of the 1000 frames
    assert torch.equal(one, many)
    _, vp = eng.video_prepare(torch.zeros(1000, 256, device=DEV), want_ctx=False, motion=m)
    assert torch.equal(vp, one)
    err = (one.cpu() - want).abs().max().item()
    print(f"[motion-proj] Dm {dm} {precision}: max |diff| vs oracle {err:.2e}")
    assert_close(one.cpu(), want, FP32_TOL if precision == "fp32" else 1e-4, f"vidproj Dm={dm} {precision}")


def test_store_path_equals_in_memory_path():
    cfg = EGO4D.replace(eval_bsz=2, v_motion_feat_dim=2304)
    ds = make_dataset(cfg, 3, [400, 90, 310], [2, 2, 2], seed=8, motion_dim=2304)
    vs = ingest.DictStore({k: ingest.encode_record(features=v) for k, v in zip(ds.video_ids, ds.videos)})
    ms = ingest.DictStore({k: ingest.encode_record(features=m) for k, m in zip(ds.video_ids, ds.motion)})
    qs = ingest.DictStore({q.query_id: ingest.encode_record(token_features=q.tokens, cls_features=q.cls) for q in ds.queries})
    eng = ConeEngine(cfg, init_state_dict(cfg, 2), device=DEV, precision="fp32", workspace_bytes=1 << 30)
    a = ingest.ground_store(eng, vs, qs, ds.annotations(), max_frames_per_step=500, motion_store=ms)
    b = ground_dataset(eng, ds.videos, ds.queries, max_frames_per_step=500, full=False, motion_videos=ds.motion)
    assert a.keys() == b.keys()
    for k in a:
        assert a[k] == b[k]


def test_refusals():
    cfg = EGO4D.replace(v_motion_feat_dim=2304)
    eng = ConeEngine(cfg, init_state_dict(cfg, 0), device=DEV, precision="fp32", workspace_bytes=256 << 20)
    frames = torch.randn(100, 256, device=DEV)
    vp = torch.empty(100, 256, device=DEV)
    ws, nb = eng._wsargs()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    # raw appearance rows are no motion input for this handle
    rc = eng.lib.cone_video_prepare(eng._handle, C.c_void_p(frames.data_ptr()), 100, None, C.c_void_p(vp.data_ptr()),
                                    ws, nb, _lib.PREC_FP32, stream)
    assert rc == -1 and b"cone_video_prepare_motion" in eng.lib.cone_last_error()
    # the stage-0 context alone is still served
    ctx = torch.empty_like(frames)
    rc = eng.lib.cone_video_prepare(eng._handle, C.c_void_p(frames.data_ptr()), 100, C.c_void_p(ctx.data_ptr()), None,
                                    ws, nb, _lib.PREC_FP32, stream)
    assert rc == 0
    with pytest.raises(ValueError, match="motion"):
        eng.video_prepare(frames)
    with pytest.raises(ValueError, match="one row per appearance frame"):
        eng.video_prepare(frames, motion=torch.randn(99, 2304, device=DEV))
    with pytest.raises(ValueError, match="one row per appearance frame"):
        eng.video_prepare(frames, motion=torch.randn(100, 1024, device=DEV))
    # m_dim % 16 != 0 is refused when the handle is created
    with pytest.raises(_lib.ConeError, match="motion feature dim"):
        ConeEngine(EGO4D.replace(v_motion_feat_dim=2300), init_state_dict(EGO4D.replace(v_motion_feat_dim=2300), 0),
                   device=DEV)
    torch.cuda.synchronize()
