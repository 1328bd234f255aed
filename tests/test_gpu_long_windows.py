"""Windows of 257 to 512 rows (max_v_l + max_q_l) on the GPU: the long-window attention kernels against the CPU oracle in
fp32 and tensor-core mode, through the whole grounding path, the drop-in module, the single-video front end, fp16
features, a motion stream, small workspaces, CONE_ATTN_TC=1 and the refusals past 512 rows.  (231, 25) is the
longest window of the short-window kernels and is checked with the same criteria.

Run as a script (`python tests/test_gpu_long_windows.py attn-tc OUT.npz`) it writes the tensor-core outputs of the
(300, 77) case, so that a subprocess can run them with CONE_ATTN_TC=1, which the library reads once per process."""
import dataclasses
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from cone_b200._lib import ConeError
from cone_b200.config import EGO4D, MAD512
from cone_b200.engine import ConeEngine
from cone_b200.inference import MODES, ground_dataset, recall_at_k
from cone_b200.model import CONE
from cone_b200.synth import make_dataset
from cone_b200.weights import init_state_dict
from oracle import cone_oracle as O
from oracle.make_golden_localizer import localizer_case
import motion_oracle as MO
from helpers import FP32_TOL, ROUND_TOL, TC_TOL, Hatch, assert_close, assert_match_close, rows_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (max_v_l, max_q_l): S = 256 (short-window kernels), 257, 377 (CLIP's 77 tokens), 512
SHAPES = [(231, 25), (232, 25), (300, 77), (480, 32)]
_cache = {}


def _cfg(lv, lt, **kw):
    return EGO4D.replace(max_v_l=lv, max_q_l=lt, topk_window=5, eval_bsz=4, **kw)


def _lengths(lv):
    """several windows with a partial last one (the first is always half-length), one window plus a bit, and a video
    shorter than one window"""
    return [int(2.7 * lv) + 1, lv + lv // 3, lv // 2 + 17]


def _data(lv, lt):
    """seeded weights and a 3-video, 7-query dataset; token counts run past max_q_l (truncation)"""
    cfg = _cfg(lv, lt)
    return cfg, init_state_dict(cfg, lv), make_dataset(cfg, 3, _lengths(lv), [3, 2, 2], seed=lv + lt)


def _case(lv, lt):
    if (lv, lt) not in _cache:
        cfg, sd, ds = _data(lv, lt)
        _cache[lv, lt] = (cfg, sd, ds, O.eval_pipeline(sd, cfg, ds.videos, ds.queries))
    return _cache[lv, lt]


def _check_fp32(cfg, ds, res, ora, name):
    """rank-lists and windows exact, raw outputs within 1e-5, R@K identical, NMS'd lists equal up to the 4-decimal rounding.
    A query whose matching score crossed a floor/ceil pooling boundary may differ; so may, counted, one other query per
    case: the candidates are sorted on scores rounded to 4 decimals (inference.py:83), a 1e-7 difference that moves one
    rounding reorders rounded ties, and NMS then keeps another row.  The (231, 25) case, which runs the short-window
    kernels, has one such query."""
    span_tol = ROUND_TOL + 2e-5 * max(len(v) for v in ds.videos) * cfg.clip_length
    hatch = Hatch(name, "NMS'd list differs from the oracle's with no pooling-boundary flip", 1)
    flips = n_same = 0
    for q in ds.queries:
        r, o = res[q.query_id], ora[q.query_id]
        assert r["ranklist"] == o["ranklist"], q.query_id
        assert r["windows"] == o["windows"], q.query_id
        assert_close(r["pred_spans"], np.stack(o["pred_spans"]), FP32_TOL, "pred_spans")
        assert_close(r["prob_fg"], np.stack(o["prob_fg"]), FP32_TOL, "prob_fg")
        f = assert_match_close(r["match"], np.stack(o["match"]), np.stack(o["pred_spans"]),
                               [n for _, n in r["windows"]], FP32_TOL)
        flips += f
        diff = [m for m in MODES if not rows_close(r[m], o[m], span_tol)]
        n_same += not diff
        if diff and not f:
            hatch.use(f"{q.query_id} {diff}")
    used = hatch.close(len(ds.queries))
    assert n_same >= len(ds.queries) - flips - used, (n_same, len(ds.queries), flips)
    gt = {q.query_id: list(q.timestamps) for q in ds.queries}
    for mode in MODES:
        want = O.recall_at_k_iou({q.query_id: ora[q.query_id][mode] for q in ds.queries}, gt)
        assert np.array_equal(np.round(recall_at_k(res, gt, mode=mode) * len(ds.queries)),
                              np.round(want * len(ds.queries))), mode


def _bounds(spans, dur):
    """[start, end) pooled-row bounds as model.py:186-192 computes them in fp32 (clipping aside)."""
    sp = np.asarray(spans, dtype=np.float32)
    x1 = (sp[..., 0] - np.float32(0.5) * sp[..., 1]) * dur
    x2 = (sp[..., 0] + np.float32(0.5) * sp[..., 1]) * dur
    return np.stack([np.maximum(np.floor(x1), 0), np.ceil(x2)])


def _check_tc(cfg, ds, res, ora, name):
    """The criteria of tests/test_gpu_tc.py: identical top-k windows (the ranking is fp32 in every mode), spans and
    probabilities within TC_TOL, matching scores within TC_TOL where both sides pool the same rows, at most 8 % of the
    proposals with moved pooling bounds, R@K hit counts equal up to max(1, 0.5 % of the queries)."""
    errs, n_prop, n_flip = [], 0, 0
    for q in ds.queries:
        r, o = res[q.query_id], ora[q.query_id]
        assert r["ranklist"][: cfg.topk_window] == o["ranklist"][: cfg.topk_window], q.query_id
        assert r["windows"] == o["windows"], q.query_id
        osp = np.stack(o["pred_spans"])
        errs.append(np.abs(r["pred_spans"] - osp).ravel())
        errs.append(np.abs(r["prob_fg"] - np.stack(o["prob_fg"])).ravel())
        dur = np.asarray([n for _, n in r["windows"]], dtype=np.float32)[:, None]
        same = np.all(_bounds(r["pred_spans"], dur) == _bounds(osp, dur), axis=0)
        dm = np.abs(r["match"] - np.stack(o["match"]))
        assert dm[same].max() <= TC_TOL, f"{q.query_id}: match differs by {dm[same].max():.3e} on identical pooled rows"
        n_prop += same.size
        n_flip += int((~same).sum())
    err = np.concatenate(errs)
    print(f"[tc-long] {name}: n {err.size} max {err.max():.3e} rms {np.sqrt(np.mean(err ** 2)):.3e}; "
          f"pooled-row bounds differ for {n_flip} of {n_prop} proposals")
    assert err.max() <= TC_TOL, f"{name}: max error {err.max():.3e} > {TC_TOL}"
    assert n_flip <= 0.08 * n_prop
    gt = {q.query_id: list(q.timestamps) for q in ds.queries}
    n = len(ds.queries)
    for mode in MODES:
        want = O.recall_at_k_iou({q.query_id: ora[q.query_id][mode] for q in ds.queries}, gt)
        dev = np.abs(np.round(recall_at_k(res, gt, mode=mode) * n) - np.round(want * n)).max()
        assert dev <= max(1, 0.005 * n), (name, mode)


def _assert_results_equal(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].keys() == b[k].keys(), k
        for f in a[k]:
            x, y = a[k][f], b[k][f]
            if isinstance(x, np.ndarray):
                assert x.dtype == y.dtype and np.array_equal(x, y, equal_nan=True), (k, f)
            else:
                assert x == y, (k, f)


@pytest.mark.parametrize("lv,lt", SHAPES)
def test_long_windows_fp32_vs_oracle(lv, lt):
    cfg, sd, ds, ora = _case(lv, lt)
    eng = ConeEngine(cfg, sd, device=DEV, precision="fp32", workspace_bytes=2 << 30)
    _check_fp32(cfg, ds, ground_dataset(eng, ds.videos, ds.queries), ora, f"fp32 {lv}+{lt}")


@pytest.mark.parametrize("lv,lt", SHAPES)
def test_long_windows_tc_vs_oracle(lv, lt):
    cfg, sd, ds, ora = _case(lv, lt)
    eng = ConeEngine(cfg, sd, device=DEV, precision="tc", workspace_bytes=2 << 30)
    _check_tc(cfg, ds, ground_dataset(eng, ds.videos, ds.queries), ora, f"{lv}+{lt}")


def _dense(cfg, lt, seed):
    """a dense padded batch with ragged lengths (1 frame and 1 token included), as start_end_collate emits it"""
    g = torch.Generator().manual_seed(seed)
    lv = cfg.max_v_l
    vlen, tlen = [lv, lv // 2, 1, lv - 1], [lt, 5, lt // 2, 1]
    B = len(vlen)
    vid = torch.randn(B, lv, cfg.v_feat_dim, generator=g)
    txt = torch.randn(B, lt, cfg.t_feat_dim, generator=g)
    txt = txt / (txt.norm(dim=-1, keepdim=True) + 1e-5)
    cls = torch.randn(B, cfg.v_feat_dim, generator=g)
    cls = cls / (cls.norm(dim=-1, keepdim=True) + 1e-5)
    vm, tm = torch.zeros(B, lv), torch.zeros(B, lt)
    for i in range(B):
        vm[i, : vlen[i]] = 1
        tm[i, : tlen[i]] = 1
        vid[i, vlen[i]:] = 0
        txt[i, tlen[i]:] = 0
    return vid, vm, txt, tm, cls


@pytest.mark.parametrize("precision", ["fp32", "tc"])
@pytest.mark.parametrize("lv,lt", [(260, 40), (480, 32)])
def test_drop_in_forward_and_matching(lv, lt, precision):
    cfg = _cfg(lv, lt)
    sd = init_state_dict(cfg, 3)
    model = CONE(cfg, sd, precision=precision, aux_loss=True).to(DEV).eval()
    vid, vm, txt, tm, cls = _dense(cfg, lt, lv + lt)
    with torch.no_grad():
        want = O.cone_forward(sd, txt, tm, vid, vm)
        wmatch = O.clip_matching(sd, cls, vid, vm, want["pred_spans"])
    out = model(src_txt=txt.to(DEV), src_txt_mask=tm.to(DEV), src_vid_motion=vid.to(DEV), src_vid_motion_mask=vm.to(DEV))
    match = model.forward_clip_matching(cls.to(DEV), vid.to(DEV), vm.to(DEV), proposal=want["pred_spans"].to(DEV))
    prob = lambda x: torch.softmax(x.cpu(), -1)
    if precision == "fp32":
        assert_close(out["pred_logits"].cpu(), want["pred_logits"], FP32_TOL, "pred_logits")
        assert_close(out["pred_spans"].cpu(), want["pred_spans"], FP32_TOL, "pred_spans")
        assert_close(out["saliency_scores"].cpu(), want["saliency_scores"], FP32_TOL, "saliency")
        assert_close(out["aux_outputs"][0]["pred_spans"].cpu(), want["aux_outputs"][0]["pred_spans"], FP32_TOL, "aux_spans")
        assert_close(out["aux_outputs"][0]["pred_logits"].cpu(), want["aux_outputs"][0]["pred_logits"], FP32_TOL,
                     "aux_logits")
        assert_close(match.cpu(), wmatch, FP32_TOL, "match")
    else:  # the criteria of tests/test_gpu_tc.py::test_tc_forward_dense_vs_oracle
        assert_close(out["pred_spans"].cpu(), want["pred_spans"], TC_TOL, "pred_spans")
        assert_close(prob(out["pred_logits"]), prob(want["pred_logits"]), TC_TOL, "class probabilities")
        assert_close(match.cpu(), wmatch, TC_TOL, "match")


def test_localizer_predict_moment_at_300_frames():
    from cone_b200.localizer import CONELocalizator
    cfg = MAD512.replace(max_v_l=300, max_before_nms=100, nms_thd=0.5, max_after_nms=5)
    sd = init_state_dict(cfg, 8)
    v, tok, cls = localizer_case(cfg, 1700, 17, 41)
    loc = CONELocalizator(sd, device=DEV, cfg=cfg, use_cuda_graph=False)
    got = loc.predict_moment(v, (tok, cls))
    ora = O.predict_moment(sd, cfg, torch.from_numpy(v), torch.from_numpy(tok), torch.from_numpy(cls))
    # tests/test_localizer.py's tolerances: the min-max fusion of 4-decimal scores amplifies one rounding step
    assert len(got) == len(ora["moments"]), (got, ora["moments"])
    for a, b in zip(got, ora["moments"]):
        assert abs(a[0] - b[0]) <= 2e-4 and abs(a[1] - b[1]) <= 2e-4 and abs(a[2] - b[2]) <= 5e-4, (a, b)
    qb = loc._query_batch(len(v), torch.from_numpy(tok), torch.from_numpy(cls)).to(DEV)
    out = loc._run(qb)
    assert [int(x) for x in out.ranklist[0].cpu().tolist() if x >= 0] == ora["ranklist"]
    k = len(ora["windows"])
    assert [(int(s), int(n)) for s, n in zip(out.win_start[0, :k].cpu(), out.win_len[0, :k].cpu())] == ora["windows"]
    for key in ("pred_spans", "prob_fg", "match"):
        assert np.abs(getattr(out, key)[0, :k].cpu().numpy() - ora[key]).max() <= FP32_TOL, key


def test_fp16_features_are_bitwise_their_upcast():
    cfg, sd, ds, _ = _case(300, 77)
    eng = ConeEngine(cfg, sd, device=DEV, precision="tc", workspace_bytes=2 << 30)
    v16 = [v.astype(np.float16) for v in ds.videos]
    q16 = [dataclasses.replace(q, tokens=q.tokens.astype(np.float16), cls=q.cls.astype(np.float16)) for q in ds.queries]
    v32 = [v.astype(np.float32) for v in v16]
    q32 = [dataclasses.replace(q, tokens=q.tokens.astype(np.float32), cls=q.cls.astype(np.float32)) for q in q16]
    _assert_results_equal(ground_dataset(eng, v16, q16), ground_dataset(eng, v32, q32))


def test_motion_stream_fp32_vs_oracle():
    cfg = _cfg(300, 77, v_motion_feat_dim=1024)
    sd = init_state_dict(cfg, 12)
    ds = make_dataset(cfg, 3, _lengths(300), [2, 2, 1], seed=12, motion_dim=1024)
    ora = MO.eval_pipeline(sd, cfg, ds.videos, ds.queries, motion_videos=ds.motion)
    eng = ConeEngine(cfg, sd, device=DEV, precision="fp32", workspace_bytes=2 << 30)
    _check_fp32(cfg, ds, ground_dataset(eng, ds.videos, ds.queries, motion_videos=ds.motion), ora, "fp32 motion 300+77")


@pytest.mark.parametrize("precision", ["fp32", "tc"])
def test_small_workspace_chunks_are_bit_identical(precision):
    """64 MB hold about two queries of five 512-row windows: the seven queries run in several chunks"""
    cfg, sd, ds, _ = _case(480, 32)
    big = ConeEngine(cfg, sd, device=DEV, precision=precision, workspace_bytes=2 << 30)
    want = ground_dataset(big, ds.videos, ds.queries)
    del big
    small = ConeEngine(cfg, sd, device=DEV, precision=precision, workspace_bytes=64 << 20)
    _assert_results_equal(ground_dataset(small, ds.videos, ds.queries), want)


def _attn_tc_case():
    cfg, sd, ds = _data(300, 77)
    eng = ConeEngine(cfg, sd, device=DEV, precision="tc", workspace_bytes=2 << 30)
    res = ground_dataset(eng, ds.videos, ds.queries)
    return {f"{qid}/{f}": np.asarray(r[f]) for qid, r in res.items() for f in ("ranklist", "pred_spans", "prob_fg", "match")}


def test_attn_tc_opt_in_falls_back_for_long_windows(tmp_path):
    """The tcgen05 attention supports at most 192 padded keys: with CONE_ATTN_TC=1 a 377-row window runs the mma.sync
    long-window kernel through enc_attn_tc_supported, so the outputs are the same bits as without the variable."""
    out = tmp_path / "attn_tc.npz"
    env = dict(os.environ, CONE_ATTN_TC="1", PYTHONPATH=os.pathsep.join([ROOT, os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "attn-tc", str(out)], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    got = dict(np.load(out))
    want = _attn_tc_case()
    assert got.keys() == want.keys()
    for k in want:
        assert got[k].dtype == want[k].dtype and np.array_equal(got[k], want[k], equal_nan=True), k


def test_refusals_past_512_rows():
    cfg = _cfg(488, 25)
    with pytest.raises(ConeError, match="512"):
        ConeEngine(cfg, init_state_dict(cfg, 1), device=DEV)
    cfg = _cfg(480, 32)
    eng = ConeEngine(cfg, init_state_dict(cfg, 1), device=DEV, precision="tc", workspace_bytes=1 << 30)
    vid = torch.randn(2, 480, cfg.v_feat_dim, device=DEV)
    vl = torch.tensor([480, 100], dtype=torch.int32, device=DEV)
    for lt in (33, 40):  # Lv + Lt = 513, 520
        txt = torch.randn(2, lt, cfg.t_feat_dim, device=DEV)
        with pytest.raises(ConeError, match="512"):
            eng.forward(txt, torch.tensor([lt, 3], dtype=torch.int32, device=DEV), vid, vl)
    # nothing faulted: the same handle runs the longest accepted window
    logits, spans, _, _, _ = eng.forward(torch.randn(2, 32, cfg.t_feat_dim, device=DEV),
                                         torch.tensor([32, 3], dtype=torch.int32, device=DEV), vid, vl)
    torch.cuda.synchronize()
    assert torch.isfinite(spans).all() and torch.isfinite(logits).all()


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "attn-tc":
        np.savez(sys.argv[2], **_attn_tc_case())
    else:
        raise SystemExit(__doc__)
