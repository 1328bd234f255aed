"""Exhaustive grounding on the GPU: stage 3 past the shared-memory limit (cone_fuse_nms_ws) against the oracle's
`postprocess_query` and bitwise against cone_fuse_nms_ex, stage 2 split inside one query's windows, and the whole path
with topk_window = every window of the longest video against `eval_pipeline`."""
import ctypes as C

import numpy as np
import pytest
import torch

from cone_b200 import _lib
from cone_b200._lib import ConeError
from cone_b200.config import EGO4D
from cone_b200.engine import ConeEngine, _ptr, _stream, pack_queries
from cone_b200.inference import MODES, evaluate_dataset, ground_dataset, recall_at_k
from cone_b200.synth import make_dataset
from cone_b200.weights import init_state_dict
from oracle import cone_oracle as O
from helpers import FP32_TOL, ROUND_TOL, TC_TOL, Hatch, assert_close, assert_match_close, oracle_window_scores, \
    pooled_bounds, ranklist_near_tie, rows_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
_cache = {}


def _engine():
    if "eng" not in _cache:
        _cache["eng"] = ConeEngine(EGO4D, init_state_dict(EGO4D, 0), device=DEV, precision="fp32", workspace_bytes=1 << 30)
    return _cache["eng"]


# ---------------------------------------------------------------------------------------------- stage 3 alone
def _stage3_inputs(nq, k, ns, seed, n_present, dur=90, clip=0.53333):
    """Raw outputs of k overlapping windows (stride dur/2) per query, with ties, repeated (st, ed) pairs and -0.0 starts.
    n_present[j] windows of query j are present (the rest have length 0)."""
    rng = np.random.default_rng(seed)
    half = dur // 2
    cx = rng.uniform(0.05, 0.95, (nq, k, ns))
    w = rng.uniform(0.02, 0.6, (nq, k, ns))
    # the second half of window t is the first half of window t + 1: the same seconds from two windows
    rep = rng.random((nq, k)) < 0.3
    cx[:, :, 0] = np.where(rep, 0.75, cx[:, :, 0]); w[:, :, 0] = np.where(rep, 0.5, w[:, :, 0])
    if ns > 1:
        cx[:, 1:, 1] = np.where(rep[:, :-1], 0.25, cx[:, 1:, 1]); w[:, 1:, 1] = np.where(rep[:, :-1], 0.5, w[:, 1:, 1])
    # spans of the first window that start just below 0 (round4 gives -0.0) or exactly at 0, with the same end
    cx[:, 0, 0], w[:, 0, 0] = 5e-7, 2e-6
    if ns > 2:
        cx[:, 0, 2], w[:, 0, 2] = 7.5e-7, 1.5e-6
    spans = np.stack([cx, w], -1).astype(np.float32)
    prob = np.round(rng.uniform(0, 1, (nq, k, ns)), 2).astype(np.float32)  # many ties
    match = rng.uniform(-1, 1, (nq, k, ns)).astype(np.float32)
    wstart = np.broadcast_to(np.arange(k, dtype=np.int32) * half, (nq, k)).copy()
    wlen = np.zeros((nq, k), dtype=np.int32)
    for j, n in enumerate(n_present):
        wlen[j, :n] = dur
    cfg = EGO4D.replace(topk_window=k, num_queries=ns, clip_length=clip)
    return cfg, [torch.from_numpy(a) for a in (spans, prob, match, wstart, wlen)]


def _oracle_fused(cfg, spans, prob, match, wstart, wlen):
    out = []
    for j in range(prob.shape[0]):
        rows = []
        for t in range(int((wlen[j] > 0).sum())):
            rows.extend(O.compose_window_rows(spans[j, t], prob[j, t], match[j, t], int(wlen[j, t]), int(wstart[j, t]),
                                              cfg.clip_length))
        out.append((rows, O.score_fusion(rows) if rows else {}))
    return out


def _ws_call(eng, cfg, t, fixed_duration=0, sort_within_window=True, ws_bytes=None):
    """cone_fuse_nms_ws on the engine's workspace (or on `ws_bytes` of it), outputs laid out like ConeEngine.fuse_nms"""
    spans, prob, match, wstart, wlen = [x.to(DEV) for x in t]
    nq_, k, ns = prob.shape
    out = torch.zeros((nq_, 3, cfg.max_after_nms, 5), dtype=torch.float64, device=DEV)
    cnt = torch.zeros((nq_, 3), dtype=torch.int32, device=DEV)
    rows = torch.zeros((nq_, k * ns, 4), dtype=torch.float64, device=DEV)
    rcnt = torch.zeros((nq_,), dtype=torch.int32, device=DEV)
    ws, nb = eng._wsargs(eng.lib.cone_fuse_nms_workspace_bytes(nq_, k, ns))
    _lib.check(eng.lib.cone_fuse_nms_ws(_ptr(spans), _ptr(prob), _ptr(match), _ptr(wstart), _ptr(wlen), nq_, k, ns,
                                        float(np.float32(cfg.clip_length)), float(cfg.nms_thd), cfg.max_before_nms,
                                        cfg.max_after_nms, fixed_duration, int(sort_within_window), _ptr(out), _ptr(cnt),
                                        _ptr(rows), _ptr(rcnt), ws, nb if ws_bytes is None else ws_bytes, _stream()),
               "cone_fuse_nms_ws")
    return out, cnt, rows, rcnt


FULL = [(thd, mb, ma) for thd in (-1, 0.5) for mb in (1, 200, 1 << 30) for ma in (1, 5, 10)]
SOME = [(-1, 200, 10), (0.5, 1, 5), (0.5, 200, 10), (0.5, 1 << 30, 1), (0.5, 1 << 30, 10)]
# (k, slots, present windows per query, knob sets): N = 2202 (one past the shared-memory limit), 4360 (872 x 5, a MAD
# movie), 14 525 (2905 x 5, the stress video) and 131 072 (16 384 x 8, the longest rank-list)
SIZES = [(1101, 2, [1101, 700, 0], FULL), (872, 5, [872, 500, 0], FULL), (2905, 5, [2905, 1900, 0], SOME),
         (16384, 8, [16384, 9000], SOME)]


@pytest.mark.parametrize("k,ns,present,knobs", SIZES, ids=[f"N{k * ns}" for k, ns, _, _ in SIZES])
def test_fuse_nms_ws_vs_oracle(k, ns, present, knobs):
    eng = _engine()
    cfg, t = _stage3_inputs(len(present), k, ns, k, present)
    fused = _oracle_fused(cfg, *t)
    for thd, mb, ma in knobs:
        c2 = cfg.replace(nms_thd=thd, max_before_nms=mb, max_after_nms=ma)
        out, cnt, rows, rcnt = eng.fuse_nms(*[x.to(DEV) for x in t], want_rows=True, cfg=c2)  # the workspace path
        out, cnt, rows, rcnt = out.cpu().numpy(), cnt.cpu().numpy(), rows.cpu().numpy(), rcnt.cpu().numpy()
        for j, (orows, of) in enumerate(fused):
            assert rcnt[j] == len(orows)
            assert rows[j, : rcnt[j]].tolist() == orows, (j, "rows")
            for m, (key, idx) in enumerate((("fusion", 2), ("proposal", 0), ("matching", 1))):
                want = O.post_processing_nms(of, idx, thd, mb, ma) if orows else []
                assert out[j, m, : cnt[j, m]].tolist() == want, (thd, mb, ma, j, key)
    assert any(x[0] == 0 and np.signbit(x[0]) for r, _ in fused for x in r), "no -0.0 start in the inputs"
    assert any(len(f) < len(r) for r, f in fused if r), "no repeated (st, ed) pair in the inputs"


def _bits(*ts):
    return [x.cpu().contiguous().view(torch.int64 if x.dtype == torch.float64 else torch.int32).numpy() for x in ts]


@pytest.mark.parametrize("variant", ["eval_epoch", "front_end"])
def test_fuse_nms_ws_is_bitwise_the_shared_memory_kernel(variant):
    """At N <= 2201 both entry points run on the same inputs, including those where the oracle's Python sort has no
    defined order (NaN scores and matches, from empty pooling slices) and -0.0 next to +0.0 and constant scores."""
    eng = _engine()
    kw = dict(fixed_duration=90, sort_within_window=False) if variant == "front_end" else {}
    for case, (k, ns) in enumerate([(30, 5), (440, 5), (275, 8), (1, 1)]):
        cfg, t = _stage3_inputs(4, k, ns, 100 + case, [k, max(k // 2, 1), 1, 0])
        spans, prob, match, wstart, wlen = t
        if case == 0:
            prob[0, 3, :] = float("nan"); match[0, 5, 1] = float("nan"); match[2, 0, 0] = float("nan")
            prob[1] = 0.5  # constant score over the whole query
            match[1, :, :] = -0.0
            match[1, ::2, :] = 0.0
        for thd, mb, ma in [(0.5, 200, 10), (-1, 200, 5), (0.5, 1 << 30, 10), (0.5, 1, 1)]:
            c2 = cfg.replace(nms_thd=thd, max_before_nms=mb, max_after_nms=ma)
            want = eng.fuse_nms(*[x.to(DEV) for x in t], want_rows=True, cfg=c2, **kw)
            got = _ws_call(eng, c2, t, **kw)
            for a, b, name in zip(_bits(*got), _bits(*want), ("out", "count", "rows", "rows_count")):
                assert np.array_equal(a, b), (variant, case, thd, mb, ma, name)


def test_fuse_nms_ws_chunks_and_refusals():
    eng = _engine()
    cfg, t = _stage3_inputs(5, 600, 5, 7, [600, 600, 300, 1, 0])
    want = _ws_call(eng, cfg, t)
    one = eng.lib.cone_fuse_nms_workspace_bytes(1, 600, 5)
    for nb in (one, 2 * one + 17):  # one and two queries per launch
        assert all(np.array_equal(a, b) for a, b in zip(_bits(*_ws_call(eng, cfg, t, ws_bytes=nb)), _bits(*want)))
    with pytest.raises(ConeError, match="cannot hold one query"):
        _ws_call(eng, cfg, t, ws_bytes=one - 1)
    big = [torch.zeros((1, 16385, 8, 2)), torch.zeros((1, 16385, 8)), torch.zeros((1, 16385, 8)),
           torch.zeros((1, 16385), dtype=torch.int32), torch.zeros((1, 16385), dtype=torch.int32)]
    with pytest.raises(ConeError, match="131072"):
        eng.fuse_nms(*[x.to(DEV) for x in big], cfg=cfg.replace(topk_window=16385, num_queries=8))


def test_stage3_of_a_150_candidate_step_is_one_launch():
    eng = _engine()
    cfg, t = _stage3_inputs(64, 30, 5, 3, [30] * 64)
    args = [x.to(DEV) for x in t]
    eng.fuse_nms(*args, cfg=cfg)
    torch.cuda.synchronize()
    _lib.reset_launch_count()
    eng.fuse_nms(*args, cfg=cfg)
    assert _lib.launch_count() == 1


# ---------------------------------------------------------------------------------------------- the whole path
def _e2e():
    """Ego4D dims at max_v_l = 6 (stride 3): 1000-2400 windows per query, every one of them grounded"""
    if "e2e" not in _cache:
        base = EGO4D.replace(max_v_l=6, eval_bsz=2)
        ds = make_dataset(base, 3, [3100, 5000, 7200], [2, 1, 2], seed=11)
        cfg = base.replace(topk_window=base.num_window(7200))
        sd = init_state_dict(cfg, 6)
        _cache["e2e"] = (cfg, sd, ds, O.eval_pipeline(sd, cfg, ds.videos, ds.queries))
    return _cache["e2e"]


def _check_exhaustive(cfg, sd, ds, res, ora, name, tc):
    """Against `eval_pipeline`, window by window.  Every window is grounded, so both sides hold the same windows; with
    thousands of windows per query, DIFFERENT frames whose scores lie within 1e-7 are common, and CPU and GPU fp32 may
    order such near-ties differently (SURVEY.md §7 H1).  Rank-lists must therefore be equal up to audited near-tie
    swaps, and each window's outputs are compared with the oracle's outputs for the same window.  A query whose
    candidate order moved (a swap) or whose matching score crossed a pooling boundary may end with other NMS'd lists;
    so may, counted, one other query in fp32 mode (4-decimal rounding of a 1e-7 difference).  Returns the queries whose
    lists differ."""
    swaps = Hatch(name, "rank-list differs from the oracle's by near-tie swaps", len(ds.queries))
    lists = Hatch(name, "NMS'd list differs from the oracle's with no swap or pooling-boundary flip",
                  len(ds.queries) if tc else 1)
    span_tol = ROUND_TOL + (TC_TOL if tc else 2e-5) * max(len(v) for v in ds.videos) * cfg.clip_length
    differ, n_prop, n_flip = [], 0, 0
    for q in ds.queries:
        r, o = res[q.query_id], ora[q.query_id]
        swapped = r["ranklist"] != o["ranklist"]
        if swapped:
            ws = oracle_window_scores(sd, cfg, ds, q)
            assert ranklist_near_tie(ws, r["ranklist"], o["ranklist"], len(o["ranklist"])), q.query_id
            swaps.use(q.query_id)
        n = len(o["windows"])
        assert len(r["windows"]) == n and sorted(r["ranklist"][:n]) == sorted(o["ranklist"][:n]), q.query_id
        pos = {w: i for i, w in enumerate(r["ranklist"][:n])}
        perm = [pos[w] for w in o["ranklist"][:n]]  # GPU window index of each oracle window
        assert [r["windows"][i] for i in perm] == o["windows"], q.query_id
        sp, pr, mt = r["pred_spans"][perm], r["prob_fg"][perm], r["match"][perm]
        osp = np.stack(o["pred_spans"])
        tol = TC_TOL if tc else FP32_TOL
        assert_close(sp, osp, tol, "pred_spans")
        assert_close(pr, np.stack(o["prob_fg"]), tol, "prob_fg")
        dur = np.asarray([ln for _, ln in o["windows"]], dtype=np.float32)[:, None]
        if tc:
            same = np.all(pooled_bounds(sp, dur) == pooled_bounds(osp, dur), axis=0)
            dm = np.abs(mt - np.stack(o["match"]))
            assert dm[same].max() <= TC_TOL, q.query_id
            n_prop += same.size
            flips = int((~same).sum())
            n_flip += flips
        else:
            flips = assert_match_close(mt, np.stack(o["match"]), osp, dur[:, 0], FP32_TOL)
        if any(not rows_close(r[m], o[m], span_tol) for m in MODES):
            differ.append(q.query_id)
            if not swapped and not flips:
                lists.use(q.query_id)
    swaps.close(len(ds.queries))
    lists.close(len(ds.queries))
    assert n_flip <= 0.08 * max(n_prop, 1)
    return differ


def test_exhaustive_fp32_vs_oracle_and_metric_counters():
    cfg, sd, ds, ora = _e2e()
    assert cfg.topk_window * cfg.num_queries > _lib.FUSE_NMS_MAX_SHARED_CANDIDATES
    eng = ConeEngine(cfg, sd, device=DEV, precision="fp32", workspace_bytes=4 << 30)
    res = ground_dataset(eng, ds.videos, ds.queries)
    assert max(len(r["windows"]) for r in res.values()) == cfg.topk_window
    differ = _check_exhaustive(cfg, sd, ds, res, ora, "fp32 exhaustive", tc=False)
    # the device counters are the recall of the device's lists, and the oracle's wherever the lists agree
    gt = {q.query_id: list(q.timestamps) for q in ds.queries}
    c = evaluate_dataset(eng, ds.videos, ds.queries, gt)
    same = [q for q in ds.queries if q.query_id not in differ]
    assert same
    for mode in MODES:
        hits = c.hits[MODES.index(mode)].cpu().numpy()
        assert np.array_equal(hits, np.round(recall_at_k(res, gt, mode=mode) * len(ds.queries)).astype(np.int64)), mode
        want = O.recall_at_k_iou({q.query_id: ora[q.query_id][mode] for q in same}, gt)
        got = recall_at_k({q.query_id: res[q.query_id] for q in same}, gt, mode=mode)
        assert np.array_equal(np.round(got * len(same)), np.round(want * len(same))), mode


def test_exhaustive_tc_vs_oracle():
    cfg, sd, ds, ora = _e2e()
    eng = ConeEngine(cfg, sd, device=DEV, precision="tc", workspace_bytes=4 << 30)
    _check_exhaustive(cfg, sd, ds, ground_dataset(eng, ds.videos, ds.queries), ora, "tc exhaustive", tc=True)


def _assert_results_equal(a, b):
    assert a.keys() == b.keys()
    for q in a:
        assert a[q].keys() == b[q].keys(), q
        for f in a[q]:
            x, y = a[q][f], b[q][f]
            if isinstance(x, np.ndarray):
                assert x.dtype == y.dtype and np.array_equal(x, y, equal_nan=True), (q, f)
            else:
                assert x == y, (q, f)


@pytest.mark.parametrize("precision", ["fp32", "tc"])
def test_stage2_inside_one_query_is_bitwise(precision):
    """64 MB hold a few hundred of the 2401 windows of one query: stage 2 runs each query in window ranges"""
    cfg, sd, ds, _ = _e2e()
    dims = _lib.ConeDims(cfg.v_feat_dim, cfg.t_feat_dim, cfg.hidden_dim, cfg.nheads, cfg.dim_feedforward, cfg.enc_layers,
                         cfg.dec_layers, cfg.num_queries, cfg.max_v_l, cfg.max_q_l, cfg.v_motion_feat_dim)
    assert _lib.load().cone_workspace_bytes(C.byref(dims), cfg.topk_window, cfg.max_v_l, cfg.max_q_l) > 64 << 20
    big = ConeEngine(cfg, sd, device=DEV, precision=precision, workspace_bytes=4 << 30)
    want = ground_dataset(big, ds.videos, ds.queries)
    del big
    small = ConeEngine(cfg, sd, device=DEV, precision=precision, workspace_bytes=64 << 20)
    _assert_results_equal(ground_dataset(small, ds.videos, ds.queries), want)


def test_stage2_refuses_a_workspace_without_room_for_one_window():
    cfg, sd, ds, _ = _e2e()
    big = ConeEngine(cfg, sd, device=DEV, precision="fp32", workspace_bytes=1 << 30)
    v = torch.from_numpy(ds.videos[0]).to(DEV)
    prepared = big.video_prepare(v)
    qs = [q for q in ds.queries if q.video_idx == 0]
    qb = pack_queries(cfg, [len(ds.videos[0])], qs).to(DEV)
    tiny = ConeEngine(cfg, sd, device=DEV, precision="fp32", workspace_bytes=16 << 10)
    with pytest.raises(ConeError, match="cannot hold one window"):
        tiny.ground(v, qb, prepared=prepared)


def test_first_windows_of_an_exhaustive_run_are_the_top30_run():
    cfg, sd, ds, _ = _e2e()
    ex = ground_dataset(ConeEngine(cfg, sd, device=DEV, precision="tc", workspace_bytes=4 << 30), ds.videos, ds.queries)
    c30 = cfg.replace(topk_window=30)
    top = ground_dataset(ConeEngine(c30, sd, device=DEV, precision="tc", workspace_bytes=4 << 30), ds.videos, ds.queries)
    for q in ds.queries:
        a, b = ex[q.query_id], top[q.query_id]
        assert a["windows"][:30] == b["windows"]
        assert np.array_equal(a["pred_spans"][:30], b["pred_spans"]), q.query_id
        assert np.array_equal(a["prob_fg"][:30], b["prob_fg"]), q.query_id
