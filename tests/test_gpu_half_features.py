"""fp16 / bf16 feature storage on the GPU.  The contract is bit-identity: every entry point, and the whole path, given
16-bit features returns exactly (torch.equal / np.array_equal, never a tolerance) what it returns for the fp32 upcast
of the same features, in fp32 and tensor-core mode, with the same number of kernel launches."""
import ctypes as C
import dataclasses
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from cone_b200 import _lib, ingest
from cone_b200.config import EGO4D, MAD512, PRESETS
from cone_b200.engine import ConeEngine, pack_queries
from cone_b200.inference import MODES, evaluate_dataset, ground_dataset
from cone_b200.synth import make_dataset
from cone_b200.weights import init_state_dict

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HALF = {"fp16": torch.float16, "bf16": torch.bfloat16}

CASES = {
    "ego4d": (EGO4D.replace(eval_bsz=4), dict(n_videos=3, frames=[700, 130, 455], queries_per_video=[4, 2, 3], seed=21)),
    "mad512": (MAD512.replace(eval_bsz=3), dict(n_videos=2, frames=[1500, 600], queries_per_video=[4, 3], seed=5)),
}
_engines = {}


def _engine(cfg, precision, ws=1 << 30):
    key = (cfg, precision, ws)
    if key not in _engines:
        _engines[key] = ConeEngine(cfg, init_state_dict(cfg, 7), device=DEV, precision=precision, workspace_bytes=ws)
    return _engines[key]


def _half_ds(ds, np_dtype=np.float16):
    """(videos, motion, queries) of `ds` rounded to `np_dtype`, and the same values upcast back to float32."""
    v16 = [v.astype(np_dtype) for v in ds.videos]
    m16 = None if ds.motion is None else [m.astype(np_dtype) for m in ds.motion]
    q16 = [dataclasses.replace(q, tokens=q.tokens.astype(np_dtype), cls=q.cls.astype(np_dtype)) for q in ds.queries]
    up = lambda a: a.astype(np.float32)
    q32 = [dataclasses.replace(q, tokens=up(q.tokens), cls=up(q.cls)) for q in q16]
    return (v16, m16, q16), ([up(v) for v in v16], None if m16 is None else [up(m) for m in m16], q32)


def _counted(fn):
    """(fn(), kernels the library launched for it)"""
    _lib.reset_launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, _lib.launch_count()


def _assert_results_equal(a, b):
    assert a.keys() == b.keys()
    for k in a:
        ra, rb = a[k], b[k]
        assert ra.keys() == rb.keys(), k
        for f in ra:
            if isinstance(ra[f], np.ndarray):
                assert ra[f].dtype == rb[f].dtype and np.array_equal(ra[f], rb[f]), (k, f)
            else:
                assert ra[f] == rb[f], (k, f)


def _bits(t):
    """the tensor's bit patterns: NaN (absent windows pool an empty slice) compares equal to the same NaN"""
    return t.view({4: torch.int32, 8: torch.int64}[t.element_size()]) if t.is_floating_point() else t


def _assert_outputs_equal(a, b):
    for f in dataclasses.fields(a):
        x, y = getattr(a, f.name), getattr(b, f.name)
        assert (x is None) == (y is None), f.name
        if x is not None:
            assert x.dtype == y.dtype and torch.equal(_bits(x), _bits(y)), f.name


# ---------------------------------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("dt", list(HALF))
def test_l2_normalize_bitwise(dt):
    eng = _engine(EGO4D, "fp32", 64 << 20)
    g = torch.Generator().manual_seed(3)
    for D in (256, 512, 768, 1024, 2304, 4096):
        for rows in (1, 13, 1001):  # 8 rows per block: none of these fill whole blocks but 1
            x = (torch.randn(rows, D, generator=g) * 3 + 0.5).to(DEV).to(HALF[dt])
            x[0, :7] = 0  # zero runs and an all-zero row: eps = 0 divides by 0 in both paths alike
            if rows > 1:
                x[1] = 0
            for eps in (1e-5, 0.0, -1e-5):
                got = eng.l2_normalize(x, eps)
                want = eng.l2_normalize(x.float(), eps)
                assert got.dtype == torch.float32
                assert torch.equal(got.nan_to_num(7.0), want.nan_to_num(7.0)), (D, rows, eps)
                assert torch.equal(got.isnan(), want.isnan())
    # [Nq, max_q_l, Dt] token batches keep their shape
    t = torch.randn(5, 20, 768, device=DEV).half()
    assert torch.equal(eng.l2_normalize(t, 1e-5), eng.l2_normalize(t.float(), 1e-5))


def _prepare_ex(eng, frames, ws_bytes, ctx=True, vidproj=True):
    n = frames.shape[0]
    out_c = torch.empty((n, eng.cfg.v_feat_dim), dtype=torch.float32, device=DEV) if ctx else None
    out_v = torch.empty((n, eng.cfg.hidden_dim), dtype=torch.float32, device=DEV) if vidproj else None
    ws = torch.empty(int(ws_bytes), dtype=torch.uint8, device=DEV)
    code = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16, torch.bfloat16: _lib.DTYPE_BF16}[frames.dtype]
    p = lambda t: C.c_void_p(0 if t is None else t.data_ptr())
    _lib.check(eng.lib.cone_video_prepare_ex(eng._handle, p(frames), code, n, p(out_c), p(out_v), p(ws), ws.numel(),
                                             eng.precision, C.c_void_p(torch.cuda.current_stream().cuda_stream)),
               "cone_video_prepare_ex")
    return out_c, out_v


@pytest.mark.parametrize("precision", ["fp32", "tc"])
@pytest.mark.parametrize("cfg", [EGO4D, MAD512], ids=["ego4d", "mad512"])
@pytest.mark.parametrize("dt", list(HALF))
def test_video_prepare_bitwise(dt, cfg, precision):
    eng = _engine(cfg, precision)
    g = torch.Generator().manual_seed(cfg.v_feat_dim)
    x = (torch.randn(1000, cfg.v_feat_dim, generator=g) * 2 + 0.3).to(DEV).to(HALF[dt])
    ctx, vp = eng.video_prepare(x)
    ctx32, vp32 = eng.video_prepare(x.float())
    assert torch.equal(ctx, ctx32) and torch.equal(vp, vp32)
    # several slabs (at most 300 of the 1000 frames): the slab offset scales with the element size
    small = eng.lib.cone_prepare_workspace_bytes(C.byref(eng.dims), 300)
    c_s, v_s = _prepare_ex(eng, x, small)
    assert torch.equal(c_s, ctx32) and torch.equal(v_s, vp32)


@pytest.mark.parametrize("precision", ["fp32", "tc"])
@pytest.mark.parametrize("dm", [1024, 2304])
@pytest.mark.parametrize("dt", list(HALF))
def test_motion_prepare_bitwise(dt, dm, precision):
    cfg = EGO4D.replace(v_motion_feat_dim=dm)
    eng = _engine(cfg, precision)
    g = torch.Generator().manual_seed(dm)
    frames = torch.randn(1000, 256, generator=g).to(DEV)
    motion = (torch.randn(1000, dm, generator=g) * 2.0 + 0.3).to(DEV).to(HALF[dt])
    ctx, vp = eng.video_prepare(frames.to(HALF[dt]), motion=motion)
    ctx32, vp32 = eng.video_prepare(frames.to(HALF[dt]).float(), motion=motion.float())
    assert torch.equal(ctx, ctx32) and torch.equal(vp, vp32)
    _, vp_mixed = eng.video_prepare(frames, want_ctx=False, motion=motion)  # fp32 appearance, 16-bit motion
    assert torch.equal(vp_mixed, vp32)
    # slabs of at most 300 frames
    n = 1000
    out = torch.empty((n, cfg.hidden_dim), dtype=torch.float32, device=DEV)
    ws = torch.empty(int(eng.lib.cone_prepare_workspace_bytes(C.byref(eng.dims), 300)), dtype=torch.uint8, device=DEV)
    _lib.check(eng.lib.cone_video_prepare_motion_ex(eng._handle, C.c_void_p(motion.data_ptr()),
                                                    {"fp16": _lib.DTYPE_F16, "bf16": _lib.DTYPE_BF16}[dt], n,
                                                    C.c_void_p(out.data_ptr()), C.c_void_p(ws.data_ptr()), ws.numel(),
                                                    eng.precision, C.c_void_p(torch.cuda.current_stream().cuda_stream)),
               "cone_video_prepare_motion_ex")
    assert torch.equal(out, vp32)


@pytest.mark.parametrize("dt", list(HALF))
def test_prefilter_bitwise(dt):
    for cfg in (EGO4D, MAD512):
        eng = _engine(cfg, "fp32")
        g = torch.Generator().manual_seed(11)
        frames = torch.randn(2300, cfg.v_feat_dim, generator=g).to(DEV).to(HALF[dt])
        cls = torch.randn(9, cfg.v_feat_dim, generator=g).to(DEV).to(HALF[dt])
        want = eng.prefilter(frames.float(), cls.float(), want_scores=True)
        for f, c in ((frames, cls), (frames, cls.float()), (frames.float(), cls)):
            got = eng.prefilter(f, c, want_scores=True)
            assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


# ------------------------------------------------------------------------------------------------------ whole path
@pytest.mark.parametrize("precision", ["fp32", "tc"])
@pytest.mark.parametrize("name", list(CASES))
def test_ground_and_evaluate_dataset_bitwise(name, precision):
    cfg, dkw = CASES[name]
    ds = make_dataset(cfg, **dkw)
    (v16, _, q16), (v32, _, q32) = _half_ds(ds)
    eng = _engine(cfg, precision)
    b = ground_dataset(eng, v32, q32, max_frames_per_step=1000)  # also the warm-up: first use fills lazy weight caches
    a, n16 = _counted(lambda: ground_dataset(eng, v16, q16, max_frames_per_step=1000))
    b2, n32 = _counted(lambda: ground_dataset(eng, v32, q32, max_frames_per_step=1000))
    assert n16 == n32 > 0  # no hidden upcast pass
    _assert_results_equal(a, b)
    _assert_results_equal(b2, b)
    gt = {q.query_id: q.timestamps for q in ds.queries}
    for flavour in ("mad", "ego4d"):
        ca = evaluate_dataset(eng, v16, q16, gt, flavour=flavour, max_frames_per_step=1000)
        cb = evaluate_dataset(eng, v32, q32, gt, flavour=flavour, max_frames_per_step=1000)
        assert torch.equal(ca.hits, cb.hits) and torch.equal(ca.window_hits, cb.window_hits)
        assert torch.equal(ca.n_queries, cb.n_queries)
        assert len(ca.top1_iou) == len(cb.top1_iou) and all(torch.equal(x, y) for x, y in zip(ca.top1_iou, cb.top1_iou))


@pytest.mark.parametrize("precision", ["fp32", "tc"])
def test_engine_ground_bf16(precision):
    cfg, dkw = CASES["ego4d"]
    ds = make_dataset(cfg, **dkw)
    eng = _engine(cfg, precision)
    qb = pack_queries(cfg, [len(v) for v in ds.videos], ds.queries).to(DEV)
    frames = torch.from_numpy(np.concatenate(ds.videos)).to(DEV).bfloat16()
    qb16 = dataclasses.replace(qb, tokens=qb.tokens.bfloat16(), cls=qb.cls.bfloat16())
    qb32 = dataclasses.replace(qb, tokens=qb16.tokens.float(), cls=qb16.cls.float())
    eng.ground(frames.float(), qb32)  # warm-up: first use fills lazy weight caches
    a, n16 = _counted(lambda: eng.ground(frames, qb16, want_rows=True))
    b, n32 = _counted(lambda: eng.ground(frames.float(), qb32, want_rows=True))
    assert n16 == n32
    _assert_outputs_equal(a, b)
    # each feature tensor independently: bf16 frames with fp32 queries
    _assert_outputs_equal(eng.ground(frames, qb32, want_rows=True), b)


@pytest.mark.parametrize("precision", ["fp32", "tc"])
def test_two_streams_bitwise(precision):
    cfg = EGO4D.replace(eval_bsz=4, v_motion_feat_dim=2304)
    ds = make_dataset(cfg, 3, [700, 130, 455], [4, 2, 3], seed=21, motion_dim=2304)
    (v16, m16, q16), (v32, m32, q32) = _half_ds(ds)
    eng = _engine(cfg, precision)
    ground_dataset(eng, v32, q32, motion_videos=m32)  # warm-up: first use fills lazy weight caches
    want, n32 = _counted(lambda: ground_dataset(eng, v32, q32, motion_videos=m32))
    both, n16 = _counted(lambda: ground_dataset(eng, v16, q16, motion_videos=m16))
    assert n16 == n32
    _assert_results_equal(both, want)
    # fp16 motion next to fp32 appearance rows and queries
    want_m = ground_dataset(eng, ds.videos, ds.queries, motion_videos=m32)
    mixed, n_mixed = _counted(lambda: ground_dataset(eng, ds.videos, ds.queries, motion_videos=m16))
    assert n_mixed == n32
    _assert_results_equal(mixed, want_m)


def test_store_path_with_float16_records():
    cfg = EGO4D.replace(eval_bsz=2)
    ds = make_dataset(cfg, 3, [400, 90, 310], [2, 2, 2], seed=8)
    (v16, _, q16), _ = _half_ds(ds)
    eng = _engine(cfg, "fp32")
    want = ground_dataset(eng, v16, q16, max_frames_per_step=500, full=False)
    for videos, queries in ((v16, q16), (ds.videos, ds.queries)):  # fp16 records pass through, fp32 ones are rounded
        vs = ingest.DictStore({k: ingest.encode_record(features=v) for k, v in zip(ds.video_ids, videos)})
        qs = ingest.DictStore({q.query_id: ingest.encode_record(token_features=q.tokens, cls_features=q.cls)
                               for q in queries})
        got = ingest.ground_store(eng, vs, qs, ds.annotations(), max_frames_per_step=500, feature_dtype=np.float16)
        _assert_results_equal(got, want)


def test_refusals():
    cfg = EGO4D
    eng = _engine(cfg, "fp32")
    x64 = torch.randn(100, 256, device=DEV, dtype=torch.float64)
    with pytest.raises(TypeError, match="float32, float16 or bfloat16"):
        eng.l2_normalize(x64, 1e-5)
    with pytest.raises(TypeError):
        eng.video_prepare(x64)
    with pytest.raises(TypeError):
        eng.prefilter(x64.half(), x64[:3])
    # a contiguous 16-bit view one element into its storage: not 8-byte aligned
    flat = torch.randn(100 * 256 + 1, device=DEV).half()
    view = flat[1:].view(100, 256)
    assert view.is_contiguous() and view.data_ptr() % 8 != 0
    with pytest.raises(_lib.ConeError, match="not 8-byte aligned"):
        eng.l2_normalize(view, 1e-5)
    with pytest.raises(_lib.ConeError, match="not 8-byte aligned"):
        eng.video_prepare(view)
    # unknown dtype code at the C ABI
    out = torch.empty(100, 256, device=DEV)
    rc = eng.lib.cone_l2_normalize_ex(C.c_void_p(flat.data_ptr()), 7, C.c_void_p(out.data_ptr()), 100, 256, 1e-5,
                                      C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == -1 and b"unknown dtype" in eng.lib.cone_last_error()
    # the reference-shaped surface and the single-video front end stay fp32-only
    B, Lv, Lt = 2, cfg.max_v_l, cfg.max_q_l
    txt = torch.randn(B, Lt, cfg.t_feat_dim, device=DEV)
    vid = torch.randn(B, Lv, cfg.v_feat_dim, device=DEV)
    lens = torch.full((B,), 10, dtype=torch.int32, device=DEV)
    with pytest.raises(TypeError):
        eng.forward(txt.half(), lens, vid, lens)
    with pytest.raises(TypeError):
        eng.forward(txt, lens, vid.bfloat16(), lens)
    spans = torch.rand(B, 5, 2, device=DEV)
    with pytest.raises(TypeError):
        eng.clip_matching(torch.randn(B, cfg.v_feat_dim, device=DEV).half(), vid, lens, spans)
    with pytest.raises(TypeError):
        eng.clip_matching(torch.randn(B, cfg.v_feat_dim, device=DEV), vid.half(), lens, spans)
    with pytest.raises(TypeError):
        eng.prepare_video(vid[0].half())
    xn, ctx, vp = eng.prepare_video(vid[0])
    qb = pack_queries(cfg, [Lv], make_dataset(cfg, 1, [Lv], 1, seed=2).queries).to(DEV)
    with pytest.raises(TypeError):
        eng.ground_video(xn, ctx, vp, dataclasses.replace(qb, tokens=qb.tokens.half()))
    with pytest.raises(TypeError):
        eng.ground_video(xn.half(), ctx, vp, qb)
    torch.cuda.synchronize()


def test_sharded_eval_float16_matches_in_process():
    args = dict(config="ego4d", videos=3, queries=2, motion_dim=1024, seed=0)
    cmd = [sys.executable, "-m", "cone_b200.tools.sharded_eval", "--config", args["config"], "--videos", str(args["videos"]),
           "--queries", str(args["queries"]), "--motion-dim", str(args["motion_dim"]), "--frames", "300", "700",
           "--flavour", "ego4d", "--feature-dtype", "float16"]
    env = {k: v for k, v in os.environ.items() if k not in ("WORLD_SIZE", "RANK", "LOCAL_RANK")}
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    cfg = PRESETS["ego4d"].replace(eval_bsz=2, v_motion_feat_dim=1024)
    ds = make_dataset(cfg, 3, None, 2, seed=0, frames_range=(300, 700), motion_dim=1024)
    (v16, m16, q16), _ = _half_ds(ds)
    eng = ConeEngine(cfg, init_state_dict(cfg, 0), device=DEV, precision="fp32", workspace_bytes=4 << 30)  # as the tool
    c = evaluate_dataset(eng, v16, q16, {q.query_id: q.timestamps for q in ds.queries}, flavour="ego4d",
                         max_frames_per_step=1, motion_videos=m16)
    want = {"world": 1, "n_queries": int(c.n_queries.item()), "window_recall": c.window_recall().tolist()}
    for m in MODES:
        rec, miou = c.recall_ego4d(m)
        want[m] = {"recall": rec.tolist(), "mIoU": miou}
    assert got == json.loads(json.dumps(want))
