"""The window pre-filter (stages 0-1) against float64 and exact-order references.

- Rank-lists (`cone_window_ranklist`) at every sort size the kernel takes, 32 to 16 384 keys (the 64 KB and 128 KB
  shared-memory opt-ins included), on synthetic frame scores with ties, NaN, +-0, +-inf and +-FLT_MAX: bit-identical to
  `torch.sort(descending=True, stable=True)` of the window maxima `torch.max` takes over the same slices.
- The grouped frame-score GEMM (`cone_frame_scores`) against an fp64 einsum under the rigorous bound of a sequential fp32
  FMA chain, and bitwise: alone or among other videos, with its queries permuted, against `cone_linear` (fp32), and with
  caller-chosen `score_offsets` (padded rows, reversed rows).
- Stage-0 context features against the oracle in float64, and bitwise across precision modes and workspace slabs.
- `cone_l2_normalize(_ex)` in its three eps forms against float64; `cone_prefilter` at the sort boundaries; the engine
  past 4096 windows per query.

Prints one `[prefilter] ...` line per case with its largest errors."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from cone_b200 import _lib
from cone_b200._lib import ConeError
from cone_b200.config import EGO4D
from cone_b200.engine import ConeEngine, _ptr, _stream
from cone_b200.inference import ground_dataset
from cone_b200.synth import make_dataset
from cone_b200.weights import init_state_dict
from oracle import cone_oracle as O
import fp64_reference as R
from helpers import FP32_TOL, Hatch, axis_cfg

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MAX_WINDOWS = 16384  # the longest rank-list cone_window_ranklist sorts
NW_SIZES = (1, 2, 31, 32, 33, 255, 256, 257, 4096, 4097, 8192, 8193, 16383, 16384)
VALUE_CLASSES = ("random", "ties", "constant", "nan", "zeros", "inf", "fltmax")
FLT_MAX = float(np.finfo(np.float32).max)
SENTINEL = 0x7FBADBAD  # a NaN bit pattern no kernel writes
_cache = {}


# ---------------------------------------------------------------------------------------------- reference helpers
def num_window(L, max_v_l):
    return math.ceil(L / int(max_v_l / 2)) + 1


def frames_for_windows(nw, max_v_l):
    """the frame count whose rank-list has nw windows (nw 1: an empty video)"""
    return (nw - 1) * int(max_v_l / 2)


def ref_window_scores(fs: torch.Tensor, max_v_l: int) -> torch.Tensor:
    """torch.max over each window's slice fs[s:e] (cone/inference.py:286-296), exact and NaN-propagating: the slices are
    gathered into one [nw, max_v_l] matrix padded with -inf, which changes no maximum of a non-empty slice.  An empty
    video's single window (the reference's torch.max would raise) is -inf, as the kernel writes it."""
    L = fs.numel()
    stride = int(max_v_l / 2)
    nw = num_window(L, max_v_l)
    start = torch.clamp((torch.arange(nw) - 1) * stride, min=0)
    end = torch.clamp((torch.arange(nw) - 1) * stride + max_v_l, max=L)
    idx = start[:, None] + torch.arange(max_v_l)[None, :]
    valid = idx < end[:, None]
    padded = torch.cat([fs.float(), torch.tensor([-math.inf])])
    return torch.where(valid, padded[torch.where(valid, idx, L)], torch.tensor(-math.inf)).max(dim=1).values


def ref_ranklist(ws: torch.Tensor) -> torch.Tensor:
    return torch.sort(ws, descending=True, stable=True).indices


def kernel_order(ws: np.ndarray) -> np.ndarray:
    """The kernel's ordering restated on the host: ascending 64-bit keys (~orderable(score) << 32) | index, where
    orderable maps NaN to the largest key and -0.0 to +0.0 (prefilter.cu)."""
    ws = np.asarray(ws, np.float32)
    u = (ws + np.float32(0.0)).view(np.uint32).astype(np.uint64)
    o = np.where(u & 0x80000000, ~u & 0xFFFFFFFF, u | 0x80000000)
    o = np.where(np.isnan(ws), 0xFFFFFFFF, o).astype(np.uint64)
    keys = ((~o & 0xFFFFFFFF) << np.uint64(32)) | np.arange(len(ws), dtype=np.uint64)
    return np.argsort(keys, kind="stable")


def synth_scores(kind: str, L: int, max_v_l: int, g: torch.Generator) -> torch.Tensor:
    """frame scores of one value class"""
    if L == 0:
        return torch.zeros(0)
    pick = lambda vals: torch.tensor(vals)[torch.randint(len(vals), (L,), generator=g)]
    if kind == "random":
        return torch.randn(L, generator=g)
    if kind == "ties":
        return torch.randint(0, 4, (L,), generator=g).float() / 4
    if kind == "constant":
        return torch.full((L,), 0.375)
    if kind == "zeros":
        return pick([0.0, -0.0, -0.0, -1.0])
    if kind == "inf":
        return torch.where(torch.rand(L, generator=g) < 0.5, pick([math.inf, -math.inf]), torch.randn(L, generator=g))
    if kind == "fltmax":
        return pick([FLT_MAX, -FLT_MAX, 3e38, -3e38, 0.0])
    assert kind == "nan"
    x = torch.randn(L, generator=g)
    x[int(torch.randint(L, (1,), generator=g))] = math.nan  # a single NaN
    x[torch.randint(L, (max(1, L // 500),), generator=g)] = math.nan  # repeated NaN
    nw = num_window(L, max_v_l)
    w = int(torch.randint(nw, (1,), generator=g))  # one window made entirely of NaN
    s, e = max((w - 1) * int(max_v_l / 2), 0), min((w - 1) * int(max_v_l / 2) + max_v_l, L)
    x[s:e] = math.nan
    return x


def fp64_scores(ctx, cls):
    """fp64 einsum of fp32 inputs and the scale of the rigorous error bound of a K-step fp32 FMA chain"""
    a, b = cls.double().cpu(), ctx.double().cpu()
    return a @ b.T, a.abs() @ b.abs().T


def audit_vs_oracle(ows, got, want, hatch, what, rel=1e-5):
    """A device rank-list against the oracle's fp32 one over every window.  The two compute frame scores in different
    summation orders (SURVEY.md §7 H1), so over thousands of windows windows whose scores lie within an ulp may swap,
    and a swap shifts the windows between them (an exactly tied pair can move as a block past a third window).  So the
    check is on inversions, not positions: both lists hold the same windows, and no window follows another in the device
    order whose oracle score is more than `rel` (relative to max(1, |s|)) below it.  Each violation is a hatch use
    (limit 0).  Returns the number of positions where the lists differ."""
    s = np.asarray(ows, np.float64)
    got, want = np.asarray(got), np.asarray(want)
    assert sorted(got.tolist()) == sorted(want.tolist()), what
    sg = s[got]
    later_max = np.maximum.accumulate(sg[::-1])[::-1]  # the best oracle score at or after each device position
    for p in np.nonzero(later_max[1:] - sg[:-1] > rel * np.maximum(1.0, np.abs(sg[:-1])))[0]:
        hatch.use(f"{what} position {p}: window {got[p]} is followed by one {later_max[p + 1] - sg[p]:.2e} above it")
    return int((got != want).sum())


# ---------------------------------------------------------------------------------------------- engines
def _engine(cfg=EGO4D, precision="fp32", ws=1 << 30, seed=0):
    key = (cfg, precision, ws, seed)
    if key not in _cache:
        _cache[key] = ConeEngine(cfg, _sd(cfg, seed), device=DEV, precision=precision, workspace_bytes=ws)
    return _cache[key]


def _sd(cfg, seed=0):
    key = ("sd", cfg, seed)
    if key not in _cache:
        _cache[key] = init_state_dict(cfg, seed)
    return _cache[key]


def _lib_ranklist(scores, offsets, counts, max_v_l, stride, winscore_margin=0):
    """cone_window_ranklist straight through the C ABI (no host-side checks); winscore has `winscore_margin` spare
    floats after the last row, filled with the sentinel and checked untouched."""
    lib = _lib.load()
    nq = counts.numel()
    rl = torch.full((nq, stride), -7, dtype=torch.int32, device=DEV)
    ws = torch.full((nq * stride + winscore_margin,), SENTINEL, dtype=torch.int32, device=DEV).view(torch.float32)
    _lib.check(lib.cone_window_ranklist(_ptr(scores), _ptr(offsets), _ptr(counts), nq, max_v_l, _ptr(rl), _ptr(ws),
                                        stride, _stream()), "cone_window_ranklist")
    torch.cuda.synchronize()
    tail = ws[nq * stride:].view(torch.int32)
    assert bool((tail == SENTINEL).all()), "cone_window_ranklist wrote past its window-score rows"
    return rl.cpu(), ws[: nq * stride].view(nq, stride).cpu()


def _frame_scores(ctx, video_offsets, q_first, cls, offsets, size, n_videos=None, margin=0):
    """cone_frame_scores into a sentinel-filled buffer of `size` + `margin` floats; returns the whole buffer (host)"""
    lib = _lib.load()
    vo, qf = video_offsets.cpu(), q_first.cpu()
    n_videos = len(vo) - 1 if n_videos is None else n_videos
    lens = (vo[1:] - vo[:-1]).tolist()
    nqs = (qf[1:] - qf[:-1]).tolist()
    out = torch.full((size + margin,), SENTINEL, dtype=torch.int32, device=DEV).view(torch.float32)
    # device copies held by name until the kernel has run (a temporary would go back to the allocator at once)
    vo_d, qf_d, off_d = video_offsets.to(DEV), q_first.to(DEV), offsets.to(DEV)
    _lib.check(lib.cone_frame_scores(_ptr(ctx), ctx.shape[1], _ptr(vo_d), _ptr(qf_d), n_videos, max(lens, default=0),
                                     max(nqs, default=0), _ptr(cls), _ptr(out), _ptr(off_d), _lib.PREC_FP32, _stream()),
               "cone_frame_scores")
    torch.cuda.synchronize()
    return out.cpu()


def _packed(lens_q):
    """packed offsets of queries with frame counts lens_q"""
    lens = torch.tensor(lens_q, dtype=torch.int64)
    return torch.cumsum(lens, 0) - lens, int(lens.sum())


def _bits(t):
    return t.contiguous().view(torch.int32)


# ---------------------------------------------------------------------------------------------- a. rank-lists
def _ranklist_case(max_v_l, nw_list, kind, seed, stride=None):
    """one launch over queries with nw_list windows; ragged offsets with gaps filled with NaN"""
    g = torch.Generator().manual_seed(seed)
    Ls = [frames_for_windows(n, max_v_l) for n in nw_list]
    fs = [synth_scores(kind, L, max_v_l, g) for L in Ls]
    gap = 3
    offs, pos, parts = [], 0, []
    for x in fs:
        parts.append(torch.full((gap,), math.nan))
        pos += gap
        offs.append(pos)
        parts.append(x)
        pos += x.numel()
    parts.append(torch.full((gap,), math.nan))
    buf = torch.cat(parts).float().to(DEV)
    stride = stride or max(nw_list)
    rl, ws = _lib_ranklist(buf, torch.tensor(offs, dtype=torch.int64, device=DEV),
                           torch.tensor(Ls, dtype=torch.int32, device=DEV), max_v_l, stride, winscore_margin=64)
    for j, (x, nw) in enumerate(zip(fs, nw_list)):
        want_ws = ref_window_scores(x, max_v_l)
        assert want_ws.numel() == nw
        want = ref_ranklist(want_ws).to(torch.int32)
        what = f"max_v_l {max_v_l} {kind} nw {nw} stride {stride}"
        assert torch.equal(rl[j, :nw], want), what
        assert bool((rl[j, nw:] == -1).all()), what
        got_ws = ws[j, :nw]
        nan = torch.isnan(want_ws)
        assert torch.equal(torch.isnan(got_ws), nan), what
        assert bool((got_ws[~nan] == want_ws[~nan]).all()), what  # == : the sign of a zero maximum is not compared
    return stride


@pytest.mark.parametrize("max_v_l", [2, 3, 90, 125])
def test_ranklist_every_sort_size_and_value_class(max_v_l):
    sizes = set()
    for c, kind in enumerate(VALUE_CLASSES):
        for t, nw in enumerate(NW_SIZES):
            # the largest rank-list of the launch sets the sort size; shorter rows of other lengths share it
            smaller = [n for n in NW_SIZES if n < nw]
            others = [1] + smaller[-1:] + smaller[len(smaller) // 2: len(smaller) // 2 + 1] if smaller else []
            stride = _ranklist_case(max_v_l, [nw] + others + [nw], kind, 1000 * c + t)
            npad = max(32, 1 << (stride - 1).bit_length())
            sizes.add(npad)
    assert sizes == {32, 64, 256, 512, 4096, 8192, 16384}
    print(f"[prefilter] ranklist max_v_l {max_v_l}: {len(VALUE_CLASSES) * len(NW_SIZES)} launches, sort sizes "
          f"{sorted(sizes)}, bit-identical to torch.sort(stable)")


def test_ranklist_strides_longer_than_every_query():
    for kind in ("random", "nan", "ties"):
        _ranklist_case(90, [300, 2, 41], kind, 7, stride=300 + 37)
        _ranklist_case(90, [1, 2, 111, 256], kind, 8, stride=MAX_WINDOWS)  # short videos in the largest sort


def test_ranklist_refuses_stride_past_16384():
    buf = torch.zeros(10, device=DEV)
    offs = torch.zeros(1, dtype=torch.int64, device=DEV)
    cnt = torch.full((1,), 10, dtype=torch.int32, device=DEV)
    with pytest.raises(ConeError, match="16384"):
        _lib_ranklist(buf, offs, cnt, 90, MAX_WINDOWS + 1)
    eng = _engine()
    with pytest.raises(ConeError, match="16384"):
        eng.window_ranklist(buf, offs, cnt, ranklist_stride=MAX_WINDOWS + 1)


def test_ranklist_short_stride_never_returns_a_wrong_prefix():
    """A stride shorter than a query's window count: the sort holds npad = pow2 >= stride keys.  A query with more than
    npad windows gets a row of -1 (winscore NaN); one with stride < nw <= npad still gets the true best `stride`."""
    g = torch.Generator().manual_seed(3)
    max_v_l = 4  # stride 2
    nws = [100, 40, 10]
    Ls = [frames_for_windows(n, max_v_l) for n in nws]
    fs = [torch.randn(L, generator=g) for L in Ls]
    # the best window of the long query lies past the first 64: a prefix sort would miss it
    fs[0][-3:] = 10.0
    offs, size = _packed(Ls)
    buf = torch.cat(fs).to(DEV)
    cnt = torch.tensor(Ls, dtype=torch.int32, device=DEV)
    for stride in (33, 16):
        npad = max(32, 1 << (stride - 1).bit_length())
        rl, ws = _lib_ranklist(buf, offs.to(DEV), cnt, max_v_l, stride, winscore_margin=npad)
        for j, (x, nw) in enumerate(zip(fs, nws)):
            want = ref_ranklist(ref_window_scores(x, max_v_l)).to(torch.int32)
            if nw > npad:
                assert bool((rl[j] == -1).all()), (stride, nw, rl[j, :8].tolist(), want[:8].tolist())
                assert bool(torch.isnan(ws[j]).all()), (stride, nw)
            else:
                n = min(nw, stride)
                assert torch.equal(rl[j, :n], want[:n]), (stride, nw)
                assert bool((rl[j, n:] == -1).all())
    # the engine refuses a short explicit stride where it knows the frame counts on the host, before any launch
    eng = _engine(EGO4D.replace(max_v_l=max_v_l))
    with pytest.raises(ValueError, match="ranklist_stride"):
        eng.window_ranklist(buf, offs.to(DEV), cnt.cpu(), ranklist_stride=33)
    with pytest.raises(ValueError, match="ranklist_stride"):
        eng.window_ranklist(buf, offs.to(DEV), cnt, ranklist_stride=33, max_frame_count=max(Ls))
    rl = eng.window_ranklist(buf, offs.to(DEV), cnt.cpu(), ranklist_stride=100)  # a host frame_count is copied over
    assert torch.equal(rl[0].cpu(), ref_ranklist(ref_window_scores(fs[0], max_v_l)).to(torch.int32))


# ---------------------------------------------------------------------------------------------- b. frame scores
def _grouped_inputs(v_dim, nq_per_video, lens, seed):
    g = torch.Generator().manual_seed(seed)
    ctx = torch.randn(sum(lens), v_dim, generator=g)
    ctx = ctx / ctx.norm(dim=1, keepdim=True)
    cls = torch.randn(sum(nq_per_video), v_dim, generator=g)
    cls = cls / cls.norm(dim=1, keepdim=True)
    vo = torch.zeros(len(lens) + 1, dtype=torch.int64)
    vo[1:] = torch.cumsum(torch.tensor(lens, dtype=torch.int64), 0)
    qf = torch.zeros(len(lens) + 1, dtype=torch.int32)
    qf[1:] = torch.cumsum(torch.tensor(nq_per_video, dtype=torch.int32), 0)
    q_len = [L for L, n in zip(lens, nq_per_video) for _ in range(n)]
    return ctx, cls, vo, qf, q_len


def _check_fp64(ctx, cls, vo, qf, scores, offs, what):
    """|got - ref| <= K 2^-24 sum|a_k b_k| per element; returns (max err, rms err, max err / bound)"""
    K = ctx.shape[1]
    errs, ratios = [], []
    for v in range(len(vo) - 1):
        q0, q1, f0, f1 = int(qf[v]), int(qf[v + 1]), int(vo[v]), int(vo[v + 1])
        if q1 == q0 or f1 == f0:
            continue
        ref, scale = fp64_scores(ctx[f0:f1], cls[q0:q1])
        got = torch.stack([scores[int(offs[q]): int(offs[q]) + f1 - f0] for q in range(q0, q1)]).double()
        err = (got - ref).abs()
        bound = K * 2.0 ** -24 * scale * 1.0001 + 1e-300
        ratios.append(float((err / bound).max()))
        assert bool((err <= bound).all()), f"{what}: video {v}: {float((err / bound).max()):.3g}x the fp32 FMA-chain bound"
        errs.append(err.flatten())
    e = torch.cat(errs)
    return float(e.max()), float(e.pow(2).mean().sqrt()), max(ratios)


QPV = (1, 127, 128, 129, 300)
FRAMES = (1, 3, 127, 128, 129, 1000, 4099)


@pytest.mark.parametrize("v_dim", [16, 48, 256, 768, 772])
def test_frame_scores_grouped_vs_fp64_and_bitwise(v_dim):
    # every queries-per-video and frames-per-video value, paired so that each M and N tile edge meets several others
    nq_per_video = [QPV[i % len(QPV)] for i in range(len(FRAMES))] + [300, 0, 129]
    lens = list(FRAMES) + [4099, 50, 128]
    ctx, cls, vo, qf, q_len = _grouped_inputs(v_dim, nq_per_video, lens, v_dim)
    offs, size = _packed(q_len)
    ctx_d, cls_d = ctx.to(DEV), cls.to(DEV)
    out = _frame_scores(ctx_d, vo, qf, cls_d, offs, size, margin=16)
    assert bool((_bits(out[size:]) == SENTINEL).all())
    mx, rms, ratio = _check_fp64(ctx, cls, vo, qf, out, offs, f"v_dim {v_dim}")
    print(f"[prefilter] frame_scores v_dim {v_dim}: {len(lens)} videos, {size} scores vs fp64: max {mx:.2e} rms "
          f"{rms:.2e}, at most {ratio:.3f} of the bound K 2^-24 sum|ab|")
    eng = _engine()
    for v in range(len(lens)):
        q0, q1, f0, f1 = int(qf[v]), int(qf[v + 1]), int(vo[v]), int(vo[v + 1])
        if q1 == q0:
            continue
        want = torch.stack([out[int(offs[q]): int(offs[q]) + f1 - f0] for q in range(q0, q1)])
        # alone
        c1, cl1 = ctx_d[f0:f1].contiguous(), cls_d[q0:q1].contiguous()
        o1, s1 = _packed([f1 - f0] * (q1 - q0))
        alone = _frame_scores(c1, torch.tensor([0, f1 - f0]), torch.tensor([0, q1 - q0], dtype=torch.int32), cl1, o1, s1)
        assert torch.equal(_bits(alone.view(q1 - q0, f1 - f0)), _bits(want)), f"v_dim {v_dim} video {v} alone"
        # queries permuted within the video
        perm = torch.randperm(q1 - q0, generator=torch.Generator().manual_seed(v))
        pm = _frame_scores(c1, torch.tensor([0, f1 - f0]), torch.tensor([0, q1 - q0], dtype=torch.int32),
                           cl1[perm.to(DEV)].contiguous(), o1, s1).view(q1 - q0, f1 - f0)
        assert torch.equal(_bits(pm), _bits(want[perm])), f"v_dim {v_dim} video {v} permuted"
        # cone_linear in fp32 mode runs the same tile
        lin = eng.linear(cl1, c1, precision="fp32")
        torch.cuda.synchronize()
        assert torch.equal(_bits(lin.cpu()), _bits(want)), f"v_dim {v_dim} video {v} vs cone_linear"


def test_frame_scores_three_hundred_videos_and_the_engine():
    rng = np.random.default_rng(11)
    n = 300
    lens = [int(x) for x in rng.integers(1, 400, n)]
    nqs = [int(x) for x in rng.integers(0, 4, n)]
    nqs[-1] = 0  # the last video has no query
    nqs[0] = 0
    lens[5] = 4099
    nqs[5] = 130
    ctx, cls, vo, qf, q_len = _grouped_inputs(256, nqs, lens, 5)
    offs, size = _packed(q_len)
    out = _frame_scores(ctx.to(DEV), vo, qf, cls.to(DEV), offs, size)
    mx, rms, ratio = _check_fp64(ctx, cls, vo, qf, out, offs, "300 videos")
    print(f"[prefilter] frame_scores 300 videos ({sum(x == 0 for x in nqs)} without queries): max {mx:.2e} rms "
          f"{rms:.2e}, at most {ratio:.3f} of the bound")
    # ConeEngine.frame_scores packs the same offsets and gives the same bits
    from cone_b200.engine import QueryBatch
    qb = QueryBatch(video_offsets=vo.to(DEV), q_first=qf.to(DEV), q_video_start=None,
                    q_video_len=torch.tensor(q_len, dtype=torch.int32, device=DEV), tokens=None, tok_len=None, cls=None,
                    q_batch=None, n_batches=1, max_video_frames=max(lens), max_video_queries=max(nqs),
                    total_scores=size, order=None, query_ids=None)
    got, got_offs = _engine().frame_scores(ctx.to(DEV), qb, cls.to(DEV))
    torch.cuda.synchronize()
    assert torch.equal(got_offs.cpu(), offs)
    assert torch.equal(_bits(got.cpu()), _bits(out))


def _layout(kind, lens_q, q_first):
    """score offsets of one caller layout: 'padded' (each row 4-aligned, gaps between rows), 'reversed' (each video's
    rows in reverse query order), 'odd' (gaps of one float: unaligned rows)"""
    nq = len(lens_q)
    offs = [0] * nq
    pos = 0
    if kind == "reversed":
        for v in range(len(q_first) - 1):
            for q in reversed(range(int(q_first[v]), int(q_first[v + 1]))):
                offs[q] = pos
                pos += lens_q[q]
    else:
        for q in range(nq):
            pos += 5 if kind == "padded" else 1
            if kind == "padded":
                pos = (pos + 3) // 4 * 4
            offs[q] = pos
            pos += lens_q[q]
    return torch.tensor(offs, dtype=torch.int64), pos + 3


@pytest.mark.parametrize("layout", ["padded", "reversed", "odd"])
def test_frame_scores_honour_custom_score_offsets(layout):
    nqs = [3, 129, 0, 2, 5]
    lens = [131, 300, 40, 4, 257]
    ctx, cls, vo, qf, q_len = _grouped_inputs(256, nqs, lens, 21)
    ctx_d, cls_d = ctx.to(DEV), cls.to(DEV)
    p_offs, p_size = _packed(q_len)
    packed = _frame_scores(ctx_d, vo, qf, cls_d, p_offs, p_size)
    offs, size = _layout(layout, q_len, qf)
    # the margin keeps a wrong write inside the buffer, where the sentinel check sees it
    got = _frame_scores(ctx_d, vo, qf, cls_d, offs, size, margin=size)
    mine = torch.zeros(got.numel(), dtype=torch.bool)
    for q, L in enumerate(q_len):
        a, b = int(offs[q]), int(p_offs[q])
        assert torch.equal(_bits(got[a:a + L]), _bits(packed[b:b + L])), f"{layout}: query {q} not at score_offsets[q]"
        mine[a:a + L] = True
    assert bool((_bits(got[~mine]) == SENTINEL).all()), f"{layout}: {int((_bits(got[~mine]) != SENTINEL).sum())} " \
                                                        "scores written outside the documented rows"
    cnt = torch.tensor(q_len, dtype=torch.int32, device=DEV)
    stride = num_window(max(q_len), 90)
    rl_p, ws_p = _lib_ranklist(packed.to(DEV), p_offs.to(DEV), cnt, 90, stride)
    rl_c, ws_c = _lib_ranklist(got.to(DEV), offs.to(DEV), cnt, 90, stride)
    assert torch.equal(rl_c, rl_p) and torch.equal(_bits(ws_c), _bits(ws_p)), layout


# ---------------------------------------------------------------------------------------------- c. stage-0 context
def _ctx_fp64(sd, frames):
    x = frames.double().numpy()
    xn = torch.from_numpy(O.l2_normalize_np(x))
    with torch.no_grad():
        return O.stage0_video_context(R.cast_state_dict(sd), xn)


def test_context_features_vs_fp64_modes_and_slabs():
    cfg = EGO4D
    sd = _sd(cfg)
    g = torch.Generator().manual_seed(4)
    frames = torch.randn(4097, cfg.v_feat_dim, generator=g) * 3
    frames[[0, 17, 4096]] = 0  # all-zero rows: normalised to 0, the adapter biases alone
    ref = _ctx_fp64(sd, frames)
    f_d = frames.to(DEV)
    ctx32, _ = _engine(cfg, "fp32").video_prepare(f_d, want_vidproj=False)
    ctxtc, _ = _engine(cfg, "tc").video_prepare(f_d, want_vidproj=False)
    torch.cuda.synchronize()
    ctx32, ctxtc = ctx32.cpu(), ctxtc.cpu()
    err = (ctx32.double() - ref).abs()
    print(f"[prefilter] stage-0 ctx vs fp64 (4097 frames, 3 zero rows): max {float(err.max()):.2e} "
          f"rms {float(err.pow(2).mean().sqrt()):.2e}")
    assert float(err.max()) <= FP32_TOL
    assert torch.equal(_bits(ctxtc), _bits(ctx32)), "ctx differs between fp32 and tensor-core handles"
    dims = _lib.ConeDims(cfg.v_feat_dim, cfg.t_feat_dim, cfg.hidden_dim, cfg.nheads, cfg.dim_feedforward,
                         cfg.enc_layers, cfg.dec_layers, cfg.num_queries, cfg.max_v_l, cfg.max_q_l, cfg.v_motion_feat_dim)
    small = _lib.load().cone_prepare_workspace_bytes(C.byref(dims), 1000)
    for prec in ("fp32", "tc"):
        eng = _engine(cfg, prec, ws=small)
        for L in (4095, 4096, 4097):
            got, _ = eng.video_prepare(f_d[:L].contiguous(), want_vidproj=False)
            torch.cuda.synchronize()
            assert torch.equal(_bits(got.cpu()), _bits(ctx32[:L])), (prec, L)
        _cache.pop((cfg, prec, small, 0))


# ---------------------------------------------------------------------------------------------- d. l2 normalise
L2_DIMS = (4, 8, 12, 16, 20, 48, 124, 128, 132, 764, 768, 772, 4096, 4100)


def _l2_ref(x, eps):
    x = x.double()
    n = x.norm(dim=-1, keepdim=True)
    return x / (n.clamp_min(-eps) if eps < 0 else n + eps)


@pytest.mark.parametrize("eps", [1e-5, 0.0, -1e-5])
def test_l2_normalize_vs_fp64(eps):
    eng = _engine()
    lib = _lib.load()
    worst = 0.0
    for D in L2_DIMS:
        for rows in (1, 7, 8, 9, 100_000):
            if rows == 100_000 and D not in (4, 132, 772):
                continue
            g = torch.Generator().manual_seed(D * 7 + rows)
            x = torch.randn(rows, D, generator=g) * 5
            if rows > 1:
                x[1] = 0  # eps 0: 0/0 = NaN as in torch; eps < 0 (F.normalize): 0
            ref = _l2_ref(x, eps)
            xd = x.to(DEV)
            got = eng.l2_normalize(xd, eps)
            inplace = xd.clone()
            _lib.check(lib.cone_l2_normalize(_ptr(inplace), _ptr(inplace), rows, D, eps, _stream()), "cone_l2_normalize")
            torch.cuda.synchronize()
            got = got.cpu()
            nan = torch.isnan(ref)
            assert torch.equal(torch.isnan(got), nan), (D, rows, eps)
            err = float((got.double() - ref)[~nan].abs().max())
            worst = max(worst, err)
            assert err <= 2e-6, (D, rows, eps, err)
            assert torch.equal(_bits(inplace.cpu()), _bits(got)), (D, rows, "in place")
            if rows <= 9 or D == 132:
                for dt in (torch.float16, torch.bfloat16):
                    xh = xd.to(dt)
                    a, b = eng.l2_normalize(xh, eps), eng.l2_normalize(xh.float(), eps)
                    torch.cuda.synchronize()
                    assert torch.equal(_bits(a.cpu()), _bits(b.cpu())), (D, rows, dt)
    print(f"[prefilter] l2_normalize eps {eps:g}: {len(L2_DIMS)} dims vs fp64: max {worst:.2e}")
    for D in (2, 6, 130):
        with pytest.raises(ConeError):
            eng.l2_normalize(torch.ones(3, D, device=DEV), eps)


# ---------------------------------------------------------------------------------------------- e. cone_prefilter
@pytest.mark.parametrize("nw", [4097, 8193, 16384])
def test_prefilter_at_sort_boundaries(nw):
    cfg = axis_cfg("window3")
    assert cfg.max_v_l == 2
    sd = _sd(cfg, 2)
    eng = _engine(cfg, "fp32", seed=2)
    L = frames_for_windows(nw, cfg.max_v_l)
    g = torch.Generator().manual_seed(nw)
    frames = torch.randn(L, cfg.v_feat_dim, generator=g)
    cls = torch.randn(3, cfg.v_feat_dim, generator=g)
    # staged entry points
    f_d, c_d = frames.to(DEV), cls.to(DEV)
    ctx, _ = eng.video_prepare(f_d, want_vidproj=False)
    cls_n = eng.l2_normalize(c_d, 1e-5)
    offs, size = _packed([L] * 3)
    scores = _frame_scores(ctx, torch.tensor([0, L]), torch.tensor([0, 3], dtype=torch.int32), cls_n, offs, size)
    rl, ws = _lib_ranklist(scores.to(DEV), offs.to(DEV), torch.full((3,), L, dtype=torch.int32, device=DEV),
                           cfg.max_v_l, nw)
    # the oracle's stage 0/1 (fp32): rank-lists equal up to near-ties (inversion audit, limit 0), window scores within
    # FP32_TOL
    with torch.no_grad():
        octx = O.stage0_video_context(sd, torch.from_numpy(O.l2_normalize_np(frames.numpy())))
    hatch = Hatch(f"prefilter nw {nw}", "rank-list inverts windows beyond a near-tie of the oracle", 0)
    werr, swapped = 0.0, 0
    for q in range(3):
        orl, ofs = O.stage1_ranklist(octx, torch.from_numpy(O.l2_normalize_np(cls[q].numpy())), cfg.max_v_l)
        ows = O.window_scores(ofs, cfg.max_v_l)
        werr = max(werr, float((ws[q].double() - ows.double()).abs().max()))
        swapped += audit_vs_oracle(ows.numpy(), rl[q].tolist(), orl, hatch, f"query {q}")
    hatch.close(3)
    assert werr <= FP32_TOL
    for topk in (1, nw - 1, nw, nw + 5, MAX_WINDOWS):
        idx, sc = eng.prefilter(f_d, c_d, topk=topk, want_scores=True)
        torch.cuda.synchronize()
        idx, sc = idx.cpu(), sc.cpu()
        n = min(topk, nw)
        assert torch.equal(idx[:, :n], rl[:, :n]), topk
        assert bool((idx[:, n:] == -1).all()) and bool(torch.isnan(sc[:, n:]).all()), topk
        assert torch.equal(_bits(sc[:, :n]), _bits(torch.gather(ws, 1, rl[:, :n].long()))), topk
    print(f"[prefilter] cone_prefilter nw {nw}: window scores vs oracle max {werr:.2e}, {swapped} of {3 * nw} rank-list "
          f"positions differ by near-ties; bitwise = staged entry points")
    if nw == MAX_WINDOWS:
        with pytest.raises(ConeError, match="16384"):
            eng.prefilter(torch.randn(L + 1, cfg.v_feat_dim, device=DEV), c_d, topk=5)


# ---------------------------------------------------------------------------------------------- f. the engine
def test_engine_past_4096_windows_every_window():
    cfg = EGO4D.replace(max_v_l=6, eval_bsz=4)
    sd = _sd(cfg, 5)
    L = 24_600
    nw = cfg.num_window(L)
    assert nw == 8201
    ds = make_dataset(cfg, 1, [L], [2], seed=17)
    full = ground_dataset(ConeEngine(cfg.replace(topk_window=nw), sd, device=DEV, precision="fp32",
                                     workspace_bytes=4 << 30), ds.videos, ds.queries)
    top = ground_dataset(ConeEngine(cfg.replace(topk_window=30), sd, device=DEV, precision="fp32",
                                    workspace_bytes=1 << 30), ds.videos, ds.queries)
    hatch = Hatch("engine 8201 windows", "rank-list inverts windows beyond a near-tie of the oracle", 0)
    with torch.no_grad():
        octx = O.stage0_video_context(sd, torch.from_numpy(O.l2_normalize_np(ds.videos[0])))
    # the staged entry points give the engine's rank-lists
    eng = _engine(cfg, seed=5)
    ctx, _ = eng.video_prepare(torch.from_numpy(ds.videos[0]).to(DEV), want_vidproj=False)
    cls_n = eng.l2_normalize(torch.from_numpy(np.stack([q.cls for q in ds.queries])).to(DEV), 1e-5)
    offs, size = _packed([L] * len(ds.queries))
    scores = _frame_scores(ctx, torch.tensor([0, L]), torch.tensor([0, len(ds.queries)], dtype=torch.int32), cls_n,
                           offs, size)
    srl, _ = _lib_ranklist(scores.to(DEV), offs.to(DEV), torch.full((len(ds.queries),), L, dtype=torch.int32,
                                                                      device=DEV), cfg.max_v_l, nw)
    ora, swapped = {}, 0
    for j, q in enumerate(ds.queries):
        r = full[q.query_id]
        orl, ofs = O.stage1_ranklist(octx, torch.from_numpy(O.l2_normalize_np(q.cls)), cfg.max_v_l)
        ora[q.query_id] = orl
        assert len(r["ranklist"]) == nw and len(r["windows"]) == nw
        assert r["ranklist"] == srl[j].tolist(), q.query_id
        swapped += audit_vs_oracle(O.window_scores(ofs, cfg.max_v_l).numpy(), r["ranklist"], orl, hatch, q.query_id)
        t = top[q.query_id]
        assert r["windows"][:30] == t["windows"]
        for k in ("pred_spans", "prob_fg", "match"):
            assert np.array_equal(np.asarray(r[k])[:30], np.asarray(t[k]), equal_nan=True), (q.query_id, k)
    hatch.close(len(ds.queries))
    # window recall on long, -1-padded rank-lists: the device's lists, and the oracle's where they agree
    stride = nw + 99
    rl = torch.full((len(ds.queries), stride), -1, dtype=torch.int32)
    for j, q in enumerate(ds.queries):
        rl[j, :nw] = torch.tensor(full[q.query_id]["ranklist"], dtype=torch.int32)
    gt = {q.query_id: list(q.timestamps) for q in ds.queries}
    topk = (1, 5, 30, 4096, 8201, stride)
    hits = eng.eval_window_recall(rl.to(DEV), torch.tensor([gt[q.query_id] for q in ds.queries], dtype=torch.float64,
                                                           device=DEV), topk=topk)
    mine = {q.query_id: full[q.query_id]["ranklist"] for q in ds.queries}
    want = O.window_recall(mine, gt, cfg.clip_length, cfg.max_v_l, topk=topk) * len(ds.queries)
    assert np.array_equal(hits.cpu().numpy(), np.round(want).astype(np.int64)), (hits.tolist(), want)
    if swapped == 0:
        assert np.array_equal(want, O.window_recall(ora, gt, cfg.clip_length, cfg.max_v_l, topk=topk) * len(ds.queries))
    print(f"[prefilter] engine, {nw} windows per query: {swapped} of {len(ds.queries) * nw} rank-list positions differ "
          f"from the oracle by near-ties, first 30 = top-30 run, window recall {hits.tolist()} = oracle.window_recall")
