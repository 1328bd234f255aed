"""Proposal matching (A9) at the operator level against the fp64 reference with the fp32 reference's pooling bounds.

`fp64_reference.clip_matching_exact_bounds` pools exactly the rows the fp32 reference pools, so no comparison here has a
floor/ceil exemption: every proposal is within FP32_TOL (fp32 mode) or TC_TOL (tensor-core mode), NaN where the
reference gives NaN.

- `cone_clip_matching` over proposals per window 1-64 (the window kernels for up to 5 and up to 8 proposals, the
  per-proposal kernel above 8), v_dim 16-4096 (fewer than 32 float4 columns, more than 256 per thread, the tcgen05 and
  the fp32 adapter GEMMs) and padded lengths 1-480 with valid lengths Lv, 1, ceil(Lv/2), Lv-1, random and 0, on
  proposals at every pooling edge (tests/helpers.py `edge_spans`).  Tensor-core mode equals fp32 mode bitwise where
  both adapter GEMMs run on the fp32 pipe.
- The per-proposal kernel gives the window kernels' bits; rows past a window's valid length are never read.
- `cone_ground_windows_ex` on crafted rank-lists over videos of 1-1000 frames: window bounds exact, `match` against the
  reference recomputed from the library's own spans, with per-eval-batch and fixed padding.
- The drop-in `CONE.forward_clip_matching` on proposals with negative slice ends.

Prints one `[matching] ...` line per case with its largest errors."""
import numpy as np
import pytest
import torch

from cone_b200 import _lib
from cone_b200.config import EGO4D
from cone_b200.engine import ConeEngine, _ptr, _stream
from cone_b200.model import CONE
from cone_b200.weights import init_state_dict
from oracle import cone_oracle as O
import fp64_reference as R
from helpers import FP32_TOL, TC_TOL, edge_spans

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = {"fp32": FP32_TOL, "tc": TC_TOL}
# (v_dim, proposals per window): every v_dim meets all three pooling kernels, every proposal count is run
SWEEP = [(16, 1), (16, 6), (16, 9), (48, 2), (48, 8), (48, 16), (320, 5), (320, 6), (320, 33),
         (1040, 5), (1040, 8), (1040, 64), (4096, 2), (4096, 8), (4096, 9)]
SWEEP_LV = (1, 2, 91, 125, 480)
_cache = {}


def _engine(cfg, precision, seed=0):
    key = (cfg, precision, seed)
    if key not in _cache:
        _cache[key] = ConeEngine(cfg, _sd(cfg, seed), device=DEV, precision=precision, workspace_bytes=1 << 30)
    return _cache[key]


def _sd(cfg, seed):
    key = ("sd", cfg, seed)
    if key not in _cache:
        _cache[key] = init_state_dict(cfg, seed)
    return _cache[key]


def _bits(x):
    return torch.as_tensor(x).detach().cpu().contiguous().view(torch.int32)


def _errors(got, want, what):
    """NaN positions identical; the largest |got - want| / max(1, |want|) over the others"""
    got, want = torch.as_tensor(got).cpu().double(), torch.as_tensor(want).cpu().double()
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan), f"{what}: NaN at {torch.nonzero(torch.isnan(got) != nan)[:8].tolist()}"
    err = (got - want).abs() / want.abs().clamp(min=1.0)
    return float(err[~nan].max()) if (~nan).any() else 0.0


def _windows(lv, nq, Dv, seed):
    """Dense windows [B, Lv, Dv] zero padded past their valid lengths (Lv, 1, ceil(Lv/2), Lv-1, random, 0), each
    valid length repeated so that its windows hold every edge proposal of it, nq to a window."""
    rng = np.random.default_rng(seed)
    vlens, spans = [], []
    for n in (lv, 1, -(-lv // 2), lv - 1, int(rng.integers(1, lv + 1)), 0):
        n = max(n, 0)
        e = edge_spans(n, lv, seed + n)
        e = e[np.arange(-(-len(e) // nq) * nq) % len(e)].reshape(-1, nq, 2)
        vlens += [n] * len(e)
        spans.append(e)
    g = torch.Generator().manual_seed(seed)
    B = len(vlens)
    vl = torch.tensor(vlens, dtype=torch.int32)
    vm = (torch.arange(lv)[None] < vl[:, None]).float()
    vid = torch.randn(B, lv, Dv, generator=g) * vm[..., None]
    cls = torch.randn(B, Dv, generator=g)
    return cls, vid, vl, vm, torch.from_numpy(np.concatenate(spans))


def _match(eng, cls, vid, vl, spans):
    return eng.clip_matching(cls.to(DEV), vid.to(DEV), vl.to(DEV), spans.to(DEV)).cpu()


# ------------------------------------------------------------------------------------------- cone_clip_matching
@pytest.mark.parametrize("Dv,nq", SWEEP, ids=[f"dv{d}-nq{n}" for d, n in SWEEP])
def test_clip_matching_sweep(Dv, nq):
    cfg = EGO4D.replace(v_feat_dim=Dv)
    sd = _sd(cfg, Dv)
    worst = {}
    for lv in SWEEP_LV:
        cls, vid, vl, vm, spans = _windows(lv, nq, Dv, 1000 * lv + nq)
        want = R.clip_matching_exact_bounds(sd, cls, vid, vm, spans)
        got = {}
        for precision in ("fp32", "tc"):
            got[precision] = _match(_engine(cfg, precision, Dv), cls, vid, vl, spans)
            err = _errors(got[precision], want, f"Dv {Dv} nq {nq} Lv {lv} {precision}")
            worst[precision] = max(worst.get(precision, 0.0), err)
            print(f"[matching] sweep Dv {Dv} nq {nq} Lv {lv} {precision}: {spans.shape[0]} windows, "
                  f"{int(torch.isnan(want).sum())} NaN of {want.numel()}, max err {err:.3e}")
            assert err <= TOL[precision], f"Dv {Dv} nq {nq} Lv {lv} {precision}: max error {err:.3e} > {TOL[precision]}"
        if Dv in (16, 48, 1040):  # neither adapter GEMM has a tcgen05 shape: tensor-core mode runs the fp32 GEMM
            assert torch.equal(_bits(got["tc"]), _bits(got["fp32"])), (Dv, nq, lv)
    print(f"[matching] sweep Dv {Dv} nq {nq}: max err fp32 {worst['fp32']:.3e} tc {worst['tc']:.3e}")


def test_per_proposal_kernel_gives_the_window_kernels_bits():
    """nq 9 (one CTA per proposal) against nq 5 and 8 (one CTA per window) on the same windows and first proposals"""
    cfg = EGO4D
    eng = _engine(cfg, "fp32")
    for lv in (91, 125):
        cls, vid, vl, _, spans = _windows(lv, 9, cfg.v_feat_dim, 7 + lv)
        nine = _match(eng, cls, vid, vl, spans)
        for k in (5, 8):
            few = _match(eng, cls, vid, vl, spans[:, :k].contiguous())
            assert torch.equal(_bits(nine[:, :k]), _bits(few)), (lv, k)


def test_rows_past_the_valid_length_are_never_read():
    """the header's zero padding: rows >= vid_len filled with large values or NaN give the bits of zero rows"""
    cfg = EGO4D.replace(v_feat_dim=48)
    for precision in ("fp32", "tc"):
        eng = _engine(cfg, precision)
        for nq in (5, 8, 9):
            cls, vid, vl, vm, spans = _windows(91, nq, cfg.v_feat_dim, 3 + nq)
            base = _match(eng, cls, vid, vl, spans)
            for fill in (1e6, float("nan")):
                junk = torch.where(vm[..., None] > 0, vid, torch.full_like(vid, fill))
                assert torch.equal(_bits(_match(eng, cls, junk, vl, spans)), _bits(base)), (precision, nq, fill)


def test_every_pooling_kernel_is_launched():
    from torch.profiler import ProfilerActivity, profile
    cfg = EGO4D.replace(v_feat_dim=48)
    eng = _engine(cfg, "fp32")
    cases = [_windows(2, nq, cfg.v_feat_dim, nq) for nq in (5, 8, 9)]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(2):  # twice: the profiler can miss the first launch of a session
            for cls, vid, vl, _, spans in cases:
                _match(eng, cls, vid, vl, spans)
        torch.cuda.synchronize()
    names = {e.key.replace(" ", "") for e in prof.key_averages()}
    want = ["span_mean_pool_window_kernel<5,", "span_mean_pool_window_kernel<8,", "span_mean_pool_kernel<",
            "norm_dot_kernel("]
    print("[matching] pooling kernels launched:\n  " + "\n  ".join(sorted(n for n in names if "pool" in n or "dot" in n)))
    missing = [k for k in want if not any(k in n for n in names)]
    assert not missing, f"not launched: {missing}"


def test_dropin_forward_clip_matching_negative_ends():
    cfg = EGO4D
    sd = _sd(cfg, 9)
    model = CONE(cfg, sd).to(DEV).eval()
    g = torch.Generator().manual_seed(4)
    vl = torch.tensor([90, 45, 61])
    vm = (torch.arange(90)[None] < vl[:, None]).float()
    vid = torch.randn(3, 90, cfg.v_feat_dim, generator=g) * vm[..., None]
    cls = torch.randn(3, cfg.v_feat_dim, generator=g)
    # negative slice ends: -27 of 90 rows (rows [0, 63)), -4, -88 (rows [0, 2)), -13, and a negative width (start > 0)
    spans = torch.tensor([[(-0.5, 0.4), (-0.05, 0.0), (-88.5 / 90, 0.0), (-0.2, 0.1), (0.3, -0.8)]] * 3)
    with torch.no_grad():
        want = O.clip_matching(sd, cls, vid, vm, spans)
    start, end = O.proposal_bounds(spans, vm)
    assert (end < 0).all() and torch.isfinite(want).all()
    got = model.forward_clip_matching(cls.to(DEV), vid.to(DEV), vm.to(DEV), proposal=spans.to(DEV)).cpu()
    assert torch.isfinite(got).all()
    err = _errors(got, want, "drop-in negative ends")
    print(f"[matching] drop-in negative ends: max err {err:.3e}")
    assert err <= FP32_TOL


# --------------------------------------------------------------------------------------- cone_ground_windows_ex
VIDEO_LENS = (1, 44, 45, 46, 91, 137, 1000)
QUERIES_PER_VIDEO = 3
GROUND_CFGS = {"ego4d_90x5": EGO4D, "odd_91x8": EGO4D.replace(max_v_l=91, num_queries=8)}


def _ranklist(cfg, L, rng):
    """window 0, the last and the second-to-last window first, then the others in random order"""
    nw = cfg.num_window(L)
    head = list(dict.fromkeys([0, nw - 1, max(nw - 2, 0)]))
    rest = [w for w in rng.permutation(nw).tolist() if w not in head]
    return head + rest


def _ground_sd(cfg):
    """perturbed weights with wide proposals, so that spans start before 0 and end past the window"""
    sd = init_state_dict(cfg, 21)
    sd["span_embed.layers.2.bias"] = torch.tensor([-0.6, 1.0])
    return sd


def _ground(eng, cfg, frames, inputs, q_batch, n_batches, topk):
    q_start, q_len, rl, tok, tok_len, cls_norm = inputs
    nq_, ns = q_len.numel(), cfg.num_queries
    _, vidproj = eng.video_prepare(frames, want_ctx=False)
    spans = torch.empty((nq_, topk, ns, 2), dtype=torch.float32, device=DEV)
    prob = torch.empty((nq_, topk, ns), dtype=torch.float32, device=DEV)
    match = torch.empty((nq_, topk, ns), dtype=torch.float32, device=DEV)
    wstart = torch.empty((nq_, topk), dtype=torch.int32, device=DEV)
    wlen = torch.empty((nq_, topk), dtype=torch.int32, device=DEV)
    ws, nb = eng._wsargs()
    _lib.check(eng.lib.cone_ground_windows_ex(
        eng._handle, _ptr(frames), _lib.DTYPE_F32, frames.shape[0], _ptr(vidproj), _ptr(q_start), _ptr(q_len), _ptr(rl),
        rl.shape[1], _ptr(tok), _ptr(tok_len), _ptr(cls_norm), _ptr(q_batch), n_batches, nq_, topk, _ptr(spans),
        _ptr(prob), _ptr(match), _ptr(wstart), _ptr(wlen), ws, nb, eng.precision, _stream()), "cone_ground_windows_ex")
    return spans.cpu(), match.cpu(), wstart.cpu(), wlen.cpu()


@pytest.mark.parametrize("name", list(GROUND_CFGS))
def test_ground_windows_matching_on_crafted_ranklists(name):
    cfg = GROUND_CFGS[name]
    sd = _ground_sd(cfg)
    rng = np.random.default_rng(3)
    g = torch.Generator().manual_seed(5)
    offs = np.concatenate([[0], np.cumsum(VIDEO_LENS)])
    n_frames = int(offs[-1])  # the last video ends at the end of the frame tensor
    frames = torch.randn(n_frames, cfg.v_feat_dim, generator=g)
    vids = [v for v in range(len(VIDEO_LENS)) for _ in range(QUERIES_PER_VIDEO)]
    nq_ = len(vids)
    stride = max(cfg.num_window(L) for L in VIDEO_LENS)
    rl = torch.full((nq_, stride), -1, dtype=torch.int32)
    for q, v in enumerate(vids):
        r = _ranklist(cfg, VIDEO_LENS[v], rng)
        rl[q, : len(r)] = torch.tensor(r, dtype=torch.int32)
    topk = 5  # more than the 2 windows of the 1- and 44-frame videos: their last 3 are absent
    tok_len = torch.from_numpy(rng.integers(1, cfg.max_q_l + 1, nq_).astype(np.int32))
    tok = torch.randn(nq_, cfg.max_q_l, cfg.t_feat_dim, generator=g) * (torch.arange(cfg.max_q_l)[None] < tok_len[:, None])[..., None]
    tok = tok / (tok.norm(dim=-1, keepdim=True) + 1e-5)
    cls = torch.randn(nq_, cfg.v_feat_dim, generator=g)
    cls_norm = cls / (cls.norm(dim=-1, keepdim=True) + 1e-5)
    q_start = torch.tensor([int(offs[v]) for v in vids], dtype=torch.int64)
    q_len = torch.tensor([VIDEO_LENS[v] for v in vids], dtype=torch.int32)
    inputs = [t.to(DEV) for t in (q_start, q_len, rl, tok, tok_len, cls_norm)]
    # eval batch 0: the 1- and 44-frame videos only (pad_len 44); batch 1: short last windows with full ones
    q_batch = torch.tensor([0 if VIDEO_LENS[v] <= 44 else 1 for v in vids], dtype=torch.int32)
    counts = dict(x1_neg=0, end_in_pad=0, end_past_pad=0, windows_padded=0)
    for precision in ("fp32", "tc"):
        eng = ConeEngine(cfg, sd, device=DEV, precision=precision, workspace_bytes=1 << 30)
        for batched in (True, False):
            spans, match, wstart, wlen = _ground(eng, cfg, frames.to(DEV), inputs, q_batch.to(DEV) if batched else None,
                                                 2 if batched else 1, topk)
            pad_of = {}
            for q, v in enumerate(vids):
                for j in range(topk):
                    L = VIDEO_LENS[v]
                    want = (0, 0)  # absent: the video has fewer than topk windows
                    if j < cfg.num_window(L):
                        s, e = cfg.window_bounds(int(rl[q, j]), L)
                        want = (s, e - s)
                    assert (int(wstart[q, j]), int(wlen[q, j])) == want, (q, j)
                    b = int(q_batch[q])
                    pad_of[b] = max(pad_of.get(b, 0), want[1])
            if batched:
                assert pad_of[0] == 44 and pad_of[1] == cfg.max_v_l, pad_of
            worst = 0.0
            for q, v in enumerate(vids):
                for j in range(topk):
                    n = int(wlen[q, j])
                    if n == 0:
                        continue
                    pad = pad_of[int(q_batch[q])] if batched else cfg.max_v_l
                    s0 = int(offs[v]) + int(wstart[q, j])
                    win = torch.zeros(1, pad, cfg.v_feat_dim)
                    win[0, :n] = frames[s0: s0 + n]  # the window's own rows: what lies past them is not its video's
                    vm = torch.zeros(1, pad)
                    vm[0, :n] = 1
                    sp = spans[q, j][None]
                    want = R.clip_matching_exact_bounds(sd, cls_norm[q][None], win, vm, sp)
                    worst = max(worst, _errors(match[q, j][None], want, f"{name} {precision} q {q} window {j}"))
                    if precision == "fp32" and batched:
                        x1, x2 = O.span_cxw_to_xx(sp[0]).unbind(-1)
                        _, end = O.proposal_bounds(sp, vm)
                        counts["x1_neg"] += int((x1 < 0).sum())
                        counts["end_in_pad"] += int(((end[0] > n) & (end[0] <= pad)).sum()) if pad > n else 0
                        counts["end_past_pad"] += int((end[0] > pad).sum())
                        counts["windows_padded"] += int(pad > n)
            print(f"[matching] ground {name} {precision} {'q_batch' if batched else 'fixed pad'}: max err {worst:.3e}")
            assert worst <= TOL[precision], f"{name} {precision}: max error {worst:.3e} > {TOL[precision]}"
    print(f"[matching] ground {name} edge counts: {counts}")
    assert min(counts.values()) >= 30, counts
