"""Shared test helpers: golden loading and tolerant comparison of prediction lists."""
import json
import os

import numpy as np

from cone_b200.inference import MODES, recall_at_k
from cone_b200.synth import make_dataset
from cone_b200.weights import init_state_dict
from oracle.make_golden import E2E_CASES, GOLDEN, dense_case  # noqa: F401  (no reference import at module load)

# How north_star's tolerances are read, stated once: "scores and spans must agree within 1e-3 relative in bf16 or
# 1e-5 in fp32".  The compared quantities are the model's raw outputs — normalised spans (cx, w) in (0, 1), class
# probabilities in (0, 1), cosine matching scores in [-1, 1] — so "relative" is taken relative to their O(1) scale:
#     |a - b| <= tol * max(1, |b|)
# i.e. ABSOLUTE for |b| <= 1 (never looser than tol) and relative above 1 (spans in seconds after scaling).  A purely
# relative reading |a-b| <= tol*|b| is not meetable by ANY finite-precision implementation for values near 0 (a width
# of 1e-4 would need 1e-9 absolute) and is not what the reference's own 4-decimal rounding (inference.py:83) resolves.
FP32_TOL = 1e-5
TC_TOL = 1e-3  # reduced-precision (tensor-core, fp16 operands) mode: max over ALL compared values, no percentile form
# After the reference's 4-decimal rounding (inference.py:83) a 1e-7 difference can move a value by one
# unit in the 4th decimal; seconds are scaled by duration*clip_length (<= ~1e4 for MAD movies).
ROUND_TOL = 1.01e-4


def load_e2e(name):
    cfg, dkw, wseed, perturb = E2E_CASES[name]
    sd = init_state_dict(cfg, wseed, perturb=perturb)
    ds = make_dataset(cfg, **dkw)
    arrays = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    with open(os.path.join(GOLDEN, name + ".json")) as f:
        lists = json.load(f)
    return cfg, sd, ds, arrays, lists


def close(a, b, tol):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.shape != b.shape:
        return False
    return bool(np.all(np.abs(a - b) <= tol * np.maximum(1.0, np.abs(b))))


def assert_close(a, b, tol, what=""):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    err = np.abs(a - b) / np.maximum(1.0, np.abs(b))
    assert np.all(err <= tol), f"{what}: max err {err.max():.3e} > {tol:.1e}"


def rows_close(a, b, span_tol, score_tol=ROUND_TOL):
    """Two lists of [st, ed, score, ...] rows: same length, same order, values within tolerance."""
    if len(a) != len(b):
        return False
    for x, y in zip(a, b):
        if len(x) != len(y):
            return False
        if abs(x[0] - y[0]) > span_tol or abs(x[1] - y[1]) > span_tol:
            return False
        for u, v in zip(x[2:], y[2:]):
            if abs(u - v) > score_tol * max(1.0, abs(v)) * (2.5 if len(x) == 5 else 1.0):
                return False
    return True


def boundary_exempt(ref_spans, durations, eps=1e-4):
    """SURVEY.md §7 H3: `start = floor(x1*dur)`, `end = ceil(x2*dur)` (model.py:187-192) turn a 1-ulp span
    difference into a +-1-frame pooling difference.  Returns a bool mask (k, nq) of proposals whose
    x1*dur or x2*dur lies within `eps` of an integer in the REFERENCE — only those may differ in the
    end-to-end matching score; everything else must meet the tolerance."""
    sp = np.asarray(ref_spans, dtype=np.float64)
    dur = np.asarray(durations, dtype=np.float64)[:, None]
    x1 = (sp[..., 0] - 0.5 * sp[..., 1]) * dur
    x2 = (sp[..., 0] + 0.5 * sp[..., 1]) * dur
    near = lambda x: np.abs(x - np.round(x)) < eps
    return near(x1) | near(x2)


def assert_match_close(got, ref, ref_spans, durations, tol, what="match"):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    assert got.shape == ref.shape
    ex = boundary_exempt(ref_spans, durations)
    err = np.abs(got - ref) / np.maximum(1.0, np.abs(ref))
    bad = (err > tol) & ~ex
    assert not bad.any(), f"{what}: max err {err[~ex].max():.3e} > {tol:.1e} away from floor/ceil boundaries"
    assert ex.mean() <= 0.05, f"{what}: {ex.mean():.1%} of proposals sit on a floor/ceil boundary"
    return int(((err > tol) & ex).sum())


class Hatch:
    """A COUNTED exception to an otherwise exact comparison.  Every use is recorded with its reason, the total is printed
    (and appended to gpurun_out/hatches.log when that directory exists) and bounded by `limit` — so a regression cannot
    hide behind a silent `continue`."""

    def __init__(self, test: str, what: str, limit: int):
        self.test, self.what, self.limit, self.uses = test, what, limit, []

    def use(self, detail: str) -> None:
        self.uses.append(detail)

    def close(self, total: int) -> int:
        line = f"[hatch] {self.test}: {self.what}: used {len(self.uses)} of {total} (limit {self.limit})"
        if self.uses:
            line += " -> " + "; ".join(self.uses[:4])
        print(line)
        d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
        if os.path.isdir(d):
            with open(os.path.join(d, "hatches.log"), "a") as f:
                f.write(line + "\n")
        assert len(self.uses) <= self.limit, line
        return len(self.uses)


def ranklist_near_tie(win_scores, got, want, k, rel=1e-5):
    """SURVEY.md §7 H1: CPU-fp32 and GPU-fp32 frame scores differ in summation order (~1e-7), so two DIFFERENT windows
    whose reference scores lie within `rel` of each other may swap.  True iff every position < k where `got` and `want`
    disagree is such a swap: the reference's scores of got[p] and want[p] are within rel * max(1, |s|).  Exact ties
    (shared frame, equal stored score) must come out in index order and never pass as a "near-tie" with themselves
    swapped, because both sides break exact ties by ascending window id."""
    s = np.asarray(win_scores, dtype=np.float64)
    for p in range(min(k, len(want))):
        if p >= len(got):
            return False
        if got[p] != want[p]:
            a, b = s[got[p]], s[want[p]]
            if not (0 < abs(a - b) <= rel * max(1.0, abs(b))):
                return False
    return True


def oracle_window_scores(sd, cfg, ds, q):
    """The reference's window scores of one query (stage 0 + 1 of the oracle), for the near-tie audit."""
    import torch
    from oracle import cone_oracle as O
    with torch.no_grad():
        ctx = O.stage0_video_context(sd, torch.from_numpy(O.l2_normalize_np(ds.videos[q.video_idx])))
        _, fs = O.stage1_ranklist(ctx, torch.from_numpy(O.l2_normalize_np(q.cls)), cfg.max_v_l)
        return O.window_scores(fs, cfg.max_v_l).numpy()


def pooled_bounds(spans, dur):
    """[start, end) pooled-row bounds as model.py:186-192 computes them in fp32 (clipping aside)."""
    sp = np.asarray(spans, dtype=np.float32)
    x1 = (sp[..., 0] - np.float32(0.5) * sp[..., 1]) * dur
    x2 = (sp[..., 0] + np.float32(0.5) * sp[..., 1]) * dur
    return np.stack([np.maximum(np.floor(x1), 0), np.ceil(x2)])


def check_grounding_fp32(cfg, ds, res, ora, name):
    """fp32 mode against the oracle's `eval_pipeline`: rank-lists and windows exact, raw outputs within 1e-5, R@K
    identical, NMS'd lists equal up to the 4-decimal rounding.  A query whose matching score crossed a floor/ceil pooling
    boundary may differ; so may, counted, one other query per case: the candidates are sorted on scores rounded to 4
    decimals (inference.py:83), a 1e-7 difference that moves one rounding reorders rounded ties, and NMS then keeps
    another row."""
    from oracle import cone_oracle as O
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


def check_grounding_tc(cfg, ds, res, ora, name):
    """Tensor-core mode against the oracle's `eval_pipeline`, the criteria of tests/test_gpu_tc.py: identical top-k
    windows (the ranking is fp32 in every mode), spans and probabilities within TC_TOL, matching scores within TC_TOL
    where both sides pool the same rows, at most 8 % of the proposals with moved pooling bounds, R@K hit counts equal up
    to max(1, 0.5 % of the queries).  Returns the largest span / probability error."""
    from oracle import cone_oracle as O
    errs, n_prop, n_flip = [], 0, 0
    for q in ds.queries:
        r, o = res[q.query_id], ora[q.query_id]
        assert r["ranklist"][: cfg.topk_window] == o["ranklist"][: cfg.topk_window], q.query_id
        assert r["windows"] == o["windows"], q.query_id
        osp = np.stack(o["pred_spans"])
        errs.append(np.abs(r["pred_spans"] - osp).ravel())
        errs.append(np.abs(r["prob_fg"] - np.stack(o["prob_fg"])).ravel())
        dur = np.asarray([n for _, n in r["windows"]], dtype=np.float32)[:, None]
        same = np.all(pooled_bounds(r["pred_spans"], dur) == pooled_bounds(osp, dur), axis=0)
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
    return float(err.max())


# ---- the configuration matrix of tests/test_config_matrix.py (CPU) and tests/test_gpu_config_matrix.py (GPU) ----------
# (Lv, Lt) of dense windows of S = Lv + Lt rows, chosen at the boundaries of the attention dispatch (attention.cu):
# S 3 / 16 / 17, the NB 14|20 (112/113), <20, true> (145..160), <32, false> (161..), NB 26|32 (208/209), short|long
# (256/257) switches, the long memory kernel's 128-row chunks (384/385), and 511 / 512.  One handle with max_v_l 480
# and max_q_l 32 runs all of them: cone_forward takes any Lv <= max_v_l with Lv + Lt <= 512.
SWEEP_ROWS = [(2, 1), (8, 8), (9, 8), (90, 22), (90, 23), (120, 24), (120, 25), (125, 25), (128, 32), (130, 31),
              (180, 28), (180, 29), (224, 32), (232, 25), (300, 20), (352, 32), (384, 1), (440, 9), (480, 31), (480, 32)]
# fp32 decoder NQ 5 / 8, memory-direct cross-attention MT 3 / 4
SWEEP_NQ = (1, 6, 8)
# model-configuration axes, on 90 + 20 row windows unless stated
AXES = {
    "layers1_nq8": dict(enc_layers=1, dec_layers=1, num_queries=8),
    "layers3_nq6_ffn2048": dict(enc_layers=3, dec_layers=3, num_queries=6, dim_feedforward=2048),
    "layers8": dict(enc_layers=8, dec_layers=8),
    "ffn128": dict(dim_feedforward=128),
    "odd_dims": dict(v_feat_dim=48, t_feat_dim=16, v_motion_feat_dim=80),
    "dims320_192": dict(v_feat_dim=320, t_feat_dim=192),
    "window3": dict(max_v_l=2, max_q_l=1, num_queries=1),
    "ffn1040": dict(dim_feedforward=1040),
}


def sweep_cfg(nq):
    from cone_b200.config import EGO4D
    return EGO4D.replace(max_v_l=480, max_q_l=32, num_queries=nq)


def axis_cfg(name):
    from cone_b200.config import EGO4D
    return EGO4D.replace(**dict(dict(max_v_l=90, max_q_l=20), **AXES[name]))


def dense_batch(cfg, lv, lt, seed):
    """B = 5 padded windows as start_end_collate emits them: valid lengths vlen = [Lv, 1, ceil(Lv/2), Lv-1, random],
    tlen = [Lt, Lt, 1, Lt//2, random] (at least 1), padding zeroed.  Returns (motion rows [B, Lv, motion_dim], appearance
    rows [B, Lv, v_feat_dim], vid mask, tokens, token mask, normalised CLS); the two row tensors are one tensor when the
    model has no separate motion stream."""
    import torch
    g = torch.Generator().manual_seed(seed)
    r = lambda n: int(torch.randint(1, n + 1, (1,), generator=g))
    vlen = [max(1, x) for x in (lv, 1, -(-lv // 2), lv - 1, r(lv))]
    tlen = [max(1, x) for x in (lt, lt, 1, lt // 2, r(lt))]
    B = len(vlen)
    mot = torch.randn(B, lv, cfg.motion_dim, generator=g)
    app = torch.randn(B, lv, cfg.v_feat_dim, generator=g) if cfg.v_motion_feat_dim else mot
    txt = torch.randn(B, lt, cfg.t_feat_dim, generator=g)
    txt = txt / (txt.norm(dim=-1, keepdim=True) + 1e-5)
    cls = torch.randn(B, cfg.v_feat_dim, generator=g)
    cls = cls / (cls.norm(dim=-1, keepdim=True) + 1e-5)
    vm, tm = torch.zeros(B, lv), torch.zeros(B, lt)
    for i in range(B):
        vm[i, : vlen[i]] = 1
        tm[i, : tlen[i]] = 1
        mot[i, vlen[i]:] = 0
        app[i, vlen[i]:] = 0
        txt[i, tlen[i]:] = 0
    return mot, app, vm, txt, tm, cls


# ---- proposals at the pooling edges of A9 (tests/test_matching.py on the CPU, tests/test_gpu_matching.py on the GPU) ----
def span_products(spans, dur):
    """fp32 (x1 * dur, x2 * dur) of proposals (cx, w), in the operation order of `O.proposal_bounds`."""
    import torch
    from oracle import cone_oracle as O
    xx = O.span_cxw_to_xx(torch.as_tensor(np.asarray(spans, np.float32))) * torch.tensor(float(dur), dtype=torch.float32)
    return xx[..., 0].numpy(), xx[..., 1].numpy()


def boundary_spans(dur, ks=(1, 3, 6), a_values=None, n_ulps=8, reach=4096):
    """fp32 proposals whose floor(x1 * dur) or ceil(x2 * dur) sits on an integer boundary: exact widths w = 2^-k, and cx
    scanned over +-n_ulps ulps (np.nextafter) around a/dur + w/2 (x1 * dur near the integer a) and a/dur - w/2
    (x2 * dur near a), then at +-16, 32, ... `reach` ulps: where dur times an ulp of x is below an ulp of a, several cx
    give the same product, and the wider steps reach the products on both sides of it.
    Returns (spans [M, 2] float32, group [M]): each group is one scan, in increasing cx."""
    if a_values is None:
        a_values = sorted({0, 1, dur // 2, dur - 1, dur})
    spans, group = [], []
    for k in ks:
        w = np.float32(2.0 ** -k)
        for a in a_values:
            for sign in (1, -1):
                c = np.float32(a / dur + sign * float(w) / 2)
                lo, hi = [c], [c]
                dn, up = c, c
                for i in range(1, reach + 1):
                    dn, up = np.nextafter(dn, np.float32(-np.inf)), np.nextafter(up, np.float32(np.inf))
                    if i <= n_ulps or (i & (i - 1)) == 0:
                        lo.append(dn)
                        hi.append(up)
                cx = np.asarray(lo[::-1] + hi[1:], np.float32)
                spans.append(np.stack([cx, np.full_like(cx, w)], 1))
                group.append(np.full(len(cx), len(group)))
    return np.concatenate(spans).astype(np.float32), np.concatenate(group)


def boundary_hits(spans, group, dur):
    """Indices of the proposals of `boundary_spans` whose x1 * dur or x2 * dur is an exact fp32 integer, and of their
    scan neighbours (one cx ulp away), which miss it."""
    x1, x2 = span_products(spans, dur)
    exact = (x1 == np.floor(x1)) | (x2 == np.floor(x2))
    keep = exact.copy()
    for i in np.nonzero(exact)[0]:
        for j in (i - 1, i + 1):
            if 0 <= j < len(spans) and group[j] == group[i]:
                keep[j] = True
    return np.nonzero(keep)[0]


def edge_spans(dur, pad, seed):
    """fp32 proposals of one window of `dur` data rows zero padded to `pad` rows, at every edge of the pooling: random
    spans, x1 < 0, ends past `dur` inside the pad, ends past `pad`, empty slices (w = 0 on an integer), start >= pad,
    negative ends (-1, -pad, -pad - 1, -0.0), a negative width, NaN, and the floor/ceil boundary spans of
    `boundary_spans` (exact hits and their 1-ulp misses)."""
    rng = np.random.default_rng(seed)
    d = float(max(dur, 1))
    neg_end = lambda e: ((e - 0.5) / d, 0.0)  # x1 = x2 = (e - 0.5) / dur: start 0, end e
    x2_in_pad = (dur + pad) / 2 / d  # [0.5 dur, (dur + pad) / 2)
    rows = [(0.05, 0.5), (0.1, 0.9), (-0.2, 0.3),  # x1 < 0
            ((0.5 + x2_in_pad) / 2, x2_in_pad - 0.5),  # end past dur, inside the pad
            (pad / d, 1.0), (2.0 * pad / d, 0.5), (0.9, 0.6),  # end past pad
            (0.0, 0.0), (1.0, 0.0), (0.5, 0.0),  # empty slices
            (3.0 * pad / d + 0.1, 0.1), (pad / d + 0.5 / d, 1.0 / d),  # start >= pad
            neg_end(-1), neg_end(-pad), neg_end(-pad - 1), (-0.4 / d, 0.0), (-0.5, 0.4), (0.3, -0.8),  # negative ends
            (0.5, -1.5),  # negative width: start > 0 > end
            (np.nan, 0.3), (0.5, np.nan), (np.nan, np.nan)]
    sp = [np.asarray(rows, np.float32),
          rng.uniform(0, 1, (12, 2)).astype(np.float32),
          np.stack([rng.uniform(-0.3, 1.3, 8), rng.uniform(0, 1.2, 8)], 1).astype(np.float32)]
    if dur > 0:
        b, g = boundary_spans(dur, ks=(1, 6), a_values=sorted({0, 1, dur // 2, dur}))
        sp.append(b[boundary_hits(b, g, dur)])
    return np.concatenate(sp).astype(np.float32)
