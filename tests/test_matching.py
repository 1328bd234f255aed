"""Proposal matching (A9) references, CPU side (tests/test_gpu_matching.py runs the kernels against them).

- `fp64_reference.clip_matching_exact_bounds` takes its [start, end) bounds from the fp32 spans, as the reference does,
  and in float32 returns exactly `O.clip_matching`'s bits (NaN included) on random spans and on every edge proposal.
- The boundary-span generator really produces proposals whose x1 * dur or x2 * dur is an exact fp32 integer, with 1-ulp
  misses on both sides of each, so a sweep built on it cannot silently lose its floor/ceil cases.
- Negative slice ends: bounds and pooled rows are those of Python slicing of the padded rows."""
import math

import numpy as np
import pytest
import torch

from cone_b200.config import EGO4D
from cone_b200.weights import init_state_dict
from oracle import cone_oracle as O
import fp64_reference as R
from helpers import boundary_hits, boundary_spans, edge_spans, span_products


def _bits(x):
    return torch.as_tensor(x).contiguous().view(torch.int32)


def _batch(cfg, vlens, pad, nq, seed):
    """zero-padded windows [B, pad, Dv], their masks, CLS vectors and, per window, the first nq edge proposals"""
    g = torch.Generator().manual_seed(seed)
    B = len(vlens)
    vid = torch.randn(B, pad, cfg.v_feat_dim, generator=g)
    vm = (torch.arange(pad)[None] < torch.tensor(vlens)[:, None]).float()
    vid = vid * vm[..., None]
    cls = torch.randn(B, cfg.v_feat_dim, generator=g)
    spans = torch.stack([torch.from_numpy(edge_spans(n, pad, seed + i)[:nq]) for i, n in enumerate(vlens)])
    return cls, vid, vm, spans


@pytest.mark.parametrize("pad,nq", [(90, 5), (91, 8), (7, 16)])
def test_exact_bounds_reference_in_float32_is_the_oracle(pad, nq):
    cfg = EGO4D.replace(v_feat_dim=48)
    sd = init_state_dict(cfg, 3)
    vlens = [pad, 1, -(-pad // 2), pad - 1, 0]
    edges = [edge_spans(n, pad, i) for i, n in enumerate(vlens)]
    cls, vid, vm, _ = _batch(cfg, vlens, pad, nq, 11)
    for lo in range(0, max(len(e) for e in edges), nq):  # every edge proposal of every window, nq at a time
        spans = torch.stack([torch.from_numpy(e[(lo + np.arange(nq)) % len(e)]) for e in edges])
        with torch.no_grad():
            want = O.clip_matching(sd, cls, vid, vm, spans)
        got = R.clip_matching_exact_bounds(sd, cls, vid, vm, spans, dtype=torch.float32)
        assert got.dtype == torch.float32 and torch.equal(_bits(got), _bits(want)), lo
        assert torch.isnan(want[-1]).all()  # the window of 0 rows: every slice is empty
    g = torch.Generator().manual_seed(5)
    cls, vid, vm, _ = _batch(cfg, vlens, pad, nq, 12)
    spans = torch.rand(len(vlens), nq, 2, generator=g)
    with torch.no_grad():
        want = O.clip_matching(sd, cls, vid, vm, spans)
    assert torch.equal(_bits(R.clip_matching_exact_bounds(sd, cls, vid, vm, spans, dtype=torch.float32)), _bits(want))
    m64 = R.clip_matching_exact_bounds(sd, cls, vid, vm, spans)
    assert m64.dtype == torch.float64
    ok = ~torch.isnan(want)
    assert torch.equal(ok, ~torch.isnan(m64))
    assert (m64[ok] - want[ok].double()).abs().max() <= 1e-5


@pytest.mark.parametrize("dur", [1, 2, 44, 45, 90, 91, 125, 480, 1000])
def test_boundary_spans_hit_and_miss_every_integer(dur):
    sp, group = boundary_spans(dur)
    x1, x2 = span_products(sp, dur)
    start, end = O.proposal_bounds(torch.from_numpy(sp)[None], torch.ones(1, dur))
    # the products are the reference's: its floor / ceil bounds are theirs
    assert torch.equal(start[0], torch.from_numpy(np.maximum(np.floor(x1), 0)).int())
    assert torch.equal(end[0], torch.from_numpy(np.ceil(x2)).int())
    hits = {1: set(), 2: set()}
    for gi in np.unique(group):
        idx = np.nonzero(group == gi)[0]
        assert np.all(np.diff(sp[idx, 0]) > 0) and len(set(sp[idx, 1])) == 1
        for which, x in ((1, x1[idx]), (2, x2[idx])):
            for i in np.nonzero(x == np.floor(x))[0]:
                # each exact hit m has a non-integer product on both sides in the same scan
                m = x[i]
                hits[which].add(float(m))
                assert np.any((x < m) & (x > m - 1)), (dur, gi, m)
                assert np.any((x > m) & (x < m + 1)), (dur, gi, m)
    # both bounds hit integers exactly: 0 and dur always (cx = +-w/2 exactly), and one inside the window when it has one.
    # Not every scan hits: when x1 has a smaller exponent than cx, x1 * dur moves by more than an ulp of a per step.
    for which in (1, 2):
        assert {0.0, float(dur)} <= hits[which], (which, sorted(hits[which]))
        assert dur < 2 or any(0 < m < dur for m in hits[which]), (which, sorted(hits[which]))
    keep = boundary_hits(sp, group, dur)
    kx1, kx2 = x1[keep], x2[keep]
    exact = (kx1 == np.floor(kx1)) | (kx2 == np.floor(kx2))
    assert exact.any() and (~exact).any()


def test_negative_ends_follow_python_slicing():
    pad, dur = 16, 8
    # row i of window 0 is the i-th unit vector: the pooled mean shows which rows were averaged
    vid = torch.eye(pad, dtype=torch.float64)[None]
    vm = torch.zeros(1, pad)
    vm[0, :dur] = 1
    # (end, span): x1 = x2 = (end - 0.5) / dur, or a span of width 0.4 centred at -0.5 (x2 * dur = -2.4)
    cases = [(-1, (-1.5 / dur, 0.0)), (-pad, (-2.0, 0.0)), (-pad - 1, (-17.5 / dur, 0.0)), (0, (-0.4 / dur, 0.0)),
             (-3, (-3.5 / dur, 0.0)), (-2, (-0.5, 0.4))]
    spans = torch.tensor([[s for _, s in cases]], dtype=torch.float32)
    start, end = O.proposal_bounds(spans, vm)
    want_end = [e for e, _ in cases]
    assert start[0].tolist() == [0] * len(cases)
    assert end[0].tolist() == want_end
    assert math.copysign(1.0, float(torch.ceil(torch.tensor(-0.4)))) < 0  # ceil gives -0.0, which is end 0
    pooled = R.pool_slices(vid, start, end)
    for j, e in enumerate(want_end):
        rows = list(range(pad))[0:e]
        if rows:
            want = torch.zeros(pad, dtype=torch.float64)
            want[rows] = 1.0 / len(rows)
            assert torch.equal(pooled[j], want), (e, rows)
        else:
            assert torch.isnan(pooled[j]).all(), e
    # the same bounds through the whole fp32 reference: finite exactly where the slice holds a row
    cfg = EGO4D.replace(v_feat_dim=16)
    sd = init_state_dict(cfg, 4)
    cls = torch.randn(1, 16, generator=torch.Generator().manual_seed(1))
    feat = torch.randn(1, pad, 16, generator=torch.Generator().manual_seed(2)) * vm[..., None]
    m = R.clip_matching_exact_bounds(sd, cls, feat, vm, spans, dtype=torch.float32)
    assert torch.isfinite(m[0]).tolist() == [len(list(range(pad))[0:e]) > 0 for e in want_end]
