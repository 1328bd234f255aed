"""CPU checks of the window pre-filter: the reference helpers of tests/test_gpu_prefilter.py against the oracle and
against torch.sort's ordering of NaN, +-0 and +-inf; the header's `ranklist_stride` and `score_offsets` contracts; and
the engine's refusal of a short explicit rank-list stride before any launch."""
import math
import os
import re

import pytest
import torch

from cone_b200.engine import ConeEngine
from oracle import cone_oracle as O
import test_gpu_prefilter as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("max_v_l", [2, 3, 90, 125])
@pytest.mark.parametrize("kind", ["random", "ties", "constant"])
def test_reference_helpers_equal_the_oracle(max_v_l, kind):
    g = torch.Generator().manual_seed(max_v_l)
    for L in (1, 2, 61, 62, 63, 500, 1001):
        fs = G.synth_scores(kind, L, max_v_l, g)
        ws = G.ref_window_scores(fs, max_v_l)
        want = O.window_scores(fs, max_v_l)
        assert ws.shape == want.shape and torch.equal(ws, want), (L, kind)
        assert G.ref_ranklist(ws).tolist() == O.window_ranklist(fs, max_v_l), (L, kind)
        assert G.num_window(L, max_v_l) == len(want)
    for nw in (2, 33, 257):
        assert G.num_window(G.frames_for_windows(nw, max_v_l), max_v_l) == nw


@pytest.mark.parametrize("kind", G.VALUE_CLASSES)
def test_kernel_key_order_equals_stable_torch_sort(kind):
    """the kernel's 64-bit keys order NaN, +-0, +-inf and +-FLT_MAX as torch.sort(descending=True, stable=True)"""
    g = torch.Generator().manual_seed(1)
    for max_v_l in (2, 90):
        for L in (1, 30, 700):
            ws = G.ref_window_scores(G.synth_scores(kind, L, max_v_l, g), max_v_l)
            assert G.kernel_order(ws.numpy()).tolist() == G.ref_ranklist(ws).tolist(), (kind, L)
    edge = torch.tensor([0.0, -0.0, math.nan, -math.inf, math.inf, math.nan, -0.0, G.FLT_MAX, -G.FLT_MAX, 1.0, 0.0])
    assert G.kernel_order(edge.numpy()).tolist() == G.ref_ranklist(edge).tolist()
    # a window made entirely of NaN scores NaN: torch.max propagates it
    assert math.isnan(float(G.ref_window_scores(torch.tensor([1.0, math.nan, math.nan, 2.0]), 4)[2]))


def test_header_states_the_stride_and_offset_contracts():
    src = open(os.path.join(ROOT, "include", "cone_b200.h")).read()
    fs = src[src.index("int cone_frame_scores") - 900: src.index("int cone_frame_scores")]
    assert "score_offsets[q]" in fs and re.search(r"padded or\s*\*?\s*ordered freely", fs)
    rl = src[src.index("int cone_window_ranklist") - 900: src.index("int cone_window_ranklist")]
    assert re.search(r"ranklist_stride must be >= num_window\(q\) for every query", rl)
    assert "16384" in rl and "-1" in rl


def _engine_stub():
    """ConeEngine.window_ranklist needs the config only until it launches: enough to see a refusal without a device"""
    from cone_b200.config import EGO4D
    eng = object.__new__(ConeEngine)
    eng.cfg = EGO4D.replace(max_v_l=4)
    return eng


def test_engine_refuses_a_short_stride_before_any_launch():
    eng = _engine_stub()
    counts = torch.tensor([198, 78, 18], dtype=torch.int32)  # 100, 40 and 10 windows at max_v_l 4
    scores = torch.zeros(int(counts.sum()))
    offs = torch.tensor([0, 198, 276], dtype=torch.int64)
    with pytest.raises(ValueError, match=r"ranklist_stride 99 .*\(100 windows"):
        eng.window_ranklist(scores, offs, counts, ranklist_stride=99)
    with pytest.raises(ValueError, match=r"ranklist_stride 33 .*"):
        eng.window_ranklist(scores, offs, counts, ranklist_stride=33, max_frame_count=198)
    # the caller's host maximum is used when given, whatever frame_count holds
    with pytest.raises(ValueError, match="ranklist_stride"):
        eng.window_ranklist(scores, offs, counts[2:], ranklist_stride=50, max_frame_count=198)
    # a stride that holds every window passes the check and stops only at the device requirement
    with pytest.raises((ValueError, RuntimeError, AssertionError)) as e:
        eng.window_ranklist(scores, offs, counts, ranklist_stride=100)
    assert "ranklist_stride" not in str(e.value)
