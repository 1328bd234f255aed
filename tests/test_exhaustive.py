"""CPU-side checks of exhaustive grounding (any topk_window, up to every window of a video): the workspace form of
stage 3 is exported with its sizing function and limits, and `sharded_eval --topk-window` resolves its argument."""
import ctypes as C
import os
import re

import pytest

from cone_b200 import _lib, build
from cone_b200.config import EGO4D, MAD768
from cone_b200.tools.sharded_eval import resolve_topk_window

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def test_new_symbols_and_limits_match_the_header(lib):
    for name in ("cone_fuse_nms_workspace_bytes", "cone_fuse_nms_ws"):
        assert name in _lib.SIGNATURES and hasattr(lib, name)
    src = open(os.path.join(ROOT, "include", "cone_b200.h")).read()
    defs = dict(re.findall(r"#define (CONE_FUSE_NMS_MAX_\w+) (\d+)", src))
    assert int(defs["CONE_FUSE_NMS_MAX_SHARED_CANDIDATES"]) == _lib.FUSE_NMS_MAX_SHARED_CANDIDATES == 2201
    assert int(defs["CONE_FUSE_NMS_MAX_CANDIDATES"]) == _lib.FUSE_NMS_MAX_CANDIDATES == 16384 * 8


def test_workspace_bytes_grow_with_queries_and_topk(lib):
    f = lib.cone_fuse_nms_workspace_bytes
    one = f(1, 441, 5)
    assert one > 0
    assert f(2, 441, 5) == 2 * one and f(640, 441, 5) == 640 * one
    assert f(1, 2905, 5) > one and f(1, 16384, 8) > f(1, 2905, 5)
    assert f(0, 30, 5) == f(1, 30, 5) > 0
    assert f(1, 16384, 8) < 16 << 20  # about 100 bytes per candidate


def test_workspace_bytes_refuse_past_the_limit(lib):
    f = lib.cone_fuse_nms_workspace_bytes
    assert f(1, 16385, 8) == 0
    assert b"131072" in lib.cone_last_error()
    assert f(1, 26215, 5) == 0 and b"131072" in lib.cone_last_error()
    assert f(1, 30, 9) == 0 and f(1, 0, 5) == 0 and f(-1, 30, 5) == 0


def test_topk_window_all_is_every_window_of_the_longest_video():
    lens = [300, 7200, 1500]
    assert resolve_topk_window("all", EGO4D, lens) == EGO4D.num_window(7200) == 7200 // 45 + 1
    assert resolve_topk_window("all", MAD768, [3000, 145000]) == MAD768.num_window(145000) == 2340
    assert resolve_topk_window("all", EGO4D.replace(max_v_l=6), [1000]) == 335
    assert resolve_topk_window("441", EGO4D, lens) == 441
    with pytest.raises(ValueError):
        resolve_topk_window("0", EGO4D, lens)
    with pytest.raises(ValueError):
        resolve_topk_window("every", EGO4D, lens)
