"""Windows of up to 512 rows (max_v_l + max_q_l <= 512), CPU side: the dims check of the library accepts them and
refuses longer ones with the limit in the message.  The kernels are covered by tests/test_gpu_long_windows.py."""
import ctypes as C
import math

import pytest

from cone_b200 import _lib, build
from cone_b200.config import MAD768
from cone_b200.weights import state_dict_shapes


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _dims(max_v_l, max_q_l):
    cfg = MAD768
    return _lib.ConeDims(cfg.v_feat_dim, cfg.t_feat_dim, cfg.hidden_dim, cfg.nheads, cfg.dim_feedforward, cfg.enc_layers,
                         cfg.dec_layers, cfg.num_queries, max_v_l, max_q_l)


@pytest.mark.parametrize("max_v_l,max_q_l", [(231, 25), (232, 25), (300, 77), (480, 32), (256, 256), (510, 2)])
def test_windows_up_to_512_rows_are_accepted(lib, max_v_l, max_q_l):
    want = sum(math.prod(s) for s in state_dict_shapes(MAD768.replace(max_v_l=max_v_l, max_q_l=max_q_l)).values())
    assert lib.cone_weights_expected_floats(C.byref(_dims(max_v_l, max_q_l))) == want
    assert lib.cone_workspace_bytes(C.byref(_dims(max_v_l, max_q_l)), 8, max_v_l, max_q_l) > 0


@pytest.mark.parametrize("max_v_l,max_q_l", [(488, 25), (256, 257), (600, 20)])
def test_windows_past_512_rows_are_refused(lib, max_v_l, max_q_l):
    d = _dims(max_v_l, max_q_l)
    assert lib.cone_weights_expected_floats(C.byref(d)) == 0
    msg = lib.cone_last_error()
    assert b"512" in msg and str(max_v_l + max_q_l).encode() in msg, msg
    assert lib.cone_workspace_bytes(C.byref(d), 8, max_v_l, max_q_l) == 0


def test_version_is_4(lib):
    assert lib.cone_version() == 4
