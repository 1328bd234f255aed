"""The configuration matrix of tests/test_gpu_config_matrix.py, CPU side.

- The fp64 reference (tests/fp64_reference.py) adds nothing but the dtype: with float32 inputs it returns exactly the
  oracle's values, and in float64 it stays within 1e-5 of the fp32 oracle on every model-configuration axis.
- The dims check of the library (`check_dims`, read through `cone_weights_expected_floats`, which returns 0 for refused
  dims) accepts every configuration of the matrix with the float count of `state_dict_shapes`, and refuses the first
  value past each of its limits."""
import ctypes as C
import math

import pytest
import torch

from cone_b200 import _lib, build
from cone_b200.config import EGO4D
from cone_b200.weights import init_state_dict, state_dict_shapes
from oracle import cone_oracle as O
import fp64_reference as R
from helpers import AXES, FP32_TOL, SWEEP_NQ, assert_close, axis_cfg, dense_batch, sweep_cfg


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def _dims(cfg, **kw):
    f = dict(v_dim=cfg.v_feat_dim, t_dim=cfg.t_feat_dim, hidden=cfg.hidden_dim, nheads=cfg.nheads,
             ffn=cfg.dim_feedforward, enc_layers=cfg.enc_layers, dec_layers=cfg.dec_layers,
             num_queries=cfg.num_queries, max_v_l=cfg.max_v_l, max_q_l=cfg.max_q_l, m_dim=cfg.v_motion_feat_dim)
    f.update(kw)
    return _lib.ConeDims(*[f[n] for n, _ in _lib.ConeDims._fields_])


def _oracle32(sd, cfg, vid, vm, txt, tm):
    with torch.no_grad():
        return O.cone_forward(sd, txt, tm, vid, vm, cfg.nheads, cfg.enc_layers, cfg.dec_layers, cfg.n_input_proj)


@pytest.mark.parametrize("name", ["layers1_nq8", "layers3_nq6_ffn2048", "odd_dims"])
def test_fp64_reference_in_float32_is_the_oracle(name):
    cfg = axis_cfg(name)
    sd = init_state_dict(cfg, 1)
    mot, app, vm, txt, tm, cls = dense_batch(cfg, cfg.max_v_l, cfg.max_q_l, 7)
    want = _oracle32(sd, cfg, mot, vm, txt, tm)
    got = R.cone_forward(sd, cfg, txt, tm, mot, vm, dtype=torch.float32)
    for k in ("pred_logits", "pred_spans", "saliency_scores"):
        assert got[k].dtype == torch.float32 and torch.equal(got[k], want[k]), k
    assert len(got["aux_outputs"]) == cfg.dec_layers - 1
    for a, b in zip(got["aux_outputs"], want["aux_outputs"]):
        assert torch.equal(a["pred_logits"], b["pred_logits"]) and torch.equal(a["pred_spans"], b["pred_spans"])
    with torch.no_grad():
        wm = O.clip_matching(sd, cls, app, vm, want["pred_spans"])
    assert torch.equal(R.clip_matching(sd, cls, app, vm, want["pred_spans"], dtype=torch.float32), wm)


@pytest.mark.parametrize("name", list(AXES))
def test_fp64_reference_agrees_with_the_fp32_oracle(name):
    cfg = axis_cfg(name)
    sd = init_state_dict(cfg, 2)
    mot, app, vm, txt, tm, cls = dense_batch(cfg, cfg.max_v_l, cfg.max_q_l, 11)
    ref = R.cone_forward(sd, cfg, txt, tm, mot, vm)
    o32 = _oracle32(sd, cfg, mot, vm, txt, tm)
    assert ref["pred_spans"].dtype == torch.float64 and ref["saliency_scores"].dtype == torch.float64
    assert len(ref["aux_outputs"]) == cfg.dec_layers - 1
    for k in ("pred_logits", "pred_spans", "saliency_scores"):
        assert_close(o32[k], ref[k], FP32_TOL, k)
    for a, b in zip(o32["aux_outputs"], ref["aux_outputs"]):
        assert_close(a["pred_logits"], b["pred_logits"], FP32_TOL, "aux_logits")
        assert_close(a["pred_spans"], b["pred_spans"], FP32_TOL, "aux_spans")
    # matching on the same proposals: only the pooled means, the adapter and the cosine differ in precision
    with torch.no_grad():
        m32 = O.clip_matching(sd, cls, app, vm, o32["pred_spans"])
    m64 = R.clip_matching(sd, cls, app, vm, o32["pred_spans"])
    assert m64.dtype == torch.float64
    assert_close(m32, m64, FP32_TOL, "match")


_MATRIX = [("sweep_nq%d" % nq, sweep_cfg(nq)) for nq in SWEEP_NQ] + [(n, axis_cfg(n)) for n in AXES]


@pytest.mark.parametrize("name,cfg", _MATRIX, ids=[n for n, _ in _MATRIX])
def test_matrix_configs_are_accepted(lib, name, cfg):
    want = sum(math.prod(s) for s in state_dict_shapes(cfg).values())
    assert lib.cone_weights_expected_floats(C.byref(_dims(cfg))) == want, lib.cone_last_error()


# the first value past each limit of check_dims (api.cu), from an accepted Ego4D configuration
PAST_LIMITS = [("hidden", 128), ("nheads", 4), ("ffn", 1000), ("ffn", 0), ("enc_layers", 0), ("enc_layers", 9),
               ("dec_layers", 0), ("dec_layers", 9), ("num_queries", 0), ("num_queries", 9), ("max_v_l", 1),
               ("max_q_l", 0), ("v_dim", 40), ("t_dim", 40), ("m_dim", 40)]


@pytest.mark.parametrize("field,value", PAST_LIMITS, ids=[f"{f}={v}" for f, v in PAST_LIMITS])
def test_first_value_past_each_limit_is_refused(lib, field, value):
    assert lib.cone_weights_expected_floats(C.byref(_dims(EGO4D))) > 0
    assert lib.cone_weights_expected_floats(C.byref(_dims(EGO4D, **{field: value}))) == 0
    assert lib.cone_last_error(), field
    assert lib.cone_workspace_bytes(C.byref(_dims(EGO4D, **{field: value})), 4, 90, 20) == 0


@pytest.mark.parametrize("field,value", [("ffn", 16), ("enc_layers", 8), ("dec_layers", 8), ("num_queries", 8),
                                         ("max_v_l", 2), ("max_q_l", 1), ("v_dim", 16), ("t_dim", 16), ("m_dim", 16)])
def test_last_value_inside_each_limit_is_accepted(lib, field, value):
    assert lib.cone_weights_expected_floats(C.byref(_dims(EGO4D, **{field: value}))) > 0, lib.cone_last_error()
