"""The transformer core over the window shapes, slot counts and layer configurations the library accepts, in fp32 and
tensor-core mode, against the oracle evaluated in float64 (tests/fp64_reference.py).

- Window rows: dense `cone_forward` (saliency and aux heads) and `cone_clip_matching` on one handle per slot count
  (max_v_l 480, max_q_l 32) at the S of helpers.SWEEP_ROWS, nq 1 / 6 / 8.
- Model axes (helpers.AXES): 1 / 3 / 8 layers, ffn 128 / 2048, feature dims that are multiples of 16 but not of 64
  or 128, 3-row windows; the drop-in `CONE` module's aux outputs; ffn 1040, which tensor-core mode refuses.
- The grounding path (`ground_dataset`), whose layer-0 row tables, TMA-gather residual and NMS the dense forward does
  not run: against the oracle's pipeline and a per-window fp64 forward.
- The profiler shows that the cases launch every attention kernel instantiation they are meant to cover.
- CONE_FUSED_TAIL=0 and CONE_ATTN_TC=1, which the library reads once per process, in child processes.

Tolerances (helpers.py): FP32_TOL on every fp32 output; TC_TOL on tensor-core spans, class probabilities (final and
aux) and matching scores.  Tensor-core saliency is held to max(TC_TOL, 2x the saliency error of the default Ego4D
configuration measured in the same process)."""
import dataclasses
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from cone_b200 import _lib
from cone_b200._lib import ConeError
from cone_b200.config import EGO4D
from cone_b200.engine import ConeEngine
from cone_b200.inference import ground_dataset
from cone_b200.model import CONE
from cone_b200.synth import make_dataset
from cone_b200.weights import init_state_dict
from oracle import cone_oracle as O
import fp64_reference as R
import motion_oracle as MO
from helpers import (AXES, FP32_TOL, SWEEP_NQ, SWEEP_ROWS, TC_TOL, assert_match_close, axis_cfg, check_grounding_fp32,
                     check_grounding_tc, dense_batch, sweep_cfg)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ATTN_TC_ROWS = 192  # covers every window the opt-in tcgen05 encoder attention takes (enc_attn_tc_supported: 160 keys)
PRECISIONS = ("fp32", "tc")

_refs = {}
_engine = {}


def _err(a, b):
    """largest |a - b| / max(1, |b|), the reading of the tolerances in helpers.py"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    return float((np.abs(a - b) / np.maximum(1.0, np.abs(b))).max()) if a.size else 0.0


def _engine_for(key, cfg, sd, precision):
    """one live engine at a time: a tensor-core handle at max_v_l 480 holds 2.4 GB of position tables"""
    if key not in _engine:
        _engine.clear()
        torch.cuda.empty_cache()
        _engine[key] = ConeEngine(cfg, sd, device=DEV, precision=precision, workspace_bytes=1 << 30)
    return _engine[key]


def _dense_ref(cfg, sd, lv, lt, seed):
    """the fp64 forward and the matching scores of the reference's spans, once per (config, shape)"""
    key = (cfg, lv, lt, seed)
    if key not in _refs:
        mot, app, vm, txt, tm, cls = dense_batch(cfg, lv, lt, seed)
        ref = R.cone_forward(sd, cfg, txt, tm, mot, vm)
        spans32 = ref["pred_spans"].float()  # the proposals both sides pool
        _refs[key] = (mot, app, vm, txt, tm, cls, ref, spans32, R.clip_matching(sd, cls, app, vm, spans32))
    return _refs[key]


def _run_dense(eng, cfg, sd, lv, lt, seed):
    mot, app, vm, txt, tm, cls, ref, spans32, rmatch = _dense_ref(cfg, sd, lv, lt, seed)
    vl, tl = vm.sum(1).int().to(DEV), tm.sum(1).int().to(DEV)
    logits, spans, sal, aux_l, aux_s = eng.forward(txt.to(DEV), tl, mot.to(DEV), vl, want_saliency=True, want_aux=True)
    match = eng.clip_matching(cls.to(DEV), app.to(DEV), vl, spans32.to(DEV))
    torch.cuda.synchronize()
    return dict(logits=logits.cpu(), spans=spans.cpu(), sal=sal.cpu(), match=match.cpu(),
                aux_l=None if aux_l is None else aux_l.cpu(), aux_s=None if aux_s is None else aux_s.cpu())


def _dense_errors(got, cfg, sd, lv, lt, seed, precision):
    """{quantity: largest error} of one dense batch; `match` is checked here with the floor/ceil exemption"""
    _, _, vm, _, _, _, ref, spans32, rmatch = _dense_ref(cfg, sd, lv, lt, seed)
    n_aux = cfg.dec_layers - 1
    assert (got["aux_l"] is None) == (n_aux == 0)
    aux = [(got["aux_l"][i], got["aux_s"][i], ref["aux_outputs"][i]) for i in range(n_aux)]
    prob = lambda x: torch.softmax(torch.as_tensor(x, dtype=torch.float64), -1)
    e = dict(spans=_err(got["spans"], ref["pred_spans"]), sal=_err(got["sal"], ref["saliency_scores"]),
             aux_spans=max([_err(s, r["pred_spans"]) for _, s, r in aux], default=0.0))
    if precision == "fp32":
        e["logits"] = _err(got["logits"], ref["pred_logits"])
        e["aux_logits"] = max([_err(lg, r["pred_logits"]) for lg, _, r in aux], default=0.0)
    else:
        e["prob"] = _err(prob(got["logits"]), prob(ref["pred_logits"]))
        e["aux_prob"] = max([_err(prob(lg), prob(r["pred_logits"])) for lg, _, r in aux], default=0.0)
    tol = FP32_TOL if precision == "fp32" else TC_TOL
    assert_match_close(got["match"], rmatch, spans32, vm.sum(1).numpy(), tol)
    e["match"] = _err(got["match"], rmatch)
    return e


def _check(errs, precision, sal_bound, what):
    """fp32: every quantity within FP32_TOL; tensor-core: within TC_TOL, saliency within `sal_bound`.  Prints the errors
    and returns the failures."""
    print(f"[matrix] {what}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    bad = []
    for k, v in errs.items():
        tol = FP32_TOL if precision == "fp32" else (sal_bound if k == "sal" else TC_TOL)
        if k == "match":
            continue  # asserted with the floor/ceil exemption in _dense_errors
        if not v <= tol:
            bad.append(f"{what}: {k} {v:.3e} > {tol:.1e}")
    return bad


@pytest.fixture(scope="module")
def sal_bound():
    """Tensor-core saliency has no contract of its own: the bound is twice the largest error of the default Ego4D
    configuration (90 + 20 rows, 5 slots, 2 / 2 layers), and never below TC_TOL.  The baseline takes the largest error
    over six batches, 2700 values, as many as the largest case compares (5 windows of 480 rows): the largest of n
    rounding errors grows with n, so a baseline over fewer values would not bound the same statistic."""
    cfg = EGO4D
    sd = init_state_dict(cfg, 3)
    eng = ConeEngine(cfg, sd, device=DEV, precision="tc", workspace_bytes=1 << 30)
    lv, lt = cfg.max_v_l, cfg.max_q_l
    base = max(_dense_errors(_run_dense(eng, cfg, sd, lv, lt, seed), cfg, sd, lv, lt, seed, "tc")["sal"]
               for seed in range(1, 7))
    bound = max(TC_TOL, 2 * base)
    print(f"[matrix] tensor-core saliency: Ego4D baseline {base:.3e}, bound {bound:.3e}")
    return bound


def _sweep_parts():
    out = []
    for precision in PRECISIONS:
        for nq in SWEEP_NQ:
            out += [(precision, nq, "upto192"), (precision, nq, "past192")]
    return out


@pytest.mark.parametrize("precision,nq,part", _sweep_parts(), ids=[f"{p}-nq{n}-{s}" for p, n, s in _sweep_parts()])
def test_window_rows(precision, nq, part, sal_bound):
    cfg = sweep_cfg(nq)
    sd = init_state_dict(cfg, 40 + nq)
    eng = _engine_for(("sweep", nq, precision), cfg, sd, precision)
    bad = []
    for lv, lt in SWEEP_ROWS:
        if (lv + lt <= ATTN_TC_ROWS) != (part == "upto192"):
            continue
        got = _run_dense(eng, cfg, sd, lv, lt, lv * 1000 + lt)
        bad += _check(_dense_errors(got, cfg, sd, lv, lt, lv * 1000 + lt, precision), precision, sal_bound,
                      f"{precision} nq {nq} S {lv + lt} ({lv}+{lt})")
    assert not bad, "\n".join(bad)


_AXIS_CASES = [(p, n) for n in AXES if n != "ffn1040" for p in PRECISIONS]


@pytest.mark.parametrize("precision,axis", _AXIS_CASES, ids=[f"{p}-{n}" for p, n in _AXIS_CASES])
def test_model_axes(precision, axis, sal_bound):
    cfg = axis_cfg(axis)
    sd = init_state_dict(cfg, 50 + list(AXES).index(axis))
    eng = _engine_for(("axis", axis, precision), cfg, sd, precision)
    lv, lt = cfg.max_v_l, cfg.max_q_l
    got = _run_dense(eng, cfg, sd, lv, lt, 7)
    bad = _check(_dense_errors(got, cfg, sd, lv, lt, 7, precision), precision, sal_bound, f"{precision} {axis}")
    assert not bad, "\n".join(bad)


def test_ffn_not_a_multiple_of_128_is_refused_in_tensor_core_mode():
    """ffn 1040 passes the dims check (a multiple of 16) but not the 128-column tcgen05 tiles of the FFN GEMMs: both
    transformer entry points refuse it up front with a message that names dim_feedforward, the calls that do not run
    the transformer work, and fp32 mode on the same weights handle matches the reference."""
    cfg = axis_cfg("ffn1040").replace(topk_window=3, eval_bsz=4)
    sd = init_state_dict(cfg, 57)
    eng = ConeEngine(cfg, sd, device=DEV, precision="tc", workspace_bytes=1 << 30)
    with pytest.raises(ConeError, match="dim_feedforward.*multiple of 128"):
        _run_dense(eng, cfg, sd, cfg.max_v_l, cfg.max_q_l, 7)
    ds = make_dataset(cfg, 2, [200, 91], [2, 1], seed=5)
    with pytest.raises(ConeError, match="cone_ground_windows: .*dim_feedforward"):
        ground_dataset(eng, ds.videos, ds.queries)  # cone_video_prepare (stage 0) ran in tensor-core mode first
    x = torch.randn(300, cfg.v_feat_dim, device=DEV)
    with torch.no_grad():
        want = O.adapter({k: v.to(DEV) for k, v in sd.items()}, x)
    assert (eng.adapter(x, residual=True, precision="tc") - want).abs().max().item() <= 5e-3 * want.abs().max().item()
    w = torch.randn(256, 128, device=DEV) / 128 ** 0.5
    assert (eng.linear(torch.randn(200, 128, device=DEV), w, precision="tc")).isfinite().all()
    eng.precision = _lib.PREC_FP32  # the same handle in fp32 mode
    got = _run_dense(eng, cfg, sd, cfg.max_v_l, cfg.max_q_l, 7)
    bad = _check(_dense_errors(got, cfg, sd, cfg.max_v_l, cfg.max_q_l, 7, "fp32"), "fp32", None, "fp32 ffn1040")
    assert not bad, "\n".join(bad)
    check_grounding_fp32(cfg, ds, ground_dataset(eng, ds.videos, ds.queries), O.eval_pipeline(sd, cfg, ds.videos,
                                                                                                ds.queries), "ffn1040")


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("axis", ["layers1_nq8", "layers3_nq6_ffn2048"])
def test_drop_in_aux_outputs(axis, precision):
    """`CONE(cfg, sd, aux_loss=True)` returns one aux entry per decoder layer but the last: none with one layer"""
    cfg = axis_cfg(axis)
    sd = init_state_dict(cfg, 60)
    model = CONE(cfg, sd, precision=precision, aux_loss=True).to(DEV).eval()
    mot, _, vm, txt, tm, _ = dense_batch(cfg, cfg.max_v_l, cfg.max_q_l, 9)
    ref = R.cone_forward(sd, cfg, txt, tm, mot, vm)
    out = model(src_txt=txt.to(DEV), src_txt_mask=tm.to(DEV), src_vid_motion=mot.to(DEV), src_vid_motion_mask=vm.to(DEV))
    assert len(out["aux_outputs"]) == cfg.dec_layers - 1 == len(ref["aux_outputs"])
    prob = lambda x: torch.softmax(torch.as_tensor(x, dtype=torch.float64).cpu(), -1)
    tol = FP32_TOL if precision == "fp32" else TC_TOL
    for a, r in zip(out["aux_outputs"] + [out], ref["aux_outputs"] + [ref]):
        assert _err(a["pred_spans"].cpu(), r["pred_spans"]) <= tol
        if precision == "fp32":
            assert _err(a["pred_logits"].cpu(), r["pred_logits"]) <= tol
        else:
            assert _err(prob(a["pred_logits"]), prob(r["pred_logits"])) <= tol


# ---- the grounding path -------------------------------------------------------------------------------------------
GROUND = {
    "layers1_nq8": axis_cfg("layers1_nq8"),
    "layers3_nq6_ffn2048_125+25": axis_cfg("layers3_nq6_ffn2048").replace(max_v_l=125, max_q_l=25),
    "odd_dims": axis_cfg("odd_dims"),
    "window3": axis_cfg("window3"),
    "nq8_440+9": sweep_cfg(8).replace(max_v_l=440, max_q_l=9),
}
_ground = {}


def _ground_case(name):
    """seeded weights, 3 videos / 7 queries (the first video several windows long, one shorter than a window), the
    oracle's fp32 pipeline, and the fp64 forward of every window it grounds"""
    if name not in _ground:
        cfg = GROUND[name].replace(topk_window=5, eval_bsz=4)
        lv = cfg.max_v_l
        sd = init_state_dict(cfg, 70 + list(GROUND).index(name))
        motion = cfg.v_motion_feat_dim or None
        ds = make_dataset(cfg, 3, [int(2.7 * lv) + 1, lv + lv // 3, lv // 2 + 17], [3, 2, 2], seed=lv, motion_dim=motion)
        ora = MO.eval_pipeline(sd, cfg, ds.videos, ds.queries, motion_videos=ds.motion if motion else None)
        rows, toks = [], []
        for q in ds.queries:
            tok, _ = O.prepare_query_text(q.tokens, q.cls, cfg.max_q_l)
            for s, n in ora[q.query_id]["windows"]:
                src = ds.motion[q.video_idx] if motion else ds.videos[q.video_idx]
                rows.append(torch.from_numpy(O.l2_normalize_np(src[s: s + n]) if motion else src[s: s + n]))
                toks.append(tok)
        # one padded batch: the padding length does not change a window's outputs
        vid, vm = O.pad_sequences(rows)
        txt, tm = O.pad_sequences(toks)
        ref = R.cone_forward(sd, cfg, txt, tm, vid, vm)
        prob = torch.softmax(ref["pred_logits"], -1)[..., 0]
        _ground[name] = (cfg, sd, ds, ora, ref["pred_spans"].numpy(), prob.numpy())
    return _ground[name]


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name", list(GROUND))
def test_grounding_path(name, precision):
    cfg, sd, ds, ora, ref_spans, ref_prob = _ground_case(name)
    eng = _engine_for(("ground", name, precision), cfg, sd, precision)
    res = ground_dataset(eng, ds.videos, ds.queries, motion_videos=ds.motion if cfg.v_motion_feat_dim else None)
    if precision == "fp32":
        check_grounding_fp32(cfg, ds, res, ora, f"fp32 {name}")
    else:
        check_grounding_tc(cfg, ds, res, ora, f"tc {name}")
    got_spans = np.concatenate([res[q.query_id]["pred_spans"] for q in ds.queries])
    got_prob = np.concatenate([res[q.query_id]["prob_fg"] for q in ds.queries])
    e = dict(spans=_err(got_spans, ref_spans), prob=_err(got_prob, ref_prob))
    print(f"[matrix] grounding {precision} {name} vs fp64, {len(ref_spans)} windows: "
          + " ".join(f"{k} {v:.2e}" for k, v in e.items()))
    tol = FP32_TOL if precision == "fp32" else TC_TOL
    assert max(e.values()) <= tol, e


@pytest.mark.parametrize("precision", PRECISIONS)
def test_odd_dims_fp16_features_are_bitwise_their_upcast(precision):
    """the row kernels (L2 norm, LayerNorm, pooling) step 4 elements per lane: D = 16, 48 and 80"""
    cfg, sd, ds, _, _, _ = _ground_case("odd_dims")
    eng = _engine_for(("ground", "odd_dims", precision), cfg, sd, precision)
    h = lambda xs: [x.astype(np.float16) for x in xs]
    u = lambda xs: [x.astype(np.float32) for x in xs]
    q16 = [dataclasses.replace(q, tokens=q.tokens.astype(np.float16), cls=q.cls.astype(np.float16)) for q in ds.queries]
    q32 = [dataclasses.replace(q, tokens=q.tokens.astype(np.float32), cls=q.cls.astype(np.float32)) for q in q16]
    a = ground_dataset(eng, h(ds.videos), q16, motion_videos=h(ds.motion))
    b = ground_dataset(eng, u(h(ds.videos)), q32, motion_videos=u(h(ds.motion)))
    assert a.keys() == b.keys()
    for k in a:
        for f in a[k]:
            x, y = a[k][f], b[k][f]
            assert (np.array_equal(x, y, equal_nan=True) and x.dtype == y.dtype) if isinstance(x, np.ndarray) else x == y, (k, f)


# ---- every instantiation the matrix claims to cover is launched --------------------------------------------------
EXPECTED_KERNELS = [
    "enc_self_attention_kernel<8>", "enc_self_attention_kernel<16>",
    "dec_cross_attention_kernel<float,5,8>", "dec_cross_attention_kernel<float,8,8>",
    "dec_cross_attention_kernel<float,5,16>", "dec_cross_attention_kernel<float,8,16>",
    "enc_attention_f16_kernel<20,true>", "enc_attention_f16_kernel<20,false>", "enc_attention_f16_kernel<32,false>",
    "enc_attention_f16_long_kernel",
] + [f"dec_cross_attention_mem_kernel<{nb},{mt}>" for nb in (14, 20, 26, 32) for mt in (3, 4)] + [
    "dec_cross_attention_mem_long_kernel<3>", "dec_cross_attention_mem_long_kernel<4>"]


def test_every_attention_instantiation_is_launched():
    """one pass over the window-rows and model-axes cases under torch.profiler: a change of a dispatch threshold that
    moves a case onto another kernel would leave an instantiation unlaunched"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for precision in PRECISIONS:
            for nq in SWEEP_NQ:
                cfg = sweep_cfg(nq)
                sd = init_state_dict(cfg, 40 + nq)
                eng = _engine_for(("sweep", nq, precision), cfg, sd, precision)
                for lv, lt in SWEEP_ROWS:
                    _run_dense(eng, cfg, sd, lv, lt, lv * 1000 + lt)
            for axis in AXES:
                if axis == "ffn1040":
                    continue
                cfg = axis_cfg(axis)
                sd = init_state_dict(cfg, 50 + list(AXES).index(axis))
                eng = _engine_for(("axis", axis, precision), cfg, sd, precision)
                _run_dense(eng, cfg, sd, cfg.max_v_l, cfg.max_q_l, 7)
    names = {e.key.replace(" ", "") for e in prof.key_averages()}
    missing = [k for k in EXPECTED_KERNELS if not any(k + ("(" if k.endswith("kernel") else "") in n for n in names)]
    launched = sorted(n for n in names if "attention" in n)
    print("[matrix] attention kernels launched:\n  " + "\n  ".join(launched))
    assert not missing, f"not launched: {missing}"


# ---- the two documented switches, read once per process -----------------------------------------------------------
def _child(env, tests):
    """run the given tensor-core tests of this module in a child process with `env` set; the child derives its saliency
    bound from the same Ego4D baseline, run with the same switch"""
    env = dict(os.environ, **env)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.environ.get("PYTHONPATH", "")])
    here = os.path.abspath(__file__)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-s", "-m", "gpu", "-p", "no:cacheprovider"]
                       + [f"{here}::{t}" for t in tests], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    print("\n".join(line for line in r.stdout.splitlines() if line.startswith("[")))
    assert r.returncode == 0, r.stdout[-6000:] + r.stderr[-3000:]
    assert f"{len(tests)} passed" in r.stdout, r.stdout[-2000:]


_TC_AXES = [f"test_model_axes[tc-{a}]" for p, a in _AXIS_CASES if p == "tc"]


def test_unfused_encoder_chain():
    """CONE_FUSED_TAIL=0: out_proj, norm1, the FFN and norm2 of the tensor-core encoder as separate GEMMs"""
    _child({"CONE_FUSED_TAIL": "0"}, [f"test_window_rows[tc-nq{n}-{s}]" for n in SWEEP_NQ for s in ("upto192", "past192")]
           + _TC_AXES + [f"test_grounding_path[{n}-tc]" for n in GROUND])


def test_tcgen05_encoder_attention():
    """CONE_ATTN_TC=1: the tcgen05 encoder attention on windows of up to 192 rows"""
    _child({"CONE_ATTN_TC": "1"}, [f"test_window_rows[tc-nq{n}-upto192]" for n in SWEEP_NQ] + _TC_AXES)
