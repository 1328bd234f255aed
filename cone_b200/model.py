"""Drop-in mirror of the reference's model surface (`cone/model.py`): `build_model(opt)` and a `CONE` module with
`forward`, `forward_clip_matching`, `adapter_layer`, whose arithmetic runs in libcone_b200 on the GPU.

It can be substituted by assignment (`cone.inference.build_model = cone_b200.build_model`) without editing
`cone/inference.py` (SURVEY.md §8b): it is an `nn.Module` with the reference's parameter names, so
`.to(device)`, `.eval()`, `.load_state_dict(checkpoint["model"])` and `.named_parameters()` behave as
`setup_model` expects (`cone/inference.py:502-537`).  Inference only: training-mode calls raise.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
from torch import nn

from . import _lib
from .config import ConeConfig
from .engine import ConeEngine
from .weights import init_state_dict, state_dict_shapes


def _prefix_lengths(mask: torch.Tensor, name: str) -> torch.Tensor:
    """Reference masks are float {0,1} prefix masks (`pad_sequences_1d`, utils/tensor_utils.py:38-53)."""
    lens = mask.sum(dim=1).to(torch.int32)
    ar = torch.arange(mask.shape[1], device=mask.device)[None, :]
    if not torch.equal(mask != 0, ar < lens[:, None]):
        raise NotImplementedError(f"{name}: only prefix (right-padded) masks are supported")
    return lens


class _AdapterLayer(nn.Module):
    """`model.adapter_layer`: MLP(Dv, 256, Dv, 2) (cone/model.py:80); callable on (..., Dv)."""

    def __init__(self, owner: "CONE"):
        super().__init__()
        object.__setattr__(self, "_owner", owner)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self._owner._engine_for(x.device).adapter(x.float(), residual=False)


class _ParamTree(nn.Module):
    pass


class CONE(nn.Module):
    """Same call surface as the reference `CONE` (cone/model.py:16-152)."""

    def __init__(self, cfg: ConeConfig, state_dict: Optional[Dict[str, torch.Tensor]] = None, precision: str = "fp32",
                 adapter_module: str = "linear", aux_loss: bool = False, workspace_bytes: int = 2 << 30):
        super().__init__()
        if adapter_module != "linear":
            raise NotImplementedError("only adapter_module='linear' is built (the reference's released setting)")
        self.cfg = cfg
        self.precision = precision
        self.adapter_module = adapter_module
        self.aux_loss = aux_loss
        self.num_queries = cfg.num_queries
        self._workspace_bytes = workspace_bytes
        self._engine: Optional[ConeEngine] = None
        self._engine_version = None
        sd = state_dict if state_dict is not None else init_state_dict(cfg, seed=0, perturb=False)
        self._names = list(state_dict_shapes(cfg))
        for name in self._names:  # nested containers so that parameter names equal the reference's
            parts = name.split(".")
            mod = self
            for p in parts[:-1]:
                if p == "adapter_layer" and mod is self:
                    if "adapter_layer" not in self._modules:
                        self.add_module("adapter_layer", _AdapterLayer(self))
                elif p not in mod._modules:
                    mod.add_module(p, _ParamTree())
                mod = mod._modules[p]
            mod.register_parameter(parts[-1], nn.Parameter(sd[name].detach().clone().float(), requires_grad=True))
        self.eval()

    # ---- plumbing -------------------------------------------------------------------------------
    def train(self, mode: bool = True):
        if mode:
            # the reference toggles train() around eval_epoch (cone/train.py); this build is inference-only
            pass
        return super().train(mode)

    def _weights_version(self):
        return tuple(p._version for p in self.parameters()) + (next(self.parameters()).device,)

    def _engine_for(self, device: torch.device) -> ConeEngine:
        if device.type != "cuda":
            raise _lib.ConeError("cone_b200.CONE runs on CUDA tensors only (no CPU fallback)")
        ver = self._weights_version()
        if self._engine is None or self._engine.device != device:
            self._engine = ConeEngine(self.cfg, dict(self.state_dict()), device=device, precision=self.precision,
                                      workspace_bytes=self._workspace_bytes)
            self._engine_version = ver
        elif ver != self._engine_version:  # load_state_dict / in-place update since the last pack
            self._engine.load_state_dict(dict(self.state_dict()))
            self._engine_version = ver
        return self._engine

    # ---- reference surface ------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, src_txt, src_txt_mask, src_vid_motion, src_vid_motion_mask):
        """cone/model.py:82-128; `src_vid_motion` is [B, L_vid, v_motion_feat_dim].  Returns pred_logits (B,nq,2), pred_spans (B,nq,2), saliency_scores (B,L_vid)
        and, with aux_loss, aux_outputs."""
        if self.training:
            raise NotImplementedError("cone_b200.CONE is inference-only: call model.eval() first")
        eng = self._engine_for(src_vid_motion.device)
        tl = _prefix_lengths(src_txt_mask, "src_txt_mask")
        vl = _prefix_lengths(src_vid_motion_mask, "src_vid_motion_mask")
        logits, spans, sal, aux_l, aux_s = eng.forward(src_txt.float(), tl, src_vid_motion.float(), vl,
                                                       want_saliency=True, want_aux=self.aux_loss)
        out = {"pred_logits": logits, "pred_spans": spans, "saliency_scores": sal}
        if self.aux_loss and aux_l is not None:
            out["aux_outputs"] = [{"pred_logits": a, "pred_spans": b} for a, b in zip(aux_l, aux_s)]
        return out

    @torch.no_grad()
    def forward_clip_matching(self, src_cls_txt, src_vid_appear, src_vid_appear_mask, proposal=None,
                              is_groundtruth=False):
        """cone/model.py:130-152 (`is_groundtruth=False` branch: the inference path)."""
        if is_groundtruth:
            raise NotImplementedError("ground-truth proposal matching is training-only (out of scope)")
        eng = self._engine_for(src_vid_appear.device)
        vl = _prefix_lengths(src_vid_appear_mask, "src_vid_appear_mask")
        return eng.clip_matching(src_cls_txt.float(), src_vid_appear.float(), vl, proposal.float())


class _NoCriterion(nn.Module):
    """`build_model` returns (model, criterion); `eval_epoch` only calls `.eval()` / `.to()` on it
    (cone/inference.py:229-233).  Losses are training-only and out of scope."""

    def forward(self, *a, **kw):
        raise NotImplementedError("SetCriterion (training losses) is out of scope of cone_b200")


def config_from_opt(opt) -> ConeConfig:
    """The fields `build_model` reads from the argparse namespace (cone/model.py:477-518)."""
    g = lambda k, d: getattr(opt, k, d)
    return ConeConfig(
        v_feat_dim=opt.v_appear_feat_dim, t_feat_dim=opt.t_feat_dim,
        v_motion_feat_dim=g("v_motion_feat_dim", 0), hidden_dim=g("hidden_dim", 256),
        nheads=g("nheads", 8), dim_feedforward=g("dim_feedforward", 1024), enc_layers=g("enc_layers", 2),
        dec_layers=g("dec_layers", 2), num_queries=g("num_queries", 5), n_input_proj=g("n_input_proj", 2),
        max_v_l=g("max_v_l", 90), max_q_l=g("max_q_l", 20), clip_length=g("clip_length", 1.0),
        topk_window=g("topk_window", 30), eval_bsz=g("eval_bsz", 32), nms_thd=g("nms_thd", -1),
        max_before_nms=g("max_before_nms", 200), max_after_nms=g("max_after_nms", 5), name=g("dset_name", "custom"))


def build_model(args):
    """Same signature and return as the reference `build_model(args) -> (model, criterion)` (cone/model.py:468)."""
    if getattr(args, "span_loss_type", "l1") != "l1" or getattr(args, "use_txt_pos", False) or getattr(args, "pre_norm", False):
        raise NotImplementedError("only span_loss_type='l1', use_txt_pos=False, pre_norm=False are built")
    model = CONE(config_from_opt(args), adapter_module=getattr(args, "adapter_module", "linear"),
                 aux_loss=getattr(args, "aux_loss", False), precision=getattr(args, "precision", "fp32"))
    return model, _NoCriterion()
