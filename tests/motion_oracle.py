"""Two-stream restatement of the oracle's `eval_pipeline` (separate motion and appearance features).

TEST INFRASTRUCTURE ONLY.  The reference reads the motion features of a window through `--motion_feat_dir` and its
appearance features through `--appearance_feat_dir` (cone/ego4d_mad_dataloader.py:77, 134-137, 284-302):

  - stages 0/1 rank windows on the normalised appearance features (unchanged);
  - stage 2 feeds Moment-DETR the motion rows of each window [s, e), each row L2-normalised x / (||x|| + 1e-5);
  - the fine matching mean-pools the RAW appearance rows of the window (unchanged);
  - window bounds, masks and durations come from the window and are shared by both streams.

No reference goldens exist for this configuration, so this module is built only from functions of
`oracle/cone_oracle.py` that the existing goldens pin, and with `motion_videos=None` it must equal that module's
`eval_pipeline` exactly (tests/test_motion_stream.py checks it).
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F

from oracle import cone_oracle as O


def check_streams(videos: Sequence[np.ndarray], motion_videos: Optional[Sequence[np.ndarray]]) -> None:
    """Both streams are sliced with the same [s, e): every video needs as many motion rows as appearance rows."""
    if motion_videos is None:
        return
    if len(motion_videos) != len(videos):
        raise ValueError(f"{len(motion_videos)} motion feature tensors for {len(videos)} videos")
    for v, (a, m) in enumerate(zip(videos, motion_videos)):
        if len(a) != len(m):
            raise ValueError(f"video {v}: {len(m)} motion rows for {len(a)} appearance rows")


def eval_pipeline(sd: Dict[str, torch.Tensor], cfg, videos: Sequence[np.ndarray], queries,
                  motion_videos: Optional[Sequence[np.ndarray]] = None, collect_raw: bool = True) -> Dict[str, dict]:
    """`oracle.cone_oracle.eval_pipeline` with an optional motion stream; same return layout."""
    check_streams(videos, motion_videos)
    nheads, el, dl, nip = cfg.nheads, cfg.enc_layers, cfg.dec_layers, cfg.n_input_proj
    with torch.no_grad():
        ctx = [O.stage0_video_context(sd, torch.from_numpy(O.l2_normalize_np(v))) for v in videos]
        raw = [torch.from_numpy(v) for v in videos]
        res: Dict[str, dict] = {}
        for q in queries:
            cls_n = torch.from_numpy(O.l2_normalize_np(q.cls))
            rl, _ = O.stage1_ranklist(ctx[q.video_idx], cls_n, cfg.max_v_l)
            res[q.query_id] = {"ranklist": rl}
        for b0 in range(0, len(queries), cfg.eval_bsz):
            batch = queries[b0: b0 + cfg.eval_bsz]
            apps, mots, toks, clss, meta = [], [], [], [], []
            for q in batch:
                tok, cls_n = O.prepare_query_text(q.tokens, q.cls, cfg.max_q_l)
                for (s, n, rows) in O.slice_query_windows(raw[q.video_idx], res[q.query_id]["ranklist"],
                                                          cfg.topk_window, cfg.max_v_l):
                    apps.append(rows)
                    if motion_videos is None:  # one feature source: the raw appearance slice is the motion input
                        mots.append(rows)
                    else:  # the motion branch of the dataloader (:284-292): slice, then normalise per row
                        mots.append(torch.from_numpy(O.l2_normalize_np(motion_videos[q.video_idx][s: s + n])))
                    toks.append(tok)
                    clss.append(cls_n)
                    meta.append((q.query_id, s, n))
            src_app, vid_mask = O.pad_sequences(apps)
            src_mot, _ = O.pad_sequences(mots)
            src_txt, txt_mask = O.pad_sequences(toks)
            src_cls = torch.FloatTensor(np.stack(clss))
            out = O.cone_forward(sd, src_txt, txt_mask, src_mot, vid_mask, nheads, el, dl, nip)
            prob = F.softmax(out["pred_logits"], -1)[..., 0]
            match = O.clip_matching(sd, src_cls, src_app, vid_mask, out["pred_spans"])
            for i, (qid, s, n) in enumerate(meta):
                r = res[qid]
                r.setdefault("windows", []).append((s, n))
                r.setdefault("rows", []).extend(
                    O.compose_window_rows(out["pred_spans"][i], prob[i], match[i], n, s, cfg.clip_length))
                if collect_raw:
                    r.setdefault("pred_spans", []).append(out["pred_spans"][i].numpy().copy())
                    r.setdefault("prob_fg", []).append(prob[i].numpy().copy())
                    r.setdefault("match", []).append(match[i].numpy().copy())
        for q in queries:
            r = res[q.query_id]
            fused = O.score_fusion(r["rows"])
            for name, idx in (("fusion", 2), ("proposal", 0), ("matching", 1)):
                r[name] = O.post_processing_nms(fused, idx, cfg.nms_thd, cfg.max_before_nms, cfg.max_after_nms)
    return res
