"""Sharded evaluation driver: one process per GPU (torchrun), videos assigned to ranks by longest-processing-time,
stages 0-3 + metric counters on every rank, ONE all-reduce of the integer counters (SURVEY.md §8e / §8(f)1).

    torchrun --nnodes=1 --nproc-per-node N -m cone_b200.tools.sharded_eval --config ego4d --videos 12 --queries 6 --out m.json

Synthetic data (seeded) so that the same command on 1 and on N GPUs must print identical tables; with real features
replace `make_dataset` by `ingest.load_queries` + feature stores.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os

import numpy as np
import torch
import torch.distributed as dist

from ..config import PRESETS
from ..engine import ConeEngine
from ..inference import MODES, evaluate_dataset
from ..sharding import lpt_assign, reduce_counters, video_cost
from ..synth import make_dataset
from ..weights import init_state_dict


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="ego4d", choices=sorted(PRESETS))
    ap.add_argument("--videos", type=int, default=12)
    ap.add_argument("--frames", type=int, nargs=2, default=(300, 1500))
    ap.add_argument("--queries", type=int, default=6, help="queries per video")
    ap.add_argument("--motion-dim", type=int, default=0, help="width of a separate motion stream (0 = none)")
    ap.add_argument("--feature-dtype", default="float32", choices=["float32", "float16"],
                    help="storage type of the videos, motion features and queries")
    ap.add_argument("--precision", default="fp32")
    ap.add_argument("--flavour", default="mad", choices=["mad", "ego4d"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    cfg = PRESETS[a.config]
    # eval batches (the unit the reference pools over, SURVEY.md §8 A9) must not straddle videos of different ranks:
    # with `queries` per video a multiple of eval_bsz every video holds whole batches
    cfg = cfg.replace(eval_bsz=a.queries, v_motion_feat_dim=a.motion_dim)
    ds = make_dataset(cfg, a.videos, None, a.queries, seed=a.seed, frames_range=tuple(a.frames), motion_dim=a.motion_dim)
    fdt = np.dtype(a.feature_dtype)
    videos = [v.astype(fdt) for v in ds.videos]
    motion = None if ds.motion is None else [m.astype(fdt) for m in ds.motion]
    queries = [dataclasses.replace(q, tokens=q.tokens.astype(fdt), cls=q.cls.astype(fdt)) for q in ds.queries]
    gt = {q.query_id: q.timestamps for q in ds.queries}
    costs = [video_cost(len(v), a.queries, cfg.topk_window) for v in ds.videos]
    mine = lpt_assign(costs, world)[rank]
    eng = ConeEngine(cfg, init_state_dict(cfg, a.seed), device=dev, precision=a.precision, workspace_bytes=4 << 30)
    # one video per step keeps the reference's eval-batch boundaries identical for every sharding
    c = evaluate_dataset(eng, videos, queries, gt, flavour=a.flavour, max_frames_per_step=1, video_ids=mine,
                         motion_videos=motion)
    reduce_counters(c)
    if rank == 0:
        out = {"world": world, "n_queries": int(c.n_queries.item()), "window_recall": c.window_recall().tolist()}
        for m in MODES:
            if a.flavour == "mad":
                out[m] = c.recall_mad(m).tolist()
            else:
                rec, miou = c.recall_ego4d(m)
                out[m] = {"recall": rec.tolist(), "mIoU": miou}
        text = json.dumps(out)
        print(text)
        if a.out:
            with open(a.out, "w") as f:
                f.write(text)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
