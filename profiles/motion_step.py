#!/usr/bin/env python
"""Cost of a separate motion stream on the benchmark's MAD-768 step: the same movies and queries grounded by a
single-stream model (the appearance rows feed Moment-DETR) and by a model that reads a `--motion-dim` motion stream.
    python profiles/motion_step.py [--motion-dim 2304] [--movies 4] [--queries-per-movie 640] [--precision tc] [--out f.json]

device: inputs resident in HBM (several movies cycled, larger than the L2), CUDA events around every step; the two
        models alternate round by round so that drift on a shared machine hits both alike.
e2e:    pinned host inputs -> H2D -> whole path -> D2H of the NMS'd predictions, one step at a time, host clock around
        work that ends in a device synchronise (no copy/compute overlap: the H2D is on the path).
The per-step frame stage (stage 0 + per-frame projections) is also timed alone, because that is where the motion
stream adds its work: an L2 norm and a Dm -> 256 projection of every frame."""
import argparse, json, os, subprocess, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cone_b200.config import MAD768
from cone_b200.engine import ConeEngine
from cone_b200.inference import stage_step
from cone_b200.synth import make_dataset
from cone_b200.weights import init_state_dict

ap = argparse.ArgumentParser()
ap.add_argument("--motion-dim", type=int, default=2304)
ap.add_argument("--movies", type=int, default=4)
ap.add_argument("--queries-per-movie", type=int, default=640)
ap.add_argument("--frames", type=int, nargs=2, default=(36000, 54000))
ap.add_argument("--precision", default="tc", choices=["tc", "fp32"])
ap.add_argument("--steps", type=int, default=12)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--out", default="")
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("motion_step.py measures the GPU path: no CUDA device")
dev = torch.device("cuda:0")

cfg1 = MAD768
cfg2 = MAD768.replace(v_motion_feat_dim=a.motion_dim)
ds = make_dataset(cfg2, a.movies, None, a.queries_per_movie, seed=0, frames_range=tuple(a.frames), motion_dim=a.motion_dim)
engines = {"single": ConeEngine(cfg1, init_state_dict(cfg1, 0), device=dev, precision=a.precision, workspace_bytes=16 << 30),
           "motion": ConeEngine(cfg2, init_state_dict(cfg2, 0), device=dev, precision=a.precision, workspace_bytes=16 << 30)}
host = {"single": [stage_step(cfg1, ds.videos, ds.queries, [v]) for v in range(a.movies)],
        "motion": [stage_step(cfg2, ds.videos, ds.queries, [v], motion_videos=ds.motion) for v in range(a.movies)]}
resident = {k: [(s.frames.to(dev), s.qb.to(dev), s.motion.to(dev) if s.motion is not None else None) for s in v]
            for k, v in host.items()}
torch.cuda.synchronize()


def device_ms(name, what):
    eng, steps = engines[name], resident[name]
    for i in range(a.warmup):
        f, qb, m = steps[i % len(steps)]
        eng.ground(f, qb, motion=m) if what == "step" else eng.video_prepare(f, motion=m)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    torch.cuda.synchronize()
    for i in range(a.steps):
        f, qb, m = steps[i % len(steps)]
        ev[i][0].record()
        eng.ground(f, qb, motion=m) if what == "step" else eng.video_prepare(f, motion=m)
        ev[i][1].record()
    torch.cuda.synchronize()
    return [s.elapsed_time(e) for s, e in ev]


def e2e_ms(name):
    eng, steps = engines[name], host[name]
    out = []
    for i in range(a.warmup + a.steps):
        s = steps[i % len(steps)]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        f = s.frames.to(dev, non_blocking=True)
        m = s.motion.to(dev, non_blocking=True) if s.motion is not None else None
        o = eng.ground(f, s.qb.to(dev), motion=m)
        nms, cnt = o.nms.cpu(), o.nms_count.cpu()  # synchronising D2H of the predictions
        if i >= a.warmup:
            out.append(1e3 * (time.perf_counter() - t0))
    return out


res = {k: {"step_ms": [], "frame_stage_ms": [], "e2e_ms": []} for k in engines}
for r in range(a.rounds):
    for name in (("single", "motion") if r % 2 == 0 else ("motion", "single")):
        res[name]["step_ms"] += device_ms(name, "step")
        res[name]["frame_stage_ms"] += device_ms(name, "prepare")
        res[name]["e2e_ms"] += e2e_ms(name)

try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:  # the numbers stay valid without it; say that the card's settings were not read
    smi = f"nvidia-smi unavailable ({e})"
n_frames = [s.frames.shape[0] for s in host["single"]]
summary = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi": smi, "precision": a.precision, "config": cfg1.name,
           "motion_dim": a.motion_dim, "movies": a.movies, "frames_per_movie": n_frames,
           "queries_per_step": a.queries_per_movie, "steps_per_round": a.steps, "rounds": a.rounds,
           "h2d_mb_per_step": {k: float(np.mean([s.h2d_bytes() for s in v])) / 1e6 for k, v in host.items()}}
for k, v in res.items():
    for m, xs in v.items():
        summary[f"{k}_{m}_median"] = float(np.median(xs))
        summary[f"{k}_{m}_p90"] = float(np.percentile(xs, 90))
for m in ("step_ms", "frame_stage_ms", "e2e_ms"):
    summary[f"extra_{m}_median"] = summary[f"motion_{m}_median"] - summary[f"single_{m}_median"]
text = json.dumps(summary)
print(text)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(text + "\n")
