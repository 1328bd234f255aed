#!/usr/bin/env python
"""fp16 against fp32 feature storage on the benchmark's MAD-768 step, without and with a separate motion stream.
    python profiles/half_features_step.py [--motion-dim 2304] [--movies 4] [--queries-per-movie 640] [--precision tc] [--out f.json]

The fp32 variant runs on the fp16 values upcast (the features are drawn once and rounded to fp16), so the two storage
types hand the library the same numbers and their outputs must be bitwise equal: every field of every step is compared.
device: inputs resident in HBM (several movies cycled, larger than the L2), CUDA events around every step.
e2e:    pinned host inputs -> H2D -> whole path -> D2H of the NMS'd predictions, one step at a time, host clock around
        work that ends in a device synchronise (no copy/compute overlap: the H2D is on the path).
The four variants alternate round by round, in rotating order, so that drift on a shared machine hits all alike."""
import argparse, dataclasses, json, os, subprocess, sys, time
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
    raise SystemExit("half_features_step.py measures the GPU path: no CUDA device")
dev = torch.device("cuda:0")

cfg1 = MAD768
cfg2 = MAD768.replace(v_motion_feat_dim=a.motion_dim)
ds = make_dataset(cfg2, a.movies, None, a.queries_per_movie, seed=0, frames_range=tuple(a.frames), motion_dim=a.motion_dim)
feats = {}
for dt in (np.float16, np.float32):  # fp16 rounding first; the fp32 variant holds the same values
    cast = lambda x: x.astype(np.float16).astype(dt)
    feats[np.dtype(dt).name] = ([cast(v) for v in ds.videos], [cast(m) for m in ds.motion],
                                [dataclasses.replace(q, tokens=cast(q.tokens), cls=cast(q.cls)) for q in ds.queries])
engines = {"single": ConeEngine(cfg1, init_state_dict(cfg1, 0), device=dev, precision=a.precision, workspace_bytes=16 << 30),
           "motion": ConeEngine(cfg2, init_state_dict(cfg2, 0), device=dev, precision=a.precision, workspace_bytes=16 << 30)}
VARIANTS = [(m, s) for m in ("single", "motion") for s in ("float32", "float16")]
host = {}
for m, s in VARIANTS:
    videos, motion, queries = feats[s]
    cfg = cfg1 if m == "single" else cfg2
    host[m, s] = [stage_step(cfg, videos, queries, [v], motion_videos=motion if m == "motion" else None)
                  for v in range(a.movies)]
resident = {k: [(s.frames.to(dev), s.qb.to(dev), s.motion.to(dev) if s.motion is not None else None) for s in v]
            for k, v in host.items()}
torch.cuda.synchronize()

# bitwise equality of the outputs of the two storage types, every step, every field
mismatch = []
for m in ("single", "motion"):
    for i in range(a.movies):
        o = [engines[m].ground(*resident[m, s][i][:2], want_rows=True, motion=resident[m, s][i][2])
             for s in ("float32", "float16")]
        for f in dataclasses.fields(o[0]):
            x, y = getattr(o[0], f.name), getattr(o[1], f.name)
            if not ((x is None and y is None) or (x is not None and y is not None and torch.equal(x, y))):
                mismatch.append(f"{m}/movie{i}/{f.name}")
torch.cuda.synchronize()
del o


def device_ms(key):
    eng, steps = engines[key[0]], resident[key]
    for i in range(a.warmup):
        f, qb, m = steps[i % len(steps)]
        eng.ground(f, qb, motion=m)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    torch.cuda.synchronize()
    for i in range(a.steps):
        f, qb, m = steps[i % len(steps)]
        ev[i][0].record()
        eng.ground(f, qb, motion=m)
        ev[i][1].record()
    torch.cuda.synchronize()
    return [s.elapsed_time(e) for s, e in ev]


def e2e_ms(key):
    eng, steps = engines[key[0]], host[key]
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


res = {k: {"step_ms": [], "e2e_ms": []} for k in VARIANTS}
for r in range(a.rounds):
    for j in range(len(VARIANTS)):
        k = VARIANTS[(j + r) % len(VARIANTS)]
        res[k]["step_ms"] += device_ms(k)
        res[k]["e2e_ms"] += e2e_ms(k)

try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:  # the numbers stay valid without it; say that the card's settings were not read
    smi = f"nvidia-smi unavailable ({e})"
summary = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi": smi, "precision": a.precision, "config": cfg1.name,
           "motion_dim": a.motion_dim, "movies": a.movies, "frames_per_movie": [len(v) for v in ds.videos],
           "queries_per_step": a.queries_per_movie, "steps_per_round": a.steps, "rounds": a.rounds,
           "outputs_bitwise_equal": not mismatch, "mismatches": mismatch[:20]}
for (m, s), v in res.items():
    summary[f"{m}_{s}_h2d_mb_per_step"] = float(np.mean([st.h2d_bytes() for st in host[m, s]])) / 1e6
    for name, xs in v.items():
        summary[f"{m}_{s}_{name}_median"] = float(np.median(xs))
        summary[f"{m}_{s}_{name}_p90"] = float(np.percentile(xs, 90))
text = json.dumps(summary)
print(text)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(text + "\n")
if mismatch:
    raise SystemExit(f"fp16 and fp32 storage gave different outputs: {mismatch[:5]}")
