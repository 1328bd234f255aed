#!/usr/bin/env python
"""The MAD-768 step at longer windows: (max_v_l, max_q_l) = (125, 25), (250, 25), (480, 32), device-resident.
    python profiles/long_window_step.py [--movies 2] [--queries-per-movie 640] [--precision tc] [--out f.json]

For each window shape: the handle's device footprint (cudaMemGetInfo around cone_weights_create plus the first call,
minus what the PyTorch allocator holds: the workspace and the output tensors), the step time (CUDA events around each
step, inputs resident in HBM, several movies cycled) and, in a separate profiled pass, the per-category kernel time
from cone_profile_*.  The card's name and power limit are read in the same run."""
import argparse, json, os, subprocess, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cone_b200 import _lib
from cone_b200.config import MAD768
from cone_b200.engine import ConeEngine, read_profile
from cone_b200.inference import stage_step
from cone_b200.synth import make_dataset
from cone_b200.weights import init_state_dict

ap = argparse.ArgumentParser()
ap.add_argument("--shapes", default="125x25,250x25,480x32")
ap.add_argument("--movies", type=int, default=2)
ap.add_argument("--queries-per-movie", type=int, default=640)
ap.add_argument("--frames", type=int, nargs=2, default=(36000, 54000))
ap.add_argument("--precision", default="tc", choices=["tc", "fp32"])
ap.add_argument("--workspace-gb", type=float, default=16.0)
ap.add_argument("--steps", type=int, default=6)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--out", default="")
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("long_window_step.py measures the GPU path: no CUDA device")
dev = torch.device("cuda:0")
try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:  # the numbers stay valid without it; say that the card's settings were not read
    smi = f"nvidia-smi unavailable ({e})"


def library_bytes_in_use():
    free, total = torch.cuda.mem_get_info(dev)
    return (total - free) - torch.cuda.memory_reserved(dev)


summary = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi": smi, "precision": a.precision, "config": MAD768.name,
           "movies": a.movies, "queries_per_step": a.queries_per_movie, "steps": a.steps, "shapes": {}}
for shape in a.shapes.split(","):
    lv, lt = (int(x) for x in shape.split("x"))
    cfg = MAD768.replace(max_v_l=lv, max_q_l=lt)
    ds = make_dataset(cfg, a.movies, None, a.queries_per_movie, seed=0, frames_range=tuple(a.frames))
    steps = [stage_step(cfg, ds.videos, ds.queries, [v]) for v in range(a.movies)]
    resident = [(s.frames.to(dev), s.qb.to(dev)) for s in steps]
    torch.cuda.synchronize()
    before = library_bytes_in_use()
    eng = ConeEngine(cfg, init_state_dict(cfg, 0), device=dev, precision=a.precision,
                     workspace_bytes=int(a.workspace_gb * (1 << 30)))
    eng.ground(*resident[0])  # the first call in tensor-core mode builds the fp16 weights and position tables
    torch.cuda.synchronize()
    handle_bytes = library_bytes_in_use() - before
    for i in range(a.warmup):
        eng.ground(*resident[i % a.movies])
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    torch.cuda.synchronize()
    _lib.reset_launch_count()
    for i in range(a.steps):
        ev[i][0].record()
        eng.ground(*resident[i % a.movies])
        ev[i][1].record()
    torch.cuda.synchronize()
    launches = _lib.launch_count() // a.steps
    ms = [s.elapsed_time(e) for s, e in ev]
    lib = _lib.load()
    lib.cone_profile_enable(1)
    read_profile()  # clears what was accumulated so far
    for i in range(a.steps):
        eng.ground(*resident[i % a.movies])
    torch.cuda.synchronize()
    prof = read_profile()
    lib.cone_profile_enable(0)
    windows = a.queries_per_movie * cfg.topk_window
    summary["shapes"][shape] = {
        "window_rows": lv + lt, "windows_per_step": windows, "launches_per_step": launches,
        "handle_device_gb": handle_bytes / 1e9, "step_ms_median": float(np.median(ms)), "step_ms_min": float(np.min(ms)),
        "kernel_ms_per_step": {k: v["ms"] / a.steps for k, v in prof.items() if v["launches"]},
    }
    print(shape, json.dumps(summary["shapes"][shape]), flush=True)
    del eng, resident
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
text = json.dumps(summary)
print(text)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(text + "\n")
