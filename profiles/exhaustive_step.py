#!/usr/bin/env python
"""The pre-filter's speed-up, measured: the MAD-768 step at topk_window = 30 against the same step grounding every
window of the movie (k = num_window(L), CONE's no-pre-filter baseline), device-resident, tensor-core mode.
    python profiles/exhaustive_step.py [--movies 2] [--queries-per-movie 640] [--out f.json]

The two steps alternate in one run (CUDA events around each step, movies cycled); the per-category kernel time comes
from cone_profile_* in a separate pass.  Stage 3 is also timed alone on seeded inputs of 640 queries: both entry points
at N = 150 (30 x 5) and N = 2201 (the shared-memory limit, 2201 windows x 1 slot), and the workspace path at N = 4360
(872 x 5, the longest bench movie) and N = 14 525 (2905 x 5, the stress video).  The card's name, power limit and
maximum SM clock are read in the same run."""
import argparse, json, os, subprocess, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cone_b200 import _lib
from cone_b200.config import MAD768
from cone_b200.engine import ConeEngine, _ptr, _stream, read_profile
from cone_b200.inference import stage_step
from cone_b200.synth import make_dataset
from cone_b200.weights import init_state_dict

ap = argparse.ArgumentParser()
ap.add_argument("--movies", type=int, default=2)
ap.add_argument("--queries-per-movie", type=int, default=640)
ap.add_argument("--frames", type=int, nargs=2, default=(36000, 54000))
ap.add_argument("--workspace-gb", type=float, default=24.0)
ap.add_argument("--steps", type=int, default=3, help="timed steps of each kind")
ap.add_argument("--nms-reps", type=int, default=20)
ap.add_argument("--out", default="")
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("exhaustive_step.py measures the GPU path: no CUDA device")
dev = torch.device("cuda:0")
try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:  # the numbers stay valid without it; say that the card's settings were not read
    smi = f"nvidia-smi unavailable ({e})"

ds = make_dataset(MAD768, a.movies, None, a.queries_per_movie, seed=0, frames_range=tuple(a.frames))
k_all = MAD768.num_window(max(len(v) for v in ds.videos))
steps = [stage_step(MAD768, ds.videos, ds.queries, [v]) for v in range(a.movies)]
resident = [(s.frames.to(dev), s.qb.to(dev)) for s in steps]
sd = init_state_dict(MAD768, 0)
ws = int(a.workspace_gb * (1 << 30))
engines = {"top30": ConeEngine(MAD768, sd, device=dev, precision="tc", workspace_bytes=ws)}
engines["all"] = ConeEngine(MAD768.replace(topk_window=k_all), sd, device=dev, precision="tc", workspace_bytes=ws)
for e in engines.values():
    for r in resident:
        e.ground(*r)
torch.cuda.synchronize()
ms = {n: [] for n in engines}
for i in range(a.steps):  # alternate the two steps
    for n, e in engines.items():
        s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        e.ground(*resident[i % a.movies])
        t.record()
        torch.cuda.synchronize()
        ms[n].append(s.elapsed_time(t))
lib = _lib.load()
kernels = {}
for n, e in engines.items():
    lib.cone_profile_enable(1)
    read_profile()  # clears what was accumulated so far
    e.ground(*resident[0])
    torch.cuda.synchronize()
    kernels[n] = {c: round(v["ms"], 3) for c, v in read_profile().items() if v["launches"]}
    lib.cone_profile_enable(0)


def stage3_ms(eng, k, ns, entry, nq=640):
    """one stage-3 call on seeded inputs of nq queries with k windows of ns slots, CUDA events over nms_reps calls"""
    g = torch.Generator(device=dev).manual_seed(k * ns)
    spans = torch.rand((nq, k, ns, 2), generator=g, device=dev) * 0.9 + 0.05
    prob = torch.round(torch.rand((nq, k, ns), generator=g, device=dev) * 100) / 100
    match = torch.rand((nq, k, ns), generator=g, device=dev) * 2 - 1
    wstart = (torch.arange(k, dtype=torch.int32, device=dev) * 62).repeat(nq, 1)
    wlen = torch.full((nq, k), 125, dtype=torch.int32, device=dev)
    out = torch.zeros((nq, 3, MAD768.max_after_nms, 5), dtype=torch.float64, device=dev)
    cnt = torch.zeros((nq, 3), dtype=torch.int32, device=dev)
    args = (_ptr(spans), _ptr(prob), _ptr(match), _ptr(wstart), _ptr(wlen), nq, k, ns, float(np.float32(MAD768.clip_length)),
            float(MAD768.nms_thd), MAD768.max_before_nms, MAD768.max_after_nms, 0, 1, _ptr(out), _ptr(cnt), None, None)
    if entry == "ex":
        call = lambda: _lib.check(lib.cone_fuse_nms_ex(*args, _stream()), "cone_fuse_nms_ex")
    else:
        wsp, nb = eng._wsargs(lib.cone_fuse_nms_workspace_bytes(nq, k, ns))
        call = lambda: _lib.check(lib.cone_fuse_nms_ws(*args, wsp, nb, _stream()), "cone_fuse_nms_ws")
    call()
    torch.cuda.synchronize()
    s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(a.nms_reps):
        call()
    t.record()
    torch.cuda.synchronize()
    return s.elapsed_time(t) / a.nms_reps


nms = {}
for k, ns, entries in ((30, 5, ("ex", "ws")), (2201, 1, ("ex", "ws")), (872, 5, ("ws",)), (2905, 5, ("ws",))):
    for entry in entries:
        nms[f"N{k * ns}_{entry}"] = round(stage3_ms(engines["top30"], k, ns, entry), 3)

med = {n: float(np.median(v)) for n, v in ms.items()}
summary = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi (name, power limit, max SM clock)": smi, "precision": "tc",
           "config": MAD768.name, "movies": [len(v) for v in ds.videos], "queries_per_step": a.queries_per_movie,
           "topk_all": k_all, "step_ms_median": med, "step_ms_all": ms,
           "exhaustive_over_top30": med["all"] / med["top30"], "kernel_ms_per_step": kernels,
           "stage3_ms_640_queries": nms}
text = json.dumps(summary)
print(text)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(text + "\n")
