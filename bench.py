#!/usr/bin/env python
"""Benchmark of the CONE coarse-to-fine grounding path on B200 (BASELINE.json metric: grounding queries/s,
MAD-shape, device-timed).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W     # the reference's own eval_epoch on the box's host cores
    python bench.py --gpus N --scaling strong                 # BASELINE.json configs[3]: fixed MAD-test-scale set, LPT-sharded
    python bench.py --gpus N --workload stress                # BASELINE.json configs[4]: one 10-hour video, queries sharded
    python bench.py --steps K --warmup W --dump-outputs DIR   # also writes the last timed step's outputs as DIR/<name>.npy

A step = one pass of the whole hot path (stages 0-3: adapter + window pre-filter + Moment-DETR on the top-k
windows + proposal matching + fusion/NMS) over one synthetic MAD-shaped movie with all its queries.  Default
(the driver's contract): per-GPU work is fixed as N grows (weak scaling): every rank owns `--movies` movies (its
shard of the movie set); ranks exchange nothing on the data path; the per-query prediction blocks are gathered
ONCE at the end (NCCL all-gather), as north_star places it.  The headline `value` is timed with the library's
per-kernel profiling OFF; the per-kernel table comes from a second pass over the same steps.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=8)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", default="mad768", choices=["mad768", "mad512", "ego4d"])
    p.add_argument("--precision", default=os.environ.get("CONE_BENCH_PRECISION", "tc"), choices=["fp32", "tc"],
                   help="tc: tcgen05 fp16-operand / fp32-accumulate projections (1e-3 class); fp32: CUDA-core parity mode (1e-5)")
    p.add_argument("--movies", type=int, default=8, help="movies resident per GPU (cycled through by the steps)")
    p.add_argument("--queries-per-movie", type=int, default=640)
    p.add_argument("--videos-per-step", type=int, default=1,
                   help="videos batched into one step (short-clip configs: Ego4D clips are 900 frames with ~4.5 queries each)")
    p.add_argument("--frames", type=int, nargs=2, default=None, help="movie length range in frames")
    p.add_argument("--cpu-sample-queries", type=int, default=256)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true", help="skip the end-to-end loop (profiler passes only)")
    p.add_argument("--workspace-gb", type=float, default=24.0)
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                   help="strong: ONE fixed MAD-test-scale set (--set-movies movies of uneven length / query count) "
                        "assigned to the ranks by longest-processing-time, every movie processed once")
    p.add_argument("--set-movies", type=int, default=112)
    p.add_argument("--workload", default="movies", choices=["movies", "stress"],
                   help="stress: one 180 000-frame video replicated on every rank, --stress-queries queries sharded")
    p.add_argument("--stress-queries", type=int, default=10000)
    p.add_argument("--no-parity-pass", action="store_true", help="skip the fp32 parity-mode pass")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last one returned (rank 0) as DIR/<name>.npy, "
                        "so that two builds can be compared output for output on the same seeded inputs")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        p.error("--dump-outputs writes the outputs of this project's path: not available with --impl reference")
    return a


def workload_name(cfg, args, frames):
    return (f"{cfg.name}: synthetic movies of {frames[0]}-{frames[1]} frames x {cfg.v_feat_dim}-d, "
            f"{args.queries_per_movie} queries/movie, window {cfg.max_v_l}, top-{cfg.topk_window} windows, "
            f"nms {cfg.nms_thd}")


def frames_range(cfg, args):
    if args.frames:
        return tuple(args.frames)
    return (36000, 54000) if cfg.name.startswith("mad") else (900, 900)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index
        self.t_begin, self.t_end = 0.0, float("inf")

    def wait_ready(self, timeout=8.0):
        """Block until the first sample has arrived: nvidia-smi's start-up (process spawn, NVML initialisation) must not
        fall into the timed region — on a fresh box it cost several ms per step of an 8-step run."""
        t0 = time.time()
        while not self.rows and time.time() - t0 < timeout and self.proc is not None and self.proc.poll() is None:
            time.sleep(0.01)

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "25"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        """Samples taken DURING the timed region only (between mark_begin and mark_end)."""
        rows = [r for t, r in self.rows if self.t_begin <= t <= self.t_end + 0.03]
        sm = [float(r[0]) for r in rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_flops_per_query(cfg):
    """SURVEY.md §8(d): transformer + heads FLOPs per query, counted as the reference computes them (text and
    video projections once per window)."""
    d, ff, S = cfg.hidden_dim, cfg.dim_feedforward, cfg.max_v_l + cfg.max_q_l
    nq = cfg.num_queries
    vid = cfg.max_v_l * (cfg.v_feat_dim * d + d * d) * 2
    txt = cfg.max_q_l * (cfg.t_feat_dim * d + d * d) * 2
    enc = cfg.enc_layers * (S * (4 * d * d + 2 * d * ff) * 2 + 2 * S * S * d * 2)
    dec = cfg.dec_layers * (S * 2 * d * d * 2 + nq * (6 * d * d + 2 * d * ff) * 2 + 2 * nq * S * d * 2 + 2 * nq * nq * d * 2)
    heads = nq * (2 * d * d + 2 * d + 2 * d) * 2
    return cfg.topk_window * (vid + txt + enc + dec + heads)


def algorithmic_bytes_per_step(cfg, n_frames, n_queries):
    """SURVEY.md §8(d): per video L*Dv*4 + Nq*Dv*4 (stage 0/1 streams the video once), per query the sliced windows
    k*Lv*Dv*4 and its tokens Lt*Dt*4 (proposal ranking re-reads the window tile: 0 extra when fused)."""
    per_video = n_frames * cfg.v_feat_dim * 4 + n_queries * cfg.v_feat_dim * 4
    per_query = cfg.topk_window * cfg.max_v_l * cfg.v_feat_dim * 4 + cfg.max_q_l * cfg.t_feat_dim * 4
    return per_video + n_queries * per_query


def cpu_oracle_sample(cfg, sd, ds, n_queries, threads):
    """The reference's CPU path (oracle port) on a bounded sample: the first movie with its first n queries."""
    import torch
    from oracle import cone_oracle as O
    torch.set_num_threads(threads)
    qs = [q for q in ds.queries if q.video_idx == 0][:n_queries]
    t0 = time.perf_counter()
    O.eval_pipeline(sd, cfg, ds.videos[:1], qs, collect_raw=False)
    dt = time.perf_counter() - t0
    return len(qs) / dt, dt, len(qs)


def reference_sample(cfg, sd, ds, n_queries, threads, model=None):
    """The UNMODIFIED reference's `eval_epoch` (cone/inference.py:227-499: DataLoader + collate + model + Python
    post-processing + metric scripts) on the box's host cores, on a bounded sample: movie 0 with its first n queries.
    Needs the reference's files (oracle/_ref, placed by oracle/vendor_ref.py).  Returns (q/s, seconds, n, model)."""
    import dataclasses
    import torch
    from oracle import ref_harness as RH
    torch.set_num_threads(threads)
    qs = [q for q in ds.queries if q.video_idx == 0][:n_queries]
    sub = dataclasses.replace(ds, videos=ds.videos[:1], queries=qs)
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):  # the reference prints its metric tables: stdout carries only the JSON line
        if model is None:
            model = RH.build_reference_model(cfg, sd)
        res = RH.run_eval_epoch_files(cfg, sub, model, device="cpu")
    return len(qs) / res["seconds"], res["seconds"], len(qs), model


def reference_runnable():
    try:
        from oracle import ref_harness as RH
        return RH.reference_available()
    except Exception:
        return False


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path, all host threads, on our arm's config.
    Each step is a bounded sample of the workload (movie 0 with n of its queries; n is sized from a probe so that the
    whole --steps/--warmup run ends within a few minutes)."""
    import torch
    from cone_b200.config import PRESETS
    from cone_b200.synth import make_dataset
    from cone_b200.weights import init_state_dict
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = PRESETS[args.config]
    fr = frames_range(cfg, args)
    threads = os.cpu_count() or 1
    sd = init_state_dict(cfg, args.seed)
    ds = make_dataset(cfg, 1, None, args.cpu_sample_queries, seed=args.seed, frames_range=fr)
    use_ref = reference_runnable()
    model = None
    if use_ref:
        _, dt, n0, model = reference_sample(cfg, sd, ds, cfg.eval_bsz, threads)  # probe (also warms torch's thread pool)
        rate = n0 / dt
    else:
        rate, dt, n0 = cpu_oracle_sample(cfg, sd, ds, cfg.eval_bsz, threads)
    budget_s = 150.0
    n = int(rate * budget_s / max(args.steps + args.warmup, 1))
    n = max(cfg.eval_bsz, min(args.cpu_sample_queries, (n // cfg.eval_bsz) * cfg.eval_bsz))
    times = []
    for i in range(args.warmup + args.steps):
        if use_ref:
            _, dt, _, model = reference_sample(cfg, sd, ds, n, threads, model)
        else:
            _, dt, _ = cpu_oracle_sample(cfg, sd, ds, n, threads)
        if i >= args.warmup:
            times.append(dt)
    total = float(np.sum(times))
    value = args.steps * n / total
    kind = "reference" if use_ref else "port"
    what = ("the unmodified reference's eval_epoch (cone/inference.py:227-499, from oracle/_ref)" if use_ref
            else "torch-CPU fp32 oracle port (reference files not placed)")
    sample = (f"each step = {what} on 1 movie of {len(ds.videos[0])} frames with {n} of its "
              f"{args.queries_per_movie} queries, torch-CPU fp32, {threads} threads, num_workers=0")
    line = {"impl": "reference", "metric": "grounding_queries_per_sec", "value": value, "unit": "queries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(cfg, args, fr), "device": "cpu", "queries_per_step": n},
            "cpu_baseline": {"value": value, "unit": "queries/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    return 0


def timed_steps(eng, dev_steps, steps, barrier, torch, profile=False):
    """`steps` passes of the path over resident inputs, CUDA events on the launching stream.  Returns (ms, queries,
    last output, per-category profile or None, launches)."""
    from cone_b200 import _lib
    from cone_b200.engine import read_profile
    lib = _lib.load()
    barrier()
    _lib.reset_launch_count()
    if profile:
        lib.cone_profile_enable(1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_queries = 0
    out = None
    ev0.record()
    for i in range(steps):
        out = eng.ground(*dev_steps[i % len(dev_steps)])
        n_queries += out.nms_count.shape[0]
    ev1.record()
    barrier()
    prof = None
    if profile:
        prof = read_profile()
        lib.cone_profile_enable(0)
    return ev0.elapsed_time(ev1), n_queries, out, prof, _lib.launch_count()


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(out, path, limit=DUMP_LIMIT_BYTES):
    """Writes the `GroundingOutput` of one step as `path/<field>.npy`: float32 fields as float32, the fp64 prediction rows
    and the integer fields as float64 (exact).  Every field has one row per query in packed order; when together they
    would exceed `limit` bytes, the same fixed seeded sample of rows is written for all of them, and its row indices as
    `query_index.npy`."""
    import dataclasses
    arrays = {}
    for f in dataclasses.fields(out):
        t = getattr(out, f.name)
        if t is not None:
            a = t.cpu().numpy()
            arrays[f.name] = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
    n = arrays["nms"].shape[0]
    total = sum(a.nbytes for a in arrays.values())
    if total > limit:
        keep = int(n * limit // (total + 8 * n))
        idx = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["query_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from cone_b200.config import PRESETS
    from cone_b200.engine import ConeEngine
    from cone_b200.inference import stage_step
    from cone_b200.sharding import gather_predictions
    from cone_b200.synth import make_dataset
    from cone_b200.weights import init_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: cone_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allreduce(x, op):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=op)
        return float(t.item())

    cfg = PRESETS[args.config]
    if args.workload == "stress":
        return run_stress(args, cfg, world, rank, dev, barrier, allreduce)
    if args.scaling == "strong":
        return run_strong(args, cfg, world, rank, dev, barrier, allreduce)
    fr = frames_range(cfg, args)
    sd = init_state_dict(cfg, args.seed)
    # every rank owns its own shard of the movie set (weak scaling): movie ids rank*M .. rank*M+M-1
    ds = make_dataset(cfg, args.movies, None, args.queries_per_movie, seed=args.seed + 1000 * rank, frames_range=fr,
                      id_offset=rank * args.movies)
    eng = ConeEngine(cfg, sd, device=dev, precision=args.precision, workspace_bytes=int(args.workspace_gb * (1 << 30)))
    vps = max(1, args.videos_per_step)
    groups = [list(range(v, min(v + vps, args.movies))) for v in range(0, args.movies, vps)]
    host_steps = [stage_step(cfg, ds.videos, ds.queries, g) for g in groups]
    dev_steps = [(s.frames.to(dev), s.qb.to(dev)) for s in host_steps]
    # Size the caching allocator once: the movies differ in length, so without this the first timed steps on a longer
    # movie than the warm-up saw call cudaMalloc (a device-synchronising call) between kernels of the timed region
    presize = torch.empty(int(4e9), dtype=torch.uint8, device=dev)
    del presize
    torch.cuda.synchronize()

    # ---- device-timed region: inputs resident in HBM (1.1 GB of movies cycled: larger than the 126 MB L2),
    #      per-kernel profiling OFF ----
    clocks = ClockSampler(local)
    clocks.__enter__()  # started before the warm-up so that its start-up stays outside the timed region
    clocks.wait_ready()
    for i in range(args.warmup):
        eng.ground(*dev_steps[i % len(dev_steps)])
    try:
        clocks.mark_begin()
        ms, n_queries, out, _, launches = timed_steps(eng, dev_steps, args.steps, barrier, torch)
        clocks.mark_end()
    finally:
        clocks.__exit__(None, None, None)
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    ms_max = allreduce(ms, dist.ReduceOp.MAX if world > 1 else None)
    nq_all = allreduce(n_queries, dist.ReduceOp.SUM if world > 1 else None)
    value = nq_all / (ms_max / 1e3)
    if args.no_e2e:
        if rank == 0:
            emit({"metric": "grounding_queries_per_sec", "value": value, "unit": "queries/s", "n_gpus": world,
                  "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "note": "profiler pass: no e2e"})
        if world > 1:
            dist.destroy_process_group()
        return 0
    # ---- second pass over the same steps with the library's per-kernel events on: the stage table ----
    ms_prof, _, out, prof, _ = timed_steps(eng, dev_steps, args.steps, barrier, torch, profile=True)

    # ---- end to end: pinned host inputs -> H2D -> path -> D2H of the predictions; across ranks the prediction blocks
    #      are gathered ONCE after the last step (north_star: "NCCL ... only to gather per-query top-k predictions") ----
    # Every step's inputs are copied from pinned host memory inside the timed region and every step's result is
    # read back to the host; the copy of step i+1 is issued on a side stream so that it overlaps step i's kernels
    # (what a serving loop does), and the host reads are asynchronous into pinned buffers, fenced at the end.
    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream()
    max_frames = max(s.frames.shape[0] for s in host_steps)
    fbuf = [torch.empty((max_frames, cfg.v_feat_dim), dtype=torch.float32, device=dev) for _ in range(2)]
    consumed = [None, None]  # event recorded on the main stream when the kernels reading fbuf[slot] have been queued
    import dataclasses
    same_shapes = all(all(getattr(s.qb, f.name).shape == getattr(host_steps[0].qb, f.name).shape
                          for f in dataclasses.fields(s.qb) if isinstance(getattr(s.qb, f.name), torch.Tensor))
                      for s in host_steps)
    qbuf = [host_steps[0].qb.to(dev, non_blocking=False) for _ in range(2)] if same_shapes else None

    def prefetch(i):
        s = host_steps[i % len(host_steps)]
        slot = i % 2
        with torch.cuda.stream(copy_stream):
            if consumed[slot] is not None:
                copy_stream.wait_event(consumed[slot])
            frames_d = fbuf[slot][: s.frames.shape[0]]
            frames_d.copy_(s.frames, non_blocking=True)
            if qbuf is None:
                qb = s.qb.to(dev)
            else:
                dst, upd = qbuf[slot], {}
                for f in dataclasses.fields(s.qb):
                    t = getattr(s.qb, f.name)
                    if isinstance(t, torch.Tensor):
                        getattr(dst, f.name).copy_(t, non_blocking=True)
                        upd[f.name] = getattr(dst, f.name)
                qb = dataclasses.replace(s.qb, **upd)  # host metadata of this step, device tensors of the slot
        return s, frames_d, qb

    # pinned landing buffers for every step's result, allocated outside the timed region (cudaHostAlloc is slow)
    probe = eng.ground(*dev_steps[0])
    pinned = [(torch.empty(tuple(probe.nms.shape), dtype=probe.nms.dtype, pin_memory=True),
               torch.empty(tuple(probe.nms_count.shape), dtype=probe.nms_count.dtype, pin_memory=True))
              for _ in range(args.steps)]
    # device-side accumulation of the per-step blocks for the single end-of-run gather
    dev_blocks = [(torch.empty_like(probe.nms), torch.empty_like(probe.nms_count)) for _ in range(args.steps)] if world > 1 else None
    del probe
    barrier()
    t0 = time.perf_counter()
    h2d = d2h = 0
    host_out = []
    nxt = prefetch(0)
    for i in range(args.steps):
        s, frames_d, qb = nxt
        main.wait_stream(copy_stream)
        if qbuf is None:
            qb.record_stream(main)
        if i + 1 < args.steps:
            nxt = prefetch(i + 1)
        out_i = eng.ground(frames_d, qb)
        consumed[i % 2] = torch.cuda.Event()
        consumed[i % 2].record(main)
        nms_h, cnt_h = pinned[i]
        nms_h.copy_(out_i.nms, non_blocking=True)  # device->host read of the step's result
        cnt_h.copy_(out_i.nms_count, non_blocking=True)
        if dev_blocks is not None:
            dev_blocks[i][0].copy_(out_i.nms)
            dev_blocks[i][1].copy_(out_i.nms_count)
        host_out.append((nms_h, cnt_h))
        h2d += s.h2d_bytes()
        d2h += nms_h.numel() * 8 + cnt_h.numel() * 4
    gathered = 0
    if world > 1:  # ONE gather of all the steps' prediction blocks, inside the timed region
        allnms = torch.cat([b[0] for b in dev_blocks])
        allcnt = torch.cat([b[1] for b in dev_blocks])
        g_nms, g_cnt = gather_predictions(allnms, allcnt, equal_shards=True)
        gathered = int(g_nms.shape[0])
    barrier()
    e2e_s = time.perf_counter() - t0
    assert all(int(c.sum()) > 0 for _, c in host_out)
    e2e_value = nq_all / allreduce(e2e_s, dist.ReduceOp.MAX if world > 1 else None)

    # ---- fp32 parity mode on the same steps (the mode that meets 1e-5 against the oracle everywhere) ----
    parity = None
    if args.precision == "tc" and not args.no_parity_pass:
        del eng
        torch.cuda.empty_cache()
        eng32 = ConeEngine(cfg, sd, device=dev, precision="fp32", workspace_bytes=int(args.workspace_gb * (1 << 30)))
        eng32.ground(*dev_steps[0])
        k32 = min(3, args.steps)
        ms32, nq32, _, _, _ = timed_steps(eng32, dev_steps, k32, barrier, torch)
        ms32_max = allreduce(ms32, dist.ReduceOp.MAX if world > 1 else None)
        nq32_all = allreduce(nq32, dist.ReduceOp.SUM if world > 1 else None)
        parity = {"precision": "fp32", "dtype": "f32", "value": nq32_all / (ms32_max / 1e3), "unit": "queries/s",
                  "steps": k32, "ms_per_step": ms32_max / k32,
                  "note": "every GEMM on the fp32 CUDA cores: 1e-5 against the reference everywhere (tests/test_gpu_parity.py)"}
        del eng32

    if rank == 0:
        peaks = load_peaks()
        line = {"metric": "grounding_queries_per_sec", "value": value, "unit": "queries/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "f16",
                "data": "synthetic",
                "config": {"workload": workload_name(cfg, args, fr), "movies_per_gpu": args.movies,
                           "queries_per_step": args.queries_per_movie * vps, "videos_per_step": vps, "precision": args.precision,
                           "l2": "inputs larger than L2: steps cycle through %d movies (%.2f GB) resident in HBM" %
                                 (args.movies, sum(v.nbytes for v in ds.videos) / 1e9),
                           "parallelism": f"movie-sharded x{world}, one all-gather of the per-query predictions at the end",
                           "profiling": "off in the timed region (stage table from a second pass)"},
                "clocks": clocks.summary(), "gpu_launches": int(launches),
                "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": h2d // args.steps,
                        "d2h_bytes_per_step": d2h // args.steps, "gathered_queries": gathered}}
        if parity:
            line["parity_mode"] = parity
        n_frames_t = float(sum(host_steps[i % len(host_steps)].frames.shape[0] for i in range(args.steps)))
        alg_bytes = algorithmic_bytes_per_step(cfg, n_frames_t / args.steps, nq_all / world / args.steps)
        line["roofline"] = roofline_entry(prof, peaks, algorithmic_flops_per_query(cfg), alg_bytes, args, cfg,
                                          ms_max / args.steps, nq_all / world / args.steps)
        if prof:
            # proposal ranking (A9): the kernel reads the rows between the earliest start and the latest end of a
            # window's proposals ONCE (span_mean_pool_window): distinct rows x Dv x 4, from the last step's own spans
            sp, wl = out.pred_spans.float(), out.win_len.float()[:, :, None]
            st = torch.clamp(torch.floor((sp[..., 0] - 0.5 * sp[..., 1]) * wl), min=0)
            en = torch.minimum(torch.ceil((sp[..., 0] + 0.5 * sp[..., 1]) * wl), wl)
            distinct = torch.clamp(en.max(dim=2).values - st.min(dim=2).values, min=0)
            if "span_pool" in prof:
                prof["span_pool"]["bytes"] = float(distinct.sum().item()) * cfg.v_feat_dim * 4.0 * args.steps
            # window pre-filter (A3): one (frame, query) score each; the rank-list kernel reads every score once
            n_scores = float(sum(host_steps[i % len(host_steps)].qb.total_scores for i in range(args.steps)))
            if "frame_scores" in prof:
                prof["frame_scores"]["flops"] = 2.0 * cfg.v_feat_dim * n_scores
                prof["frame_scores"]["bytes"] = 4.0 * (n_scores + cfg.v_feat_dim * (n_frames_t + nq_all / world))
            if "window_ranklist" in prof:
                prof["window_ranklist"]["bytes"] = 4.0 * n_scores
            line["stages"] = stage_table(prof, peaks, args.steps)
            line["stages"]["_profiled_ms_per_step"] = round(ms_prof / args.steps, 3)
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            if reference_runnable():
                n_s = min(args.cpu_sample_queries, 64)
                qps, dt, n, _ = reference_sample(cfg, sd, ds, n_s, threads)
                line["cpu_baseline"] = {"value": qps, "unit": "queries/s", "cores": threads, "kind": "reference",
                                        "sample": f"the unmodified reference's eval_epoch (oracle/_ref) on movie 0 "
                                                  f"({len(ds.videos[0])} frames) with {n} of its {args.queries_per_movie} "
                                                  f"queries, torch-CPU fp32, num_workers=0, {dt:.1f} s"}
            else:
                qps, dt, n = cpu_oracle_sample(cfg, sd, ds, args.cpu_sample_queries, threads)
                line["cpu_baseline"] = {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
                                        "sample": f"stages 0-3 on movie 0 ({len(ds.videos[0])} frames) with {n} of its "
                                                  f"{args.queries_per_movie} queries, torch-CPU fp32 oracle port, {dt:.1f} s"}
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_strong(args, cfg, world, rank, dev, barrier, allreduce):
    """BASELINE.json configs[3]: ONE fixed MAD-test-scale synthetic set (default 112 movies of 36-54 k frames with
    uneven query counts, ~72 k queries), whole movies assigned to ranks by longest-processing-time on
    cost = alpha L + beta Nq k (sharding.lpt_assign), every movie processed once, predictions gathered once at the end.
    Reports total queries / max-over-ranks time, per-rank busy time and the imbalance."""
    import torch
    import torch.distributed as dist
    from cone_b200.engine import ConeEngine
    from cone_b200.inference import stage_step
    from cone_b200.sharding import gather_predictions, lpt_assign, video_cost
    from cone_b200.synth import make_dataset
    from cone_b200.weights import init_state_dict
    fr = frames_range(cfg, args)
    sd = init_state_dict(cfg, args.seed)
    rng = np.random.default_rng(args.seed + 77)
    lens = [int(x) for x in rng.integers(fr[0], fr[1] + 1, size=args.set_movies)]
    nqs = [int(x) for x in rng.integers(args.queries_per_movie // 2, args.queries_per_movie * 3 // 2 + 1, size=args.set_movies)]
    costs = [video_cost(L, n, cfg.topk_window) for L, n in zip(lens, nqs)]
    mine = lpt_assign(costs, world)[rank]
    eng = ConeEngine(cfg, sd, device=dev, precision=args.precision, workspace_bytes=int(args.workspace_gb * (1 << 30)))
    # each rank synthesises only its own movies (seeded by movie id: the set is the same whatever the world size)
    host_steps = []
    for m in mine:
        ds = make_dataset(cfg, 1, [lens[m]], [nqs[m]], seed=args.seed + 10007 * (m + 1), id_offset=m)
        host_steps.append(stage_step(cfg, ds.videos, ds.queries, [0]))
    presize = torch.empty(int(6e9), dtype=torch.uint8, device=dev)
    del presize
    for s in host_steps[: min(2, len(host_steps))]:  # warm-up
        eng.ground(s.frames.to(dev), s.qb.to(dev))
    barrier()
    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    outs = []
    nxt = None
    with torch.cuda.stream(copy_stream):
        if host_steps:
            nxt = (host_steps[0].frames.to(dev, non_blocking=True), host_steps[0].qb.to(dev))
    for i, s in enumerate(host_steps):
        main.wait_stream(copy_stream)
        frames_d, qb = nxt
        frames_d.record_stream(main)
        qb.record_stream(main)
        if i + 1 < len(host_steps):
            with torch.cuda.stream(copy_stream):
                nxt = (host_steps[i + 1].frames.to(dev, non_blocking=True), host_steps[i + 1].qb.to(dev))
        o = eng.ground(frames_d, qb)
        outs.append((o.nms, o.nms_count))
    ev1.record()
    torch.cuda.synchronize()
    busy_ms = ev0.elapsed_time(ev1)
    nms = torch.cat([o[0] for o in outs]) if outs else torch.zeros((0, 3, cfg.max_after_nms, 5), dtype=torch.float64, device=dev)
    cnt = torch.cat([o[1] for o in outs]) if outs else torch.zeros((0, 3), dtype=torch.int32, device=dev)
    g_nms, g_cnt = gather_predictions(nms, cnt)  # once, at the end
    host_nms = g_nms.cpu() if rank == 0 else None
    barrier()
    wall = time.perf_counter() - t0
    if args.dump_outputs and rank == 0 and host_steps:
        dump_outputs(o, args.dump_outputs)
    wall_max = allreduce(wall, dist.ReduceOp.MAX if world > 1 else None)
    busy = torch.zeros(world, dtype=torch.float64, device=dev)
    busy[rank] = busy_ms
    if world > 1:
        dist.all_reduce(busy)
    nq_all = sum(nqs)
    if rank == 0:
        b = busy.cpu().numpy()
        assert host_nms.shape[0] == nq_all, (host_nms.shape, nq_all)
        emit({"metric": "grounding_queries_per_sec", "value": nq_all / wall_max, "unit": "queries/s", "n_gpus": world,
              "steps": max(len(x) for x in lpt_assign(costs, world)), "warmup": 2, "ms_per_step": 1e3 * wall_max / max(len(mine), 1),
              "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16" if args.precision == "tc" else "f32",
              "data": "synthetic",
              "config": {"workload": f"{cfg.name}: fixed set of {args.set_movies} movies ({sum(lens)} frames, {nq_all} queries), "
                                     f"LPT-sharded by movie, host inputs, one all-gather at the end", "precision": args.precision},
              "e2e": {"value": nq_all / wall_max, "unit": "queries/s", "h2d_bytes_per_step": int(sum(s.h2d_bytes() for s in host_steps) / max(len(host_steps), 1)),
                      "d2h_bytes_per_step": int(host_nms.numel() * 8 / max(len(host_steps), 1))},
              "strong": {"wall_s": wall_max, "rank_busy_ms": [round(float(x), 1) for x in b],
                         "imbalance": float(b.max() / b.mean()) if b.mean() > 0 else None,
                         "movies_per_rank": [len(x) for x in lpt_assign(costs, world)]}})
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_stress(args, cfg, world, rank, dev, barrier, allreduce):
    """BASELINE.json configs[4]: one 10-hour video (180 000 frames at 5 fps) replicated on every rank, its queries
    sharded in whole eval batches (sharding.shard_queries).  Stage 0 runs once per rank; the queries go through in
    steps of --queries-per-movie."""
    import torch
    import torch.distributed as dist
    from cone_b200.engine import ConeEngine, pack_queries
    from cone_b200.sharding import gather_predictions, shard_queries
    from cone_b200.synth import make_dataset
    from cone_b200.weights import init_state_dict
    sd = init_state_dict(cfg, args.seed)
    L = 180000
    ds = make_dataset(cfg, 1, [L], args.stress_queries, seed=args.seed + 5)
    mine = shard_queries(list(enumerate(ds.queries)), world, rank, eval_bsz=cfg.eval_bsz)
    eng = ConeEngine(cfg, sd, device=dev, precision=args.precision, workspace_bytes=int(args.workspace_gb * (1 << 30)))
    frames = torch.from_numpy(ds.videos[0]).pin_memory()
    chunk = args.queries_per_movie
    qbs = []
    for c0 in range(0, len(mine), chunk):
        part = mine[c0:c0 + chunk]
        qbs.append(pack_queries(cfg, [L], [q for _, q in part], dataset_indices=[i for i, _ in part]).pin())
    barrier()
    frames_d = frames.to(dev)
    prepared = eng.video_prepare(frames_d)
    if qbs:
        eng.ground(frames_d, qbs[0].to(dev), prepared=prepared)  # warm-up
    barrier()
    t0 = time.perf_counter()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    frames_d = frames.to(dev, non_blocking=True)  # H2D of the 553 MB video inside the timed region
    prepared = eng.video_prepare(frames_d)
    outs = []
    for qb in qbs:
        o = eng.ground(frames_d, qb.to(dev), prepared=prepared)
        outs.append((o.nms, o.nms_count))
    ev1.record()
    nms, cnt = torch.cat([o[0] for o in outs]), torch.cat([o[1] for o in outs])
    g_nms, _ = gather_predictions(nms, cnt)
    host = g_nms.cpu() if rank == 0 else None
    barrier()
    wall_max = allreduce(time.perf_counter() - t0, dist.ReduceOp.MAX if world > 1 else None)
    dev_ms = allreduce(ev0.elapsed_time(ev1), dist.ReduceOp.MAX if world > 1 else None)
    if args.dump_outputs and rank == 0 and qbs:
        dump_outputs(o, args.dump_outputs)
    if rank == 0:
        nq_all = len(ds.queries)
        assert host.shape[0] == nq_all
        emit({"metric": "grounding_queries_per_sec", "value": nq_all / (dev_ms / 1e3), "unit": "queries/s", "n_gpus": world,
              "steps": len(qbs), "warmup": 1, "ms_per_step": dev_ms / max(len(qbs), 1), "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None, "dtype": "f16" if args.precision == "tc" else "f32", "data": "synthetic",
              "config": {"workload": f"{cfg.name} stress: one {L}-frame video x {nq_all} queries ({cfg.num_window(L)} windows "
                                     f"each), video replicated, queries sharded x{world}", "precision": args.precision},
              "e2e": {"value": nq_all / wall_max, "unit": "queries/s", "h2d_bytes_per_step": int((frames.numel() * 4 + sum(q.h2d_bytes() for q in qbs)) / max(len(qbs), 1)),
                      "d2h_bytes_per_step": int(host.numel() * 8 / max(len(qbs), 1))}})
    if world > 1:
        dist.destroy_process_group()
    return 0


def load_peaks():
    """Roofline denominators: MEASURED_PEAKS.json (driver-written) or the fallback B200_PROFILING.md states."""
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        src = "measured (MEASURED_PEAKS.json)"
    except Exception:
        pk, src = {}, "fallback (B200_PROFILING.md: 6.65 TB/s copy, 1.59 PFLOP/s burst / ~1.4 sustained)"
    return {"hbm_gbs": float(pk.get("hbm_gbs", 6650.0)),
            "tflops": float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops", 1400.0))), "source": src}


def load_traffic():
    """DRAM bytes per launch / per step from the committed ncu launch list of this same command
    (profiles/r02_traffic.json, written by profiles/summarize_step.py --traffic); {} when not captured."""
    for name in ("r02_traffic.json",):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", name)))
        except Exception:
            pass
    return {}


def roofline_entry(prof, peaks, flops_per_query, alg_bytes_step, args, cfg, ms_step, queries_step):
    """SURVEY.md §8(d).  The step is TENSOR-bound (K4, the transformer, carries 99 % of the FLOPs).
    * `achieved` / `frac`: the dominant kernel (largest share of the step in the per-kernel pass): ALGORITHMIC FLOPs of
      its launches (2 M N K of the fp32 problem: split GEMMs counted once) / their summed duration, against the
      sustained cuBLAS bf16 peak of MEASURED_PEAKS.json;
    * `step`: whole-step algorithmic FLOP/s (21.05 GFLOP/query x queries / step time, the reference's count) and whole-
      step algorithmic bytes (slicing 11.52 MB/query + one movie + tokens) against the copy peak;
    * `traffic` / `traffic_ratio`: DRAM bytes from the committed ncu capture of this command, per launch of the
      dominant kernel and per step, the latter divided by the algorithmic bytes (wasted round trips)."""
    tr = load_traffic()
    step_tf = flops_per_query * queries_step / (ms_step * 1e-3) / 1e12
    step = {"algorithmic_tflops": step_tf, "frac_of_tensor_peak": step_tf / peaks["tflops"],
            "algorithmic_gflop_per_query": flops_per_query / 1e9,
            "algorithmic_bytes_per_step": alg_bytes_step,
            "algorithmic_gbs": alg_bytes_step / (ms_step * 1e-3) / 1e9,
            "frac_of_hbm_peak": alg_bytes_step / (ms_step * 1e-3) / 1e9 / peaks["hbm_gbs"],
            "traffic_bytes_per_step": tr.get("step_dram_bytes"),
            "traffic_ratio": (tr["step_dram_bytes"] / alg_bytes_step) if tr.get("step_dram_bytes") else None}
    detail = None
    if prof and prof.get("enc_tail_gather", {}).get("launches"):
        # the fused encoder tail runs twice per step: on layer 0 it also does the window slicing (its residual rows arrive by
        # TMA gather4 from the per-frame / per-token tables), on layer 1 its residual rows are dense.  One kernel: the roofline
        # entry is the sum of both; the two forms are listed under `detail`
        a, b = prof.get("enc_tail", {"ms": 0, "launches": 0, "flops": 0, "bytes": 0}), prof["enc_tail_gather"]
        detail = {}
        for name, v in (("layer 1: dense residual rows", a), ("layer 0: + window slicing by TMA gather4", b)):
            if v["launches"]:
                tfl = v["flops"] / (v["ms"] * 1e-3) / 1e12
                detail[name] = {"avg_launch_ms": v["ms"] / v["launches"], "TFLOPs": tfl, "frac": tfl / peaks["tflops"]}
        prof = dict(prof)
        prof["enc_tail"] = {k: a[k] + b[k] for k in ("ms", "launches", "flops", "bytes")}
        del prof["enc_tail_gather"]
    cands = [k for k in ("enc_tail", "gemm_tc", "gemm_fp32", "enc_attention") if prof and k in prof and prof[k]["launches"]]
    if not cands:
        return {"bound": "tensor", "achieved": None, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": None,
                "traffic": None, "step": step, "note": "per-kernel profile unavailable"}
    key = max(cands, key=lambda k: prof[k]["ms"])
    p = prof[key]
    sec = p["ms"] * 1e-3
    tf = p["flops"] / sec / 1e12
    total = max(sum(v["ms"] for v in prof.values()), 1e-9)
    ent = {"bound": "tensor", "kernel": key, "achieved": tf, "peak": peaks["tflops"], "unit": "TFLOP/s",
           "frac": tf / peaks["tflops"], "launches": p["launches"], "avg_launch_ms": p["ms"] / p["launches"],
           "share_of_step": p["ms"] / total, "peak_source": peaks["source"],
           "declared_hbm_gbs": p["bytes"] / sec / 1e9,
           "traffic": (tr.get("kernels", {}).get(key, {}) or {}).get("dram_bytes_per_launch"),
           "step": step}
    if detail and key == "enc_tail":
        ent["detail"] = detail
    if key == "gemm_fp32":
        fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12
        ent.update(bound="fp32", peak=fp32_peak, frac=tf / fp32_peak,
                   peak_source="nominal fp32 FMA rate (no measured fp32 peak in MEASURED_PEAKS.json)")
    return ent


def stage_table(prof, peaks, steps):
    """Per kernel category: ms/step and achieved GB/s / TFLOP/s from the algorithmic work the launches declared."""
    out = {}
    for k, v in prof.items():
        if not v["launches"]:
            continue
        sec = v["ms"] * 1e-3
        e = {"ms": round(v["ms"] / steps, 3), "launches": v["launches"] // steps}
        if v["bytes"]:
            e["GBps"] = round(v["bytes"] / sec / 1e9, 1)
            e["hbm_frac"] = round(v["bytes"] / sec / 1e9 / peaks["hbm_gbs"], 3)
        if v["flops"]:
            e["TFLOPs"] = round(v["flops"] / sec / 1e12, 2)
        out[k] = e
    return out


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, written to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


if __name__ == "__main__":
    a = parse_args()
    # native libraries (NCCL's version banner, driver notices) write to fd 1: keep stdout for the JSON line only
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    sys.exit(run_reference(a) if a.impl == "reference" else run_ours(a))
