"""bench.py's contract: the product arm fails loudly without a CUDA device (no CPU path, no JSON line), the reference arm
(`--impl reference`: the unmodified reference's eval_epoch on the host cores, or the CPU oracle port where the reference's
files are not placed) prints exactly ONE JSON line on stdout with the result keys, and `--dump-outputs` writes every field
of a step's output."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True, text=True,
                          timeout=timeout, env=env)


def test_product_arm_fails_loudly_without_a_gpu():
    r = _run("--steps", "1", "--warmup", "0", env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode != 0
    assert "no CPU path" in (r.stdout + r.stderr)
    assert not any(line.strip().startswith("{") for line in r.stdout.splitlines())


def test_reference_arm_prints_one_json_line():
    from oracle import ref_harness as RH
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample-queries", "16")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "grounding_queries_per_sec" and d["unit"] == "queries/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["steps"] == 1 and d["warmup"] == 0
    kind = "reference" if RH.reference_available() else "port"
    assert d["cpu_baseline"]["kind"] == kind and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def _load(path):
    return {f[:-4]: np.load(os.path.join(path, f)) for f in os.listdir(path)}


def test_dump_outputs_writes_every_field_and_samples_rows_past_the_limit(tmp_path):
    from cone_b200.engine import GroundingOutput
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    g = torch.Generator().manual_seed(0)
    nq, k, ns = 50, 4, 5
    out = GroundingOutput(
        ranklist=torch.randint(-1, 90, (nq, 9), dtype=torch.int32, generator=g),
        win_start=torch.randint(0, 1 << 20, (nq, k), dtype=torch.int32, generator=g),
        win_len=torch.randint(0, 125, (nq, k), dtype=torch.int32, generator=g),
        pred_spans=torch.rand((nq, k, ns, 2), generator=g), prob_fg=torch.rand((nq, k, ns), generator=g),
        match=torch.rand((nq, k, ns), generator=g), nms=torch.rand((nq, 3, 5, 5), dtype=torch.float64, generator=g),
        nms_count=torch.randint(0, 6, (nq, 3), dtype=torch.int32, generator=g))
    fields = ("ranklist", "win_start", "win_len", "pred_spans", "prob_fg", "match", "nms", "nms_count")
    bench.dump_outputs(out, str(tmp_path / "all"))
    full = _load(tmp_path / "all")
    assert sorted(full) == sorted(fields)
    for name in fields:
        want = getattr(out, name).numpy()
        assert full[name].dtype == (np.float32 if want.dtype == np.float32 else np.float64), name
        assert np.array_equal(full[name], want), name
    limit = sum(a.nbytes for a in full.values()) // 3
    for d in ("a", "b"):
        bench.dump_outputs(out, str(tmp_path / d), limit=limit)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sorted(a) == sorted(fields + ("query_index",))
    assert sum(x.nbytes for x in a.values()) <= limit
    idx = a["query_index"].astype(np.int64)
    assert 0 < len(idx) < nq and np.all(np.diff(idx) > 0)
    for name in a:
        assert np.array_equal(a[name], b[name]), name  # the same sample every time
        if name != "query_index":
            assert np.array_equal(a[name], full[name][idx]), name
