"""bench.py output contract, checked on CPU through the reference arm (the only arm that runs without a GPU):
stdout carries exactly ONE JSON line with the keys a caller reads; under torchrun only rank 0 prints; our arm
refuses to run without a CUDA device instead of falling back to anything.  On a GPU: what --dump-outputs writes."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _run(cmd, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run(cmd, cwd=ROOT, env=e, capture_output=True, text=True, timeout=timeout)


def _check_reference_line(stdout):
    lines = [ln for ln in stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["higher_is_better"] is True and d["unit"] == "graphs/s" and d["value"] > 0
    assert d["vs_baseline"] is None
    assert d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    return d


def test_reference_arm_prints_one_json_line():
    r = _run([sys.executable, BENCH, "--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-batch", "4"])
    assert r.returncode == 0, r.stderr[-2000:]
    d = _check_reference_line(r.stdout)
    assert d["n_gpus"] == 1 and d["steps"] == 1


def test_reference_arm_under_torchrun_only_rank0_prints():
    r = _run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
              "--master-port", "29533", BENCH, "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1",
              "--cpu-batch", "4"])
    assert r.returncode == 0, r.stderr[-2000:]
    d = _check_reference_line(r.stdout)
    assert d["n_gpus"] == 2


@pytest.mark.gpu
def test_dump_outputs_repeat_from_run_to_run(cuda_lib, tmp_path):
    """--dump-outputs writes the last timed step's output and gradients as float32 .npy files, 64 MB at most (the output
    rows above 2^22 elements sampled), and two runs with the same arguments write the same arrays."""
    import numpy as np
    args = [sys.executable, BENCH, "--batch", "512", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-e2e",
            "--no-structured", "--no-graph"]
    shapes = {"out": (4194304 // 500, 500), "lin_src.weight.grad": (3000, 1260), "att_src.grad": (1, 6, 500),
              "att_dst.grad": (1, 6, 500), "lin_edge.weight.grad": (3000, 126), "att_edge.grad": (1, 6, 500), "bias.grad": (500,)}
    dumps = []
    for k in range(2):
        r = _run(args + ["--dump-outputs", str(tmp_path / str(k))])
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout)["steps"] == 2
        dumps.append({p.name[:-4]: np.load(p) for p in (tmp_path / str(k)).glob("*.npy")})
    a, b = dumps
    assert {k: v.shape for k, v in a.items()} == shapes
    assert all(v.dtype == np.float32 for v in a.values()) and sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in shapes:
        assert np.isfinite(a[k]).all() and np.abs(a[k]).max() > 0, k
        assert np.abs(a[k] - b[k]).max() <= 1e-6 * np.abs(b[k]).max(), k


def test_our_arm_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = _run([sys.executable, BENCH, "--steps", "1", "--warmup", "1"])
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)
    assert not any(ln.startswith("{") for ln in r.stdout.splitlines())
