"""bench.py contract (CPU side): the reference arm prints ONE JSON line with the agreed keys, and the CUDA arm
refuses to run without a GPU instead of falling back to anything (the product path has no CPU route)."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True,
                          text=True, timeout=timeout)


def test_reference_arm_prints_one_contract_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "mel-frames/sec" and d["unit"] == "mel-frames/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["steps"] == 1 and d["n_gpus"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] == d["value"] and c["sample"]
    # a step is a bounded sample (2 of the 31 Euler intervals), extrapolated to the whole utterance
    assert abs(d["value"] - 937 / (d["ms_per_step"] / 1e3 * 15.5)) / d["value"] < 1e-6


def test_dump_outputs_is_reproducible_and_stays_within_its_budget(tmp_path, monkeypatch):
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    small = torch.arange(1000, dtype=torch.float64).reshape(10, 100)
    big = torch.randn(3, 50_000, generator=torch.Generator().manual_seed(0))
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"big": big, "small": small})
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 200_000
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float32 and np.array_equal(s, small.float().numpy())          # written whole
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and 0 < a.size < big.numel() and np.array_equal(a, b)  # the same sample every run
    assert np.isin(a, big.numpy().ravel()).all()
    r = _run("--impl", "reference", "--dump-outputs", str(tmp_path / "c"))
    assert r.returncode != 0 and not (tmp_path / "c").exists()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_cuda_arm_fails_loudly_without_a_gpu():
    r = _run("--steps", "1", "--warmup", "0", timeout=300)
    assert r.returncode != 0
    assert r.stdout.strip() == ""                       # no JSON line: nothing was measured
    assert "no CUDA device" in r.stderr
