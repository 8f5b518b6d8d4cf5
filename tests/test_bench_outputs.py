"""bench.py --dump-outputs: the labels the last timed step returned, written as float32 .npy (a fixed seeded sample of a
large volume), identical from run to run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_keeps_small_arrays_and_samples_large_ones(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_VALUES", 1000)
    small = (torch.arange(600) % 3 == 0).to(torch.uint8).reshape(2, 300)
    big = (torch.arange(5000) % 7 == 0).to(torch.uint8).reshape(5, 10, 100)
    info = bench.dump_outputs(str(tmp_path / "d"), {"small": small, "big": big})
    s = np.load(tmp_path / "d" / "small.npy")
    assert s.dtype == np.float32 and np.array_equal(s, small.float().numpy())
    b = np.load(tmp_path / "d" / "big.npy")
    idx = np.sort(np.random.default_rng(0).integers(0, 5000, 1000))
    assert b.dtype == np.float32 and np.array_equal(b, big.reshape(-1)[idx].float().numpy())
    assert info["arrays"]["big"]["shape"] == [5, 10, 100] and info["arrays"]["big"]["dtype"] == "uint8"
    assert "sample" in info["arrays"]["big"] and "sample" not in info["arrays"]["small"]


def test_bench_rejects_zero_steps():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode != 0 and "--steps" in res.stderr and res.stdout == ""


@pytest.mark.gpu
def test_bench_dump_is_identical_run_to_run(tmp_path):
    runs = []
    for tag in ("a", "b"):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "wide", "--steps", "2", "--warmup", "0",
                              "--no-cpu-baseline", "--no-library-bar", "--dump-outputs", str(tmp_path / tag)],
                             capture_output=True, text=True, timeout=900)
        assert res.returncode == 0, res.stderr[-2000:]
        lines = [l for l in res.stdout.splitlines() if l.strip()]
        assert len(lines) == 1
        d = json.loads(lines[0])
        assert d["steps"] == 2 and os.listdir(tmp_path / tag) == ["labels.npy"]
        runs.append((d, np.load(tmp_path / tag / "labels.npy")))
    (d, a), (_, b) = runs
    entry = d["dump_outputs"]["arrays"]["labels"]
    assert int(np.prod(entry["shape"])) == d["config"]["classes"] * 96 ** 3 and entry["dtype"] == "uint8"
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_MAX_VALUES,) and a.nbytes <= 64 << 20
    assert set(np.unique(a).tolist()) <= {0.0, 1.0} and 0 < a.sum() < a.size
    assert np.array_equal(a, b)
