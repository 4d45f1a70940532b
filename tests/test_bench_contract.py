"""bench.py prints one JSON line with the contract's keys.  On CPU only the
reference arm can run (the product arm needs a GPU and must refuse without one)."""
import json
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from conftest import ROOT, TOL
from oracle import generators as G
from oracle import ref_port as P


def _run(*args):
    return subprocess.run([sys.executable, "bench.py", *args], cwd=ROOT, capture_output=True, text=True, timeout=600)


def test_reference_arm_json_line():
    r = _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--batch", "200000")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "matrices/s" and d["higher_is_better"] is True
    assert d["metric"] == "batched sym-solve matrices/sec" and d["vs_baseline"] is None and d["dtype"] == "f32"
    assert d["steps"] == 2 and d["value"] > 0 and "workload" in d["config"]
    base = d["cpu_baseline"]
    # the reference's own code when it is installed (oracle/load_reference.py), else the pinned port
    assert base["kind"] in ("reference", "port") and base["cores"] >= 1 and base["value"] == d["value"] and "sample" in base
    assert d["e2e"] == {"value": d["value"], "unit": "matrices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_product_arm_refuses_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = _run("--steps", "1", "--warmup", "3", "--batch", "1000")
    assert r.returncode != 0
    assert "CUDA" in (r.stderr + r.stdout)


def test_arguments_are_checked_before_any_work():
    r = _run("--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr
    r = _run("--impl", "reference", "--dump-outputs", "unused")
    assert r.returncode == 2 and "--dump-outputs" in r.stderr


def test_dump_output_keeps_a_seeded_sample_of_rows(tmp_path):
    out = torch.arange(1000 * 3, dtype=torch.float64).view(1000, 3)
    bench.dump_output(out, str(tmp_path / "whole.npy"), 1 << 20)
    assert np.array_equal(np.load(tmp_path / "whole.npy"), out.numpy())
    bench.dump_output(out, str(tmp_path / "a.npy"), 100 * 3 * 8)
    bench.dump_output(out, str(tmp_path / "b.npy"), 100 * 3 * 8)
    a = np.load(tmp_path / "a.npy")
    assert a.dtype == np.float64 and a.shape == (100, 3)
    assert np.array_equal(a, np.load(tmp_path / "b.npy"))        # the same rows on every run
    rows = a[:, 0] / 3
    assert np.all(np.diff(rows) > 0)                              # distinct rows, in ascending order
    assert np.array_equal(a, out.numpy()[rows.astype(np.int64)])


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
    batch, steps, warmup = 200_000, 5, 3
    r = _run("--steps", str(steps), "--warmup", str(warmup), "--batch", str(batch), "--no-cpu", "--no-e2e",
             "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == steps and d["gpu_launches"] == steps    # 3x3 solve: one launch per step
    got = np.load(tmp_path / "sym_solve3.npy")
    assert got.dtype == np.float32 and got.shape == (batch, 3)
    nsets = bench.operand_set_count(batch * bench.algorithmic_bytes("sym_solve", 3, 4))
    assert nsets > 1                                               # the rotation is exercised
    seed = bench.operand_seed(0, bench.timed_set(warmup, steps - 1, nsets))
    mat, vec = bench.make_inputs("sym_solve", 3, torch.float32, batch, "cuda:0", seed=seed)
    assert G.rel_err(torch.from_numpy(got), P.sym_solve(mat.cpu(), vec.cpu())) <= TOL[torch.float32]


@pytest.mark.gpu
def test_dump_outputs_has_the_shape_of_the_public_api(tmp_path):
    """batchinv returns (..., n, n): the dump of the dense inverse workload does as well."""
    r = _run("--workload", "dense_inv4_f64", "--steps", "2", "--warmup", "3", "--batch", "100000", "--no-cpu",
             "--no-e2e", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    got = np.load(tmp_path / "dense_inv4_f64.npy")
    assert got.dtype == np.float64 and got.shape == (100_000, 4, 4)
    nsets = bench.operand_set_count(100_000 * bench.algorithmic_bytes("batch_inv", 4, 8))
    a, = bench.make_inputs("batch_inv", 4, torch.float64, 100_000, "cuda:0",
                           seed=bench.operand_seed(0, bench.timed_set(3, 1, nsets)))
    assert G.rel_err(torch.from_numpy(got), P.batchinv(a.cpu()), 2) <= TOL[torch.float64]
