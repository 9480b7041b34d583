"""bench.py on a machine without a GPU: the reference arm (`--impl reference`, the CPU port of the reference formulation)
must print exactly one JSON line with the keys the driver's contract names, and the B200 arm must refuse to run rather
than fall back to anything."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, env=env)


def test_reference_arm_prints_the_contract_line():
    out = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-molecules", "16")
    assert out.returncode == 0, out.stderr[-500:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "atoms/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 0 and d["gpu_launches"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "16 molecules" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_b200_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        return                                  # on a GPU box this arm simply runs; the GPU suite covers it
    out = _run("--steps", "1", "--warmup", "0", "--no-cpu-baseline")
    assert out.returncode != 0
    assert "no CPU fallback" in (out.stderr + out.stdout)


import pytest


def test_dump_outputs_writes_float_arrays_and_a_fixed_sample(tmp_path, monkeypatch):
    """--dump-outputs: small outputs are written whole; above the size limit both arrays hold the same seeded sample of atoms
    in atom order, the same on every run."""
    sys.path.insert(0, ROOT)
    import bench
    q64 = np.arange(5000) + 0.25                     # each value names its atom
    q32 = (q64 - 0.5).astype(np.float32)
    bench.dump_outputs(str(tmp_path / "whole"), q32, q64)
    assert np.array_equal(np.load(tmp_path / "whole" / "charges.npy"), q32)
    assert np.array_equal(np.load(tmp_path / "whole" / "charges_f64.npy"), q64)
    monkeypatch.setattr(bench, "DUMP_MAX_ATOMS", 1000)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), q32, q64)
    a32, a64 = np.load(tmp_path / "a" / "charges.npy"), np.load(tmp_path / "a" / "charges_f64.npy")
    assert a32.dtype == np.float32 and a64.dtype == np.float64 and a32.shape == a64.shape == (1000,)
    atoms = (a64 - 0.25).astype(np.int64)
    assert np.all(np.diff(atoms) > 0) and np.array_equal(a32, q32[atoms])
    assert np.array_equal(np.load(tmp_path / "b" / "charges.npy"), a32) and np.array_equal(np.load(tmp_path / "b" / "charges_f64.npy"), a64)


@pytest.mark.gpu
def test_b200_arm_prints_the_contract_line_with_roofline_baseline_and_secondary_blocks(tmp_path):
    """The default invocation (`python bench.py`), shrunk: one JSON line on stdout carrying the base contract, the
    roofline / cpu_baseline / e2e objects of this tier and the secondary blocks (strong scaling, live-GNN checkpoints, the
    reference's three own configurations); --dump-outputs leaves the charges of the last timed step."""
    out = _run("--molecules", "20000", "--steps", "2", "--warmup", "3", "--ref-molecules", "64", "--strong-atoms", "3000",
               "--dump-outputs", str(tmp_path))
    assert out.returncode == 0, out.stderr[-800:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline", "secondary"):
        assert k in d, k
    assert d["unit"] == "atoms/s" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["vs_baseline"] is None
    assert d["value"] > 1e6 and d["gpu_launches"] > 20 and "workload" in d["config"] and "model" not in d["config"]
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] > 0
    r = d["roofline"]
    assert r["bound"] == "fp32" and 0 < r["frac"] < 1 and r["peak"] > 50 and r["traffic"] and 0 < r["algorithmic"]["frac"] < 1.2
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and "64 molecules" in cb["sample"]
    assert d["checks"]["max_abs_sum_q_minus_Q"] < 1e-6
    s = d["secondary"]
    for k in ("strong_qm9", "strong_protein", "live_gnn_model2_weights", "live_gnn_model_weights", "config_qm9_test", "config_ssi", "config_galectin3c"):
        assert k in s and s[k]["value"] > 0, k
    assert s["config_qm9_test"]["precision_used"] == 64 and s["config_ssi"]["precision_used"] == 32
    assert s["config_galectin3c"]["max_abs_dq_vs_reference_preds_npy"] < 1e-5
    assert s["strong_protein"]["checks"]["max_abs_sum_q_minus_Q"] < 1e-6
    q32, q64 = np.load(tmp_path / "charges.npy"), np.load(tmp_path / "charges_f64.npy")
    assert q32.dtype == np.float32 and q64.dtype == np.float64 and q32.shape == q64.shape == (d["config"]["atoms_per_gpu_per_step"],)
    assert np.abs(q32 - q64).max() < 1e-6 and abs(q64.sum()) < 20000 * 1e-6          # 20000 neutral molecules
