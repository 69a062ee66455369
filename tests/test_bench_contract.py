"""bench.py contract checks: the reference arm (CPU oracle port) prints one JSON line with the required keys, the
committed round-1 bench line carries the roofline / cpu_baseline / e2e / clocks objects, and (GPU) --dump-outputs writes
the same arrays in every run with the same arguments."""
import json
import os
import subprocess
import sys

import pytest

from tests.conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config"}


def test_reference_arm_prints_one_json_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["steps"] == 2 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    # --dump-outputs: the last step's probabilities and head outputs, float32
    import numpy as np
    probs = np.load(tmp_path / "forward_probs.npy")
    assert probs.dtype == np.float32 and probs.shape == (1, 174) and abs(float(probs.sum()) - 1.0) < 1e-4
    for name in ("forward_logits", "forward_obj_desc", "forward_pred_bboxes", "forward_pred_contact_state"):
        assert np.load(tmp_path / f"{name}.npy").dtype == np.float32


def test_dump_outputs_samples_above_the_budget(tmp_path, monkeypatch):
    import numpy as np
    import torch

    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4 * 1000)
    a, b = torch.arange(3000.0).reshape(30, 100), torch.ones(1000, dtype=torch.float64)
    for d in ("x", "y"):
        bench.dump_outputs(str(tmp_path / d), {"a": a, "b": b})
    ga, gb = np.load(tmp_path / "x" / "a.npy"), np.load(tmp_path / "x" / "b.npy")
    assert ga.dtype == gb.dtype == np.float32 and ga.size == 750 and gb.size == 250
    assert len(np.unique(ga)) == 750 and np.all(np.diff(ga) > 0)  # distinct elements, in storage order
    assert np.array_equal(ga, np.load(tmp_path / "y" / "a.npy"))  # the same sample from run to run


def test_reference_arm_non_zero_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_committed_bench_line_has_the_contract_objects():
    d = json.loads(open(os.path.join(ROOT, "profiles", "r1_final_bench_1gpu.json")).read())
    assert BASE_KEYS <= set(d)
    assert d["config"]["workload"].startswith("SViT") and "model" not in d["config"]
    roof = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(roof)
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["gpu_launches"] > 0 and d["clocks"]["sm_max_mhz"] > 0
    assert d["vs_baseline"] is None  # BASELINE.md holds no published number for this metric


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(tmp_path):
    """Two runs of the CUDA arm with the same arguments: the same seeded inputs, so the same outputs, bit for bit."""
    import numpy as np

    args = ["--batch", "4", "--steps", "2", "--warmup", "1", "--no-train", "--no-cpu-baseline", "--no-torch-gpu-baseline"]
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path / run)],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b"))
    assert {"forward_probs.npy", "forward_logits.npy", "forward_obj_desc.npy", "e2e_probs.npy"} <= set(names)
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float32 and np.isfinite(a).all(), n
        assert np.array_equal(a, b), n
    assert np.load(tmp_path / "a" / "forward_probs.npy").shape == (4, 174)
