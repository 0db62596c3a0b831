"""bench.py contract checks: the reference arm (the CPU restatement of the reference path) prints one JSON line with the
agreed keys, alone and under torchrun (rank 0 prints, the other ranks exit 0 without work); on a GPU, --dump-outputs
writes what the timed path computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-n", "48", "--cpu-cg-iters", "5", "--cpu-solve-n", "32",
        "--grid", "48"]
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _json_lines(out):
    return [json.loads(line) for line in out.splitlines() if line.startswith("{")]


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + ARGS, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1
    d = lines[0]
    assert KEYS <= set(d) and d["impl"] == "reference" and d["unit"] == "DoFs/s" and d["value"] > 0
    # the CPU arm runs with all the host threads it can use; the serial walk of the reference is reported next to it
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == (os.cpu_count() or 1) and "sample" in d["cpu_baseline"]
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["one_core"]["cores"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "DoFs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"] and d["config"]["cells"] == 48 * 48
    # the "CG solve s" half of the metric: a Jacobi-CG solve to 1e-10 on a bounded sample
    assert d["cpu_baseline"]["solve"]["relative_residual"] <= 1e-10 and d["cpu_baseline"]["solve"]["iterations"] > 0


def test_reference_arm_under_torchrun_prints_on_rank_zero_only():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(ROOT, "bench.py"), "--gpus", "2"] + ARGS
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1 and lines[0]["n_gpus"] == 2 and lines[0]["impl"] == "reference"


def test_arguments_without_a_meaning_are_refused():
    for extra in (["--steps", "0"], ["--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + ARGS + extra, capture_output=True, text=True,
                           timeout=300, cwd=ROOT)
        assert r.returncode == 2 and extra[0] in r.stderr, r.stderr[-2000:]
    assert not os.path.exists(os.path.join(ROOT, "unused"))


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_step_and_repeat(gpu, tmp_path):
    """--dump-outputs on a 64^2 grid (no array is sampled): solution, system matrix values and rhs of the timed path equal
    the oracle's, and a second run with the same arguments writes the same arrays"""
    from dune_hdd_b200 import grids
    from oracle import oracle as o
    from tests.helpers import direct_solve, oracle_system, rel
    n = 64
    args = ["--steps", "2", "--warmup", "1", "--grid", str(n), "--no-cpu-baseline", "--no-e2e", "--no-estimator",
            "--no-parity"]
    runs = []
    for k in range(2):
        out = tmp_path / str(k)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args + ["--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert len(_json_lines(r.stdout)) == 1
        runs.append({p.stem: np.load(p) for p in out.glob("*.npy")})
    a, b = runs
    assert sorted(a) == ["rhs", "solution", "system_matrix"] and all(v.dtype == np.float64 for v in a.values())
    _, rp, col, A, rhs = oracle_system(grids.cube(n, partitions=(8, 8)), o.const(1.0), o.esv2007_force())
    assert a["system_matrix"].shape == A.shape and rel(a["system_matrix"], A) <= 1e-12
    assert a["rhs"].shape == rhs.shape and rel(a["rhs"], rhs) <= 1e-12
    assert rel(a["solution"], direct_solve(rp, col, A, rhs)) <= 1e-8
    for key in a:
        assert rel(b[key], a[key]) <= (1e-8 if key == "solution" else 1e-12), key
