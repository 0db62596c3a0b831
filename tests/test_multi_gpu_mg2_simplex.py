"""Solver type "cg.mg2.simplex" on two GPUs: runs tests/multi_gpu_mg2_simplex_check.py under torchrun when the box has at
least two devices (replicated vertex hierarchy, one all-reduce of the level-0 operator per solve and of P^T r per
application, against the oracle on every rank and against the one-rank iteration count).  Skipped on single-GPU boxes."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_cg_mg2_simplex_on_two_ranks(gpu):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29534", os.path.join(ROOT, "tests", "multi_gpu_mg2_simplex_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.count("multi-GPU cg.mg2.simplex check ok") == 3
