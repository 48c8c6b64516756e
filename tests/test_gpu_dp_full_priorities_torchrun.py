"""Data-parallel full-neighbourhood PBR priorities under torchrun (one process per GPU): the PBR trainer with
priority_neighbourhood="full" keeps bit-identical priority trees on every rank, equal to a one-rank recompute of the same weights,
and the sharded losses are bit-equal to the one-rank call.  Needs >= 2 GPUs (skipped otherwise); tests/test_gpu_full_priorities.py
runs every rank in one process on one GPU."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_pbr_full_priorities_two_ranks():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(ROOT, "tools", "dp_full_priorities_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    res = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert res["world"] == 2 and res["trees_equal"] and res["losses_equal"] and res["ranks_equal"], res
