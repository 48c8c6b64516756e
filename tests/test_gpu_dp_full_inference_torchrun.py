"""Data-parallel full inference under torchrun (one process per GPU): the drop-in trainers with eval_neighbourhood="full" write
the same CSV rows as a one-rank evaluation of the same weights, and the sharded logits are bit-equal to the one-rank call on every
rank.  Needs >= 2 GPUs (skipped otherwise); tests/test_gpu_full_inference_sharded.py runs every rank in one process on one GPU."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_trainers_full_evaluation_two_ranks():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29535", os.path.join(ROOT, "tools", "dp_full_inference_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    res = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert res["world"] == 2 and res["rows_equal"] and res["logits_equal"] and res["ranks_equal"], res
