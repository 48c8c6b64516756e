"""bench.py --dump-outputs: after the timed steps the outputs of the last one (updated weights, that step's gradient, its loss
sum) are written as fp32 .npy files under the 64 MB cap, and --steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    import bench
    from ogl_b200.graphsage.pytorch.graphsage_dgl import xavier_state_dict

    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3", "--workload", "arxiv",
           "--no-aux", "--no-cpu-baseline", "--no-alt", "--no-parity", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 1, r.stdout[-3000:]
    line = json.loads(lines[0])
    assert line["steps"] == 2 and line["cuda_graph"]["replays_in_timed_region"] > 0

    w = bench.WORKLOADS["arxiv"]
    init = xavier_state_dict(w["F"], w["H"], w["C"], 1, seed=0)
    files = sorted(os.listdir(out))
    assert files == sorted(["loss_sum.npy"] + [k + ".npy" for k in init] + ["grad.%s.npy" % k for k in init])
    assert sum(os.path.getsize(out / f) for f in files) <= bench.DUMP_LIMIT_BYTES
    for k, v in init.items():
        a, g = np.load(out / (k + ".npy")), np.load(out / ("grad.%s.npy" % k))
        assert a.dtype == g.dtype == np.float32 and a.shape == g.shape == tuple(v.shape), k
        assert np.isfinite(a).all() and np.isfinite(g).all(), k
        assert not np.array_equal(a, v.float().numpy()), k + " was not trained"
    loss = np.load(out / "loss_sum.npy")
    assert loss.dtype == np.float32 and loss.shape == (1,)
    assert 0.0 < float(loss[0]) / w["B"] < 20.0
