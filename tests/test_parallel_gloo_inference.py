"""Host logic of data-parallel full inference on CPU: edge-balanced row bounds (one process) and the in-place row exchange
allgather_rows under gloo with world size 2 (uneven and empty slices)."""
import importlib.util
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _parallel(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "online-gnn-learning_b200", "parallel.py"))
    par = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(par)
    return par


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_edge_balanced_bounds():
    par = _parallel("ogl_parallel_bounds")
    rng = np.random.default_rng(3)
    skewed = rng.integers(0, 40, 5000)
    skewed[[17, 2500, 4999]] = [30000, 12000, 9000]                   # hubs, one of them the last row
    cases = [skewed, np.zeros(300, dtype=np.int64), np.array([0, 5, 0, 100, 1, 1, 2]), np.array([7]), np.zeros(0, dtype=np.int64)]
    for deg in cases:
        cost = deg.astype(np.int64) + 1
        prefix = np.concatenate([[0], np.cumsum(cost)])
        for w in (1, 2, 3, 8, 13, len(deg) + 5):
            b = par.edge_balanced_bounds(torch.as_tensor(deg), w)
            assert len(b) == w + 1 and b[0] == 0 and b[-1] == len(deg)
            assert all(x <= y for x, y in zip(b, b[1:]))
            share = cost.sum() / w
            worst = cost.max() if len(deg) else 0
            for r in range(w):
                assert abs(prefix[b[r + 1]] - prefix[b[r]] - share) <= worst, (w, r, b)
    # W > V leaves ranks without rows; a graph without edges splits its rows evenly
    b = par.edge_balanced_bounds(torch.zeros(3, dtype=torch.int64), 8)
    assert b[-1] == 3 and sum(1 for r in range(8) if b[r + 1] == b[r]) == 5
    assert par.edge_balanced_bounds(torch.zeros(300, dtype=torch.int64), 3) == [0, 100, 200, 300]
    assert par.shard_bounds(10, 3) == [0, 4, 7, 10] and par.shard_bounds(2, 4) == [0, 1, 2, 2, 2]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    par = _parallel("ogl_parallel_rows")
    res = []
    for bounds in ([0, 3, 7], [0, 0, 5], [0, 6, 6], [0, 1, 9]):
        table = torch.zeros(12, 5)                                   # rows past bounds[-1] (table padding) are left alone
        lo, hi = bounds[rank], bounds[rank + 1]
        table[lo:hi] = torch.arange(lo, hi, dtype=torch.float32)[:, None] * 10 + rank + torch.arange(5)[None, :] * 0.5
        assert par.allgather_rows(table, bounds) is table
        res.append(table.tolist())
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_allgather_rows_world_size_two():
    world = 2
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
        r0, r1 = out[0], out[1]
    for i, bounds in enumerate(([0, 3, 7], [0, 0, 5], [0, 6, 6], [0, 1, 9])):
        want = torch.zeros(12, 5)
        for r in range(world):
            lo, hi = bounds[r], bounds[r + 1]
            want[lo:hi] = torch.arange(lo, hi, dtype=torch.float32)[:, None] * 10 + r + torch.arange(5)[None, :] * 0.5
        assert r0[i] == r1[i] == want.tolist(), bounds


def test_allgather_rows_is_a_noop_on_one_process():
    par = _parallel("ogl_parallel_rows1")
    t = torch.arange(6.0).reshape(3, 2)
    assert par.allgather_rows(t, [0, 3]) is t and t.tolist() == [[0, 1], [2, 3], [4, 5]]
