"""The loss exchange of data-parallel full-neighbourhood priorities on CPU: allgather_rows on a 1-D fp32 loss vector under gloo
with world size 2, uneven and empty slices."""
import importlib.util
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUNDS = ([0, 3, 7], [0, 0, 5], [0, 6, 6], [0, 1, 9], [0, 0, 0])


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


def _mine(lo, hi, rank):
    return torch.arange(lo, hi, dtype=torch.float32) * 0.25 + rank * 100.0


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    par = _parallel("ogl_parallel_losses")
    res = []
    for bounds in BOUNDS:
        losses = torch.full((bounds[-1],), float("nan"))              # another rank's entries are garbage until the exchange
        lo, hi = bounds[rank], bounds[rank + 1]
        losses[lo:hi] = _mine(lo, hi, rank)
        assert par.allgather_rows(losses, bounds) is losses
        res.append(losses.tolist())
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_allgather_rows_of_a_loss_vector_world_size_two():
    world = 2
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
        r0, r1 = out[0], out[1]
    for i, bounds in enumerate(BOUNDS):
        want = torch.empty(bounds[-1])
        for r in range(world):
            want[bounds[r]:bounds[r + 1]] = _mine(bounds[r], bounds[r + 1], r)
        assert r0[i] == r1[i] == want.tolist(), bounds
