"""Data-parallel full-neighbourhood inference: parallel.infer_full with every rank of a world run in one process (one plan per rank,
the row exchange a local copy) must give logits torch.equal to the one-call Plan.infer_full, in every arithmetic mode, on the
streamed skewed graph of test_gpu_full_inference.py (in-degrees 0 .. 120000, hubs).  Also: Plan.infer_full_layer over a row list
equals it over a range, shards with hand-picked bounds, training state across a sharded call, and argument errors."""
import threading

import numpy as np
import pytest
import torch

from test_gpu_full_inference import _features, _graph, _model

pytestmark = pytest.mark.gpu
DEGS = [0, 1, 31, 32, 33, 255, 256, 1000, 5000, 120000]
HUB = len(DEGS) - 1


def _skewed(V=6000, seed=1):
    rng = np.random.default_rng(seed)
    dst = np.concatenate([np.full(d, v) for v, d in enumerate(DEGS)] + [rng.integers(len(DEGS), V, 30000)]).astype(np.int64)
    src = rng.integers(0, V, dst.size).astype(np.int64)
    perm = rng.permutation(dst.size)
    g = _graph(V, src[perm], dst[perm], batches=7)
    assert g.stats()["relocations"] > 0 and g.degrees()[:len(DEGS)].tolist() == DEGS
    return g


def _sharded(plans, g, f, w, vertices=None):
    """parallel.infer_full on ranks 0 .. w-1 of a world in this process: one thread per rank, taking turns (one lock), the exchange
    a copy of the other ranks' rows out of their tables once every rank has computed its own (a barrier)"""
    from ogl_b200 import parallel
    lock, barrier = threading.Lock(), threading.Barrier(w, timeout=300)
    posted, results, errors = {}, [None] * w, []

    def run(r):
        calls = [0]

        def exchange(table, bounds):
            k = calls[0]
            calls[0] += 1
            posted.setdefault(k, [None] * w)[r] = table
            for phase in range(2):             # 0: every rank has posted its rows; 1: every rank has copied
                lock.release()
                try:
                    barrier.wait()
                finally:
                    lock.acquire()
                if phase == 0:
                    for q in range(w):
                        if q != r and bounds[q + 1] > bounds[q]:
                            table[bounds[q]:bounds[q + 1]].copy_(posted[k][q][bounds[q]:bounds[q + 1]])

        try:
            with lock:
                results[r] = parallel.infer_full(plans[r], g, f, vertices, exchange=exchange, r=r, w=w)
        except BaseException as e:             # (the other ranks would wait at the barrier for ever)
            errors.append(e)
            barrier.abort()

    threads = [threading.Thread(target=run, args=(r,)) for r in range(w)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    torch.cuda.synchronize()
    return results


@pytest.mark.parametrize("mode", ["fp32", "tf32", "fp16", "bf16"])
@pytest.mark.parametrize("dims", [(50, 24, 5), (20, 16, 16, 3)])
def test_sharded_logits_equal_the_one_gpu_call(mode, dims):
    from ogl_b200 import parallel
    g = _skewed()
    V = g.num_vertices
    _, _, f = _features(V, dims[0], mode)
    plans = [_model(dims, mode, V)[2] for _ in range(9)]
    ref = plans[8].infer_full(g, f)
    rng = np.random.default_rng(2)
    some = torch.as_tensor(np.concatenate([rng.permutation(V)[:500], [HUB, HUB, 0, V - 1]]), device="cuda")
    ref_some = plans[8].infer_full(g, f, some)
    # at W = 8 the hub is the last row of rank 0 and several ranks have no rows
    b8 = parallel.edge_balanced_bounds(g.degrees(), 8)
    assert b8[1] == HUB + 1 and sum(1 for r in range(8) if b8[r + 1] == b8[r]) >= 3, b8
    for w in (1, 2, 3, 8):
        for got in _sharded(plans, g, f, w):
            assert torch.equal(got, ref), (mode, dims, w)
        for got in _sharded(plans, g, f, w, some):
            assert torch.equal(got, ref_some), (mode, dims, w, "vertex list")
        # an uneven vertex list with fewer vertices than ranks
        for got in _sharded(plans, g, f, w, some[:2]):
            assert torch.equal(got, ref_some[:2])


@pytest.mark.parametrize("mode", ["fp16", "tf32"])
def test_layer_over_rows_and_hand_picked_bounds(mode):
    """every layer over a row list equals it over the same range; shards of hand-picked bounds (the hub alone, the hub first in a
    shard, an empty shard, one row) assembled in one table give the one-call logits"""
    g = _skewed()
    V = g.num_vertices
    dims = (20, 16, 16, 3)
    _, _, f = _features(V, dims[0], mode)
    _, _, plan = _model(dims, mode, V)
    ref = plan.infer_full(g, f)
    for bounds in ([0, HUB, HUB + 1, HUB + 1, V], [0, 3, HUB, 2000, 2001, V], [0, V, V]):
        h = None
        tables = []
        for l in range(plan.L):
            last = l == plan.L - 1
            out = torch.empty(V, dims[-1], device="cuda") if last else plan.hidden_table(l, V)
            for lo, hi in zip(bounds, bounds[1:]):
                got = plan.infer_full_layer(g, f, l, h, row0=lo, n=hi - lo, out=out[lo:hi])
                by_list = plan.infer_full_layer(g, f, l, h, rows=torch.arange(lo, hi, device="cuda"))
                assert torch.equal(by_list, got), (bounds, l, lo, hi)
            tables.append(out)
            h = out
        assert torch.equal(tables[-1], ref), bounds
    # a row list in any order, with repeats, equals the rows of the one call; a logits buffer with a wider pitch
    rows = torch.as_tensor([HUB, 5, 5, V - 1, 0, HUB], device="cuda")
    wide = torch.full((rows.numel(), 8), 7.0, device="cuda")
    got = plan.infer_full_layer(g, f, plan.L - 1, tables[-2], rows=rows, out=wide)
    assert torch.equal(got[:, :dims[-1]], ref[rows]) and bool((wide[:, dims[-1]:] == 7.0).all())


def _train_run(mode, with_infer):
    from ogl_b200 import parallel
    rng = np.random.default_rng(6)
    V, E, dims, fan, B = 1500, 9000, (50, 24, 5), (6, 4), 64
    src, dst = rng.integers(0, V, E).astype(np.int64), rng.integers(0, V, E).astype(np.int64)
    g = _graph(V, src, dst, symmetric=True)
    _, _, f = _features(V, dims[0], mode)
    _, flat, plan = _model(dims, mode, V, fanouts=fan, max_seeds=B)
    batches = [torch.as_tensor(rng.permutation(V)[:B], device="cuda") for _ in range(7)]
    losses = []
    for i, sd in enumerate(batches):
        per = torch.empty(B, device="cuda")
        if i == 3:
            plan.prefetch(g, f, sd)
            if with_infer:
                parallel.infer_full(plan, g, f, exchange=lambda t, b: None, r=1, w=3)
                parallel.infer_full(plan, g, f, sd, exchange=lambda t, b: None, r=0, w=2)
            plan.step_finish(f, 1.0 / B, per_vertex_out=per)
        else:
            plan.train_step(g, f, sd, loss_scale=1.0 / B, per_vertex_out=per)
        losses.append(per)
    torch.cuda.synchronize()
    return torch.stack(losses), flat.clone()


@pytest.mark.parametrize("mode", ["fp16", "tf32"])
def test_sharded_call_leaves_training_bit_identical(mode):
    l0, w0 = _train_run(mode, False)
    l1, w1 = _train_run(mode, True)
    assert torch.equal(l0, l1) and torch.equal(w0, w1)


def test_layer_errors():
    import ogl_b200
    rng = np.random.default_rng(9)
    V, dims = 500, (20, 16, 4)
    g = _graph(V, rng.integers(0, V, 3000), rng.integers(0, V, 3000), symmetric=True)
    _, _, f = _features(V, dims[0], "fp16")
    _, _, plan = _model(dims, "fp16", V)
    h = plan.hidden_table(0, V)
    plan.infer_full_layer(g, f, 0, None, out=h[:V])
    for layer in (-1, 2):
        with pytest.raises(ogl_b200.OglError, match="out of range"):
            plan.infer_full_layer(g, f, layer, h, row0=0, n=4, out=torch.empty(4, 16, dtype=torch.float16, device="cuda"))
    wide = torch.zeros(V, 24, dtype=torch.float16, device="cuda")
    with pytest.raises(ogl_b200.OglError, match="h must be"):
        plan.infer_full_layer(g, f, 1, wide, row0=0, n=4)
    with pytest.raises(ogl_b200.OglError, match="not vertices"):
        plan.infer_full_layer(g, f, 1, h, row0=V - 5, n=10, out=torch.empty(10, dims[-1], device="cuda"))
    with pytest.raises(ogl_b200.OglError, match="not vertices"):
        plan.infer_full_layer(g, f, 0, None, row0=-1, n=2)
    with pytest.raises(ogl_b200.OglError, match="out must be"):
        plan.infer_full_layer(g, f, 0, None, row0=0, n=4, out=torch.empty(4, 24, dtype=torch.float16, device="cuda"))
    # an empty range is a no-op, also at the end of the graph
    assert plan.infer_full_layer(g, f, 1, h, row0=V, n=0).shape == (0, dims[-1])
    assert plan.error_flags() == 0
