"""Full-neighbourhood PBR priorities: Plan.infer_full_loss (infer_full + the per-vertex cross entropy on its logits), Plan.full_xent,
the sharded parallel.infer_full_loss with every rank of a world run in one process, and the PBR trainer's
priority_neighbourhood="full".  The skewed streamed graph (in-degrees 0 .. 120000) is the one of test_gpu_full_inference_sharded.py."""
import os
import random
import subprocess
import sys
import threading

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_gpu_full_inference import _features, _graph, _model, close
from test_gpu_full_inference_sharded import HUB, _skewed

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = ["fp32", "tf32", "fp16", "bf16"]


# ----------------------------------------------------------------------------------------------------------- 1. logits and losses
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("dims", [(50, 24, 5), (20, 16, 16, 3)])
def test_loss_logits_equal_infer_full_and_losses_match_cross_entropy(mode, dims):
    g = _skewed()
    V = g.num_vertices
    _, y, f = _features(V, dims[0], mode)
    _, _, plan = _model(dims, mode, V)
    ref_logits = plan.infer_full(g, f)
    logits = torch.empty_like(ref_logits)
    loss = plan.infer_full_loss(g, f, logits_out=logits)
    assert torch.equal(logits, ref_logits)
    close(loss, F.cross_entropy(logits.double(), y.cuda(), reduction="none"), 2e-6, "losses of every vertex")
    assert torch.equal(plan.infer_full_loss(g, f), loss)                       # without a logits buffer: the same bits
    rng = np.random.default_rng(2)
    some = torch.as_tensor(np.concatenate([rng.permutation(V)[:500], [HUB, HUB, 0, V - 1, 7, 7]]), device="cuda")
    logits_s = torch.empty(some.numel(), dims[-1], device="cuda")
    loss_s = plan.infer_full_loss(g, f, some, logits_out=logits_s)
    assert torch.equal(logits_s, plan.infer_full(g, f, some))
    close(loss_s, F.cross_entropy(logits_s.double(), y.cuda()[some], reduction="none"), 2e-6, "losses of a vertex list")
    assert torch.equal(loss_s[-6], loss_s[-5]) and torch.equal(loss_s[-2], loss_s[-1])
    # the loss on its own over the same logits block (the sharded path): the same bits, by range and by list
    assert torch.equal(plan.full_xent(f, ref_logits), loss)
    assert torch.equal(plan.full_xent(f, ref_logits[100:900], row0=100), loss[100:900])
    assert torch.equal(plan.full_xent(f, logits_s, rows=some), loss_s)
    assert plan.error_flags() == 0


# ----------------------------------------------------------------------------------------------------------- 2. sampled == full
@pytest.mark.parametrize("mode", MODES)
def test_full_losses_equal_sampled_eval_when_every_in_degree_is_0_or_1(mode):
    """with in-degree <= 1 the sampled and the full neighbourhood coincide; the two losses share the arithmetic (warp_logsumexp), so
    they are bit-identical"""
    rng = np.random.default_rng(4)
    V, dims = 1000, (50, 24, 5)
    dst = rng.permutation(V)[:700].astype(np.int64)
    src = rng.integers(0, V, dst.size).astype(np.int64)
    g = _graph(V, src, dst)
    assert int(g.degrees().max()) == 1
    _, _, f = _features(V, dims[0], mode)
    _, _, plan = _model(dims, mode, V, fanouts=(6, 4), max_seeds=128)
    seeds = torch.as_tensor(np.concatenate([rng.permutation(V)[:125], rng.permutation(np.setdiff1d(np.arange(V), dst))[:3]]),
                            device="cuda")
    sampled = torch.empty(seeds.numel(), device="cuda")
    plan.eval_step(g, f, seeds, per_vertex_out=sampled)
    full = plan.infer_full_loss(g, f, seeds)
    assert torch.equal(full, sampled)


# ----------------------------------------------------------------------------------------------------------- 3. sharded
def _sharded(fn, plans, g, f, w, vertices=None):
    """fn (parallel.infer_full_loss) on ranks 0 .. w-1 of a world in this process: one thread per rank, taking turns (one lock), the
    exchange a copy of the other ranks' rows out of their tables once every rank has computed its own (a barrier)"""
    lock, barrier = threading.Lock(), threading.Barrier(w, timeout=300)
    posted, results, errors = {}, [None] * w, []
    exchanged = [[] for _ in range(w)]

    def run(r):
        calls = [0]

        def exchange(table, bounds):
            k = calls[0]
            calls[0] += 1
            exchanged[r].append((table.dtype, tuple(table.shape)))
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
                results[r] = fn(plans[r], g, f, vertices, exchange=exchange, r=r, w=w)
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
    return results, exchanged


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("dims", [(50, 24, 5), (20, 16, 16, 3)])
def test_sharded_losses_equal_the_one_gpu_call(mode, dims):
    from ogl_b200 import parallel
    g = _skewed()
    V = g.num_vertices
    _, _, f = _features(V, dims[0], mode)
    plans = [_model(dims, mode, V)[2] for _ in range(9)]
    ref = plans[8].infer_full_loss(g, f)
    rng = np.random.default_rng(2)
    some = torch.as_tensor(np.concatenate([rng.permutation(V)[:500], [HUB, HUB, 0, V - 1]]), device="cuda")
    ref_some = plans[8].infer_full_loss(g, f, some)
    # at W = 8 the hub is the last row of rank 0 and several ranks have no rows
    b8 = parallel.edge_balanced_bounds(g.degrees(), 8)
    assert b8[1] == HUB + 1 and sum(1 for r in range(8) if b8[r + 1] == b8[r]) >= 3, b8
    for w in (1, 2, 3, 8):
        got, exchanged = _sharded(parallel.infer_full_loss, plans, g, f, w)
        for r in range(w):
            assert torch.equal(got[r], ref), (mode, dims, w)
            # the hidden tables, then the fp32 losses [V] only -- no logits
            assert exchanged[r][-1] == (torch.float32, (V,)) and len(exchanged[r]) == len(dims) - 1, exchanged[r]
        for got_r in _sharded(parallel.infer_full_loss, plans, g, f, w, some)[0]:
            assert torch.equal(got_r, ref_some), (mode, dims, w, "vertex list")
        # an uneven vertex list with fewer vertices than ranks
        for got_r in _sharded(parallel.infer_full_loss, plans, g, f, w, some[:2])[0]:
            assert torch.equal(got_r, ref_some[:2])
    assert all(p.error_flags() == 0 for p in plans)


# ----------------------------------------------------------------------------------------------------------- 4. errors
def test_errors():
    import ogl_b200
    from ogl_b200 import parallel
    from ogl_b200._lib import check, lib
    rng = np.random.default_rng(9)
    V, dims = 500, (20, 16, 4)
    C = dims[-1]
    g = _graph(V, rng.integers(0, V, 3000), rng.integers(0, V, 3000), symmetric=True)
    x, y, f = _features(V, dims[0], "fp16")
    _, _, plan = _model(dims, "fp16", V)
    assert plan.error_flags() == 0
    good = plan.infer_full_loss(g, f)
    assert bool(torch.isfinite(good).all()) and plan.error_flags() == 0
    # an out-of-range id: vertex 0 is scored instead (its logits and its label), bit 0
    bad_ids = torch.as_tensor([1, V + 5, -1, 2], device="cuda")
    logits = torch.empty(4, C, device="cuda")
    got = plan.infer_full_loss(g, f, bad_ids, logits_out=logits)
    assert plan.error_flags() == 1
    assert torch.equal(got[1], good[0]) and torch.equal(got[2], good[0]) and torch.equal(got[0], good[1])
    assert torch.equal(plan.full_xent(f, logits, rows=torch.as_tensor([1, V + 7, -3, 2], device="cuda")), got)
    assert plan.error_flags() == 1
    # the sharded call does the same
    assert torch.equal(parallel.infer_full_loss(plan, g, f, bad_ids, exchange=lambda t, b: None, r=0, w=1), got)
    assert plan.error_flags() == 1
    # labels outside [0, C): NaN at those rows, bit 1 (and the other rows untouched)
    y2 = y.clone()
    y2[7], y2[9] = C + 2, -1
    f2 = ogl_b200.native.Features(V, dims[0], ogl_b200.OGL_FP16)
    f2.write(0, x.cuda(), y2.cuda())
    l2 = plan.infer_full_loss(g, f2)
    assert plan.error_flags() == 2
    nan = torch.isnan(l2)
    assert nan[7] and nan[9] and int(nan.sum()) == 2
    keep = torch.ones(V, dtype=torch.bool, device="cuda")
    keep[[7, 9]] = False
    assert torch.equal(l2[keep], good[keep])
    l3 = plan.full_xent(f2, plan.infer_full(g, f2, torch.as_tensor([7, 3], device="cuda")), rows=torch.as_tensor([7, 3], device="cuda"))
    assert torch.isnan(l3[0]) and torch.equal(l3[1], good[3]) and plan.error_flags() == 2
    # n == 0 is a no-op
    empty = torch.empty(0, dtype=torch.int64, device="cuda")
    assert plan.infer_full_loss(g, f, empty).shape == (0,)
    assert plan.full_xent(f, torch.empty(0, C, device="cuda")).shape == (0,)
    assert plan.full_xent(f, torch.empty(0, C, device="cuda"), rows=empty).shape == (0,)
    assert plan.error_flags() == 0
    # wrong dtype, shape or stride
    lg = plan.infer_full(g, f)
    for bad in (lg.double(), lg.half(), lg[:, :C - 1], torch.empty(C, V, device="cuda").t(), lg[:, 0]):
        with pytest.raises(AssertionError):
            plan.full_xent(f, bad)
    with pytest.raises(AssertionError):
        plan.full_xent(f, lg, rows=torch.arange(V - 1, device="cuda"))
    with pytest.raises(AssertionError):
        plan.full_xent(f, lg, out=torch.empty(V, dtype=torch.float64, device="cuda"))
    with pytest.raises(AssertionError):
        plan.infer_full_loss(g, f, loss_out=torch.empty(V + 1, device="cuda"))
    with pytest.raises(AssertionError):
        plan.infer_full_loss(g, f, logits_out=torch.empty(V, C + 1, device="cuda"))
    # the C ABI rejects a row pitch below the class count and a range past the feature store
    out = torch.empty(V, device="cuda")
    with pytest.raises(ogl_b200.OglError, match="ld >="):
        check(lib.ogl_plan_full_xent(plan._h, f._h, lg.data_ptr(), C - 1, None, 0, V, out.data_ptr(), None))
    with pytest.raises(ogl_b200.OglError, match="not rows"):
        plan.full_xent(f, lg, row0=1)
    for bad in (ogl_b200.native.Features(V, dims[0] + 1, ogl_b200.OGL_FP16), ogl_b200.native.Features(V, dims[0], ogl_b200.OGL_BF16)):
        with pytest.raises(ogl_b200.OglError, match="feature store"):
            plan.infer_full_loss(g, bad)
    shard = _graph(V, rng.integers(0, V, 100), rng.integers(0, V, 100))
    shard.set_source_bound(4 * V)
    with pytest.raises(ogl_b200.OglError, match="shard"):
        plan.infer_full_loss(shard, f)
    assert plan.error_flags() == 0


# ----------------------------------------------------------------------------------------------------------- 5. no side effects
def _train_run(mode, with_loss, prefetch):
    from ogl_b200 import parallel
    rng = np.random.default_rng(6)
    V, E, dims, fan, B = 1500, 9000, (50, 24, 5), (6, 4), 64
    src, dst = rng.integers(0, V, E).astype(np.int64), rng.integers(0, V, E).astype(np.int64)
    g = _graph(V, src, dst, symmetric=True)
    _, _, f = _features(V, dims[0], mode)
    params, flat, plan = _model(dims, mode, V, fanouts=fan, max_seeds=B)
    batches = [torch.as_tensor(rng.permutation(V)[:B], device="cuda") for _ in range(7)]
    losses = []
    for i, sd in enumerate(batches):
        per = torch.empty(B, device="cuda")
        if prefetch and i == 3:
            plan.prefetch(g, f, sd)
            if with_loss:
                plan.infer_full_loss(g, f)
                parallel.infer_full_loss(plan, g, f, sd, exchange=lambda t, b: None, r=1, w=3)
            plan.step_finish(f, 1.0 / B, per_vertex_out=per)
        else:
            plan.train_step(g, f, sd, loss_scale=1.0 / B, per_vertex_out=per)
            if with_loss and not prefetch and i == 3:
                plan.infer_full_loss(g, f, sd, logits_out=torch.empty(B, dims[-1], device="cuda"))
                plan.full_xent(f, torch.zeros(B, dims[-1], device="cuda"), rows=sd)
        losses.append(per)
    torch.cuda.synchronize()
    return torch.stack(losses), flat.clone()


@pytest.mark.parametrize("mode", ["fp16", "tf32"])
@pytest.mark.parametrize("prefetch", [False, True])
def test_loss_calls_leave_training_bit_identical(mode, prefetch):
    l0, w0 = _train_run(mode, False, prefetch)
    l1, w1 = _train_run(mode, True, prefetch)
    assert torch.equal(l0, l1) and torch.equal(w0, w1)


# ----------------------------------------------------------------------------------------------------------- 6. PBR trainer
def _pbr(priority_neighbourhood, faithful, matching=False, seed=5):
    """a PBR trainer on a small planted edge stream (matching=True: disjoint vertex pairs, every in-degree 0 or 1) after one timestep"""
    import ogl_b200
    from ogl_b200 import config
    from ogl_b200.graph.train_test_graph import TrainTestGraph
    from test_gpu_trainers import _planted, _relabel_first_appearance
    config.set_faithful(faithful)
    config.set_precision("fp16")
    random.seed(1)
    np.random.seed(1)
    torch.manual_seed(1)
    V, E, F_, C, H = 1200, 9000, 12, 3, 16
    src, dst, x, y = _planted(V, E, F_, C, seed=seed)
    if matching:
        perm = np.random.default_rng(seed).permutation(V)
        src, dst = perm[0:V - 200:2].astype(np.int64), perm[1:V - 200:2].astype(np.int64)
    src, dst, x, y = _relabel_first_appearance(src, dst, x, y)
    GraphSAGE, _, PrioT, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, -1)
    dyn = ogl_b200.DynamicGraphEdge(6, set(range(len(x))))
    dyn.build(x, y, edge_timestamps={"src": src, "dst": dst})
    gu = TrainTestGraph(dyn, split=0.15, start_prior_alpha=4, end_prior_alpha=50, scale=1, max_priority=10)
    t = PrioT(GraphSAGE(F_, H, C, 1, act, 0, "pool").cuda(), 4, 32, y, 5, ogl_b200.LossPriority(), full_pass=2, cuda=True,
              batch_full=128, n_workers=0, priority_neighbourhood=priority_neighbourhood)
    t.build_optimizer()
    t.train_timestep(gu)
    gu.evolve()
    t.train_timestep(gu)
    return t, gu


@pytest.fixture
def small_buffer():
    from ogl_b200.graph import train_test_graph as ttg
    old = ttg.SIZE_BUFFER
    ttg.SIZE_BUFFER = 1 << 12
    yield
    ttg.SIZE_BUFFER = old


def _sub(gu, vertices):
    return torch.as_tensor(np.asarray(gu.get_original_to_subgraph_map()[np.asarray(vertices)], dtype=np.int64), device="cuda")


@pytest.mark.parametrize("faithful", [False, True])
def test_pbr_full_priorities_are_the_transform_of_inference_loss(small_buffer, faithful):
    import ogl_b200
    t, gu = _pbr("full", faithful)
    assert t._device_priorities() == (not faithful)
    train = list(gu.get_train_set())
    graph = gu.get_graph()
    for vertices in (train, list(gu.get_new_train_nodes())):
        t.recompute_priorities(gu, vertices)
        got = gu.dump_priorities(train)
        losses = t.graphsage_model.inference_loss(graph, _sub(gu, vertices))
        assert bool(torch.isfinite(losses).all())
        if len(vertices) == len(train):
            # a whole-train-set update rebuilds the buffer: the same losses pushed again give the same leaves
            if faithful:
                pri = ogl_b200.LossPriority().get_priorities(vertices, losses.cpu().numpy())
                gu.update_priorities(dict(zip(vertices, pri)))
            else:
                gu.update_priorities_device(vertices, losses)
            assert gu.dump_priorities(train) == got
        assert all(np.isfinite(got))
    with pytest.raises(ValueError):
        _pbr("exact", faithful)


def test_pbr_full_and_sampled_trees_agree_when_every_in_degree_is_0_or_1(small_buffer):
    t, gu = _pbr("sampled", False, matching=True)
    graph = gu.get_graph()
    assert int(graph.native.degrees().max()) <= 1
    train = list(gu.get_train_set())
    t.recompute_priorities(gu, train)
    sampled = gu.dump_priorities(train)
    t.priority_neighbourhood = "full"
    t.recompute_priorities(gu, train)
    assert gu.dump_priorities(train) == sampled


def _step_after(recompute):
    t, gu = _pbr("full", False)
    graph = gu.get_graph()
    if recompute:
        t.recompute_priorities(gu, list(gu.get_train_set()))
    seeds = _sub(gu, list(gu.get_train_set())[:32])
    per = torch.empty(seeds.numel(), device="cuda")
    t._fused_step(graph, seeds, per_vertex_out=per)
    ev = torch.empty(seeds.numel(), device="cuda")
    t._eval_plan(graph).eval_step(graph.native, graph.features, seeds, per_vertex_out=ev)
    torch.cuda.synchronize()
    return per, ev, t.graphsage_model._flat.clone()


def test_pbr_full_recompute_leaves_the_philox_step(small_buffer):
    """the next train step (and the next sampled evaluation) after a "full" recompute is bit-identical to the one without it"""
    a = _step_after(False)
    b = _step_after(True)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


# ----------------------------------------------------------------------------------------------------------- 7. driver
def test_driver_full_priorities(tmp_path):
    def run(args):
        r = subprocess.run([sys.executable] + args, cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]

    data = str(tmp_path / "reddit")
    run(["tools/make_synthetic_dataset.py", "reddit", data, "--vertices", "1500", "--edges", "8000", "--feats", "24"])
    out = str(tmp_path / "res.csv")
    run(["train", "reddit", "pytorch", out, str(tmp_path / "tsne"), "--cuda", "--path", data, "--snapshots", "20", "--delta", "2",
         "--eval", "3", "--batch_timestep", "4", "--batch_size", "32", "--embedding_size", "16", "--samples", "5", "--train_offline", "4",
         "--epochs_offline", "1", "--batch_full", "256", "--max_timesteps", "12", "--priority_neighbourhood", "full"])
    rows = [l for l in open(out).read().strip().split("\n") if l]
    pbr = [r for r in rows if r.split(";")[0] == "prioritized"]
    assert len(pbr) >= 2 and all(len(r.split(";")) == 4 for r in pbr)
    scored = [float(r.split(";")[1]) for r in pbr if r.split(";")[1]]
    assert scored and all(0.0 <= s <= 1.0 for s in scored)
