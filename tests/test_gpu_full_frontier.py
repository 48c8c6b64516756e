"""Full-neighbourhood inference of short vertex lists over their in-neighbourhood frontier: Graph.in_frontier against torch, and
Plan.infer_full / infer_full_loss over a list torch.equal to the whole-graph call indexed by the list, in every arithmetic mode,
whichever path the plan takes.  Hidden rows outside a layer's frontier keep stale contents, which no needed row may read.  Also:
training state across a frontier call, and the trainers' full evaluation and PBR priorities on snapshot lists that take it.
The graphs are streamed with in-degrees from 0 to 120,000 (hubs cut into chunks), relocated rows and snapshot tails, as in
test_gpu_full_inference.py."""
import random

import numpy as np
import pytest
import torch

from test_gpu_full_inference import DIMS, _features, _graph, _model
from test_gpu_full_inference_sharded import DEGS, HUB, _skewed

pytestmark = pytest.mark.gpu
MODES = ["fp32", "tf32", "fp16", "bf16"]
# the edge shares (sum over a layer's rows of in-degree + 1, over E + V) of the short lists below stay under this; the plan's
# threshold (DESIGN.md 3d) is above it, so these lists take the frontier path
SHORT_SHARE = 0.5


def _ref_frontier(g, rows):
    """torch.unique(cat(rows, sources of rows' in-edges)) over the exported CSR (ids outside the graph dropped), sum(deg + 1)"""
    indptr, indices, _ = g.export_csr()
    V = indptr.numel() - 1
    r = rows[(rows >= 0) & (rows < V)]
    a, b = indptr[r], indptr[r + 1]
    lens = b - a
    first = torch.repeat_interleave(a - (torch.cumsum(lens, 0) - lens), lens)
    src = indices[first + torch.arange(int(lens.sum()), device="cuda")]
    ref = torch.unique(torch.cat([r, src]))
    deg = indptr[1:] - indptr[:-1]
    return ref, int((deg[ref] + 1).sum())


def _short_graph(V=6000, seed=2):
    """the skewed degrees of DEGS on vertices 0..9, but no edge leaves them: a list of other vertices has a small frontier at every
    depth, and a list with the hub a frontier of most edges"""
    rng = np.random.default_rng(seed)
    dst = np.concatenate([np.full(d, v) for v, d in enumerate(DEGS)] + [rng.integers(len(DEGS), V, 30000)]).astype(np.int64)
    src = rng.integers(len(DEGS), V, dst.size).astype(np.int64)
    perm = rng.permutation(dst.size)
    g = _graph(V, src[perm], dst[perm], batches=7)
    assert g.stats()["relocations"] > 0 and g.degrees()[:len(DEGS)].tolist() == DEGS
    return g


def _share(g, rows, depth):
    """edge share of the rows the deepest of `depth` expansions of `rows` reaches"""
    cost = 0
    for _ in range(depth):
        rows, cost = g.in_frontier(rows)
    return cost / (g.num_edges + g.num_vertices)


def _stages(plan, fn):
    """fn()'s result and the names of the plan's stages that launched kernels in it"""
    plan.profile(True)
    out = fn()
    stages, _, _ = plan.profile_read()
    plan.profile(False)
    return out, {k for k, (_, launches) in stages.items() if launches > 0}


# ----------------------------------------------------------------------------------------------------------- 1. the kernel
def test_in_frontier_matches_torch():
    g = _skewed()
    V = g.num_vertices
    rng = np.random.default_rng(3)
    lists = {
        "duplicates, hub, isolated": [HUB, 0, 0, 5, HUB, 17, 17, 17] + rng.integers(0, V, 40).tolist(),
        "scattered": rng.permutation(V)[:700].tolist() + [8, 8, 7],
        "every vertex": list(range(V)),
        "one isolated vertex": [0],
        "empty": [],
        "out of range": [-1, V, V + 7, 3, 2**40, 3],
    }
    for what, rows in lists.items():
        t = torch.as_tensor(rows, dtype=torch.int64, device="cuda")
        got, cost = g.in_frontier(t)
        ref, ref_cost = _ref_frontier(g, t)
        assert got.dtype == torch.int64 and torch.equal(got, ref), what
        assert cost == ref_cost, what
    _, cost = g.in_frontier(torch.arange(V, device="cuda"))
    assert cost == g.num_edges + V


def test_in_frontier_on_a_vertex_stream_prefix():
    import ogl_b200
    from oracle.graph import in_csr
    rng = np.random.default_rng(8)
    V, E, n_active = 1200, 6000, 700
    src, dst = rng.integers(0, V, E), rng.integers(0, V, E)
    ip, ix, ei = in_csr(np.concatenate([src, dst]), np.concatenate([dst, src]), V)
    g = ogl_b200.native.Graph(V, 2 * E + 16)
    g.load_parent(ip, ix, ei)
    g.set_active_prefix(n_active)
    assert g.num_vertices == n_active
    for rows in (rng.permutation(n_active)[:30], [0, 1, 699, 700, 1100]):
        t = torch.as_tensor(np.asarray(rows, dtype=np.int64), device="cuda")
        got, cost = g.in_frontier(t)
        ref, ref_cost = _ref_frontier(g, t)
        assert torch.equal(got, ref) and cost == ref_cost
        assert int(got.max()) < n_active


# ----------------------------------------------------------------------------------------------------------- 2. logits and losses
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("dims,fanouts", DIMS)
def test_frontier_inference_equals_the_whole_graph_call(mode, dims, fanouts):
    """a short list (duplicates, an isolated vertex, an out-of-range id scored as vertex 0) runs every hidden layer on its frontier;
    a list with the hub runs them over all rows; both give the bits of the whole-graph call indexed by the list"""
    g = _short_graph()
    V, L = g.num_vertices, len(dims) - 1
    _, _, f = _features(V, dims[0], mode)
    _, _, plan = _model(dims, mode, V, fanouts=fanouts)
    whole = plan.infer_full(g, f)
    rng = np.random.default_rng(4)
    short = torch.as_tensor(np.concatenate([rng.integers(len(DEGS), V, 24), [31, 31, 0, V + 5]]), device="cuda")
    long = torch.as_tensor(np.concatenate([[HUB], rng.permutation(V)[:3000]]), device="cuda")
    assert _share(g, short, max(L - 1, 1)) < SHORT_SHARE
    assert _share(g, long, 1) > 0.95                # (above the plan's threshold: layer 0 runs over all rows)
    for rows, frontier in ((short, True), (long, False)):
        idx = torch.where((rows >= 0) & (rows < V), rows, torch.zeros_like(rows))
        got, stages = _stages(plan, lambda: plan.infer_full(g, f, rows))
        assert torch.equal(got, whole[idx])
        ran = {s for s in stages if s.endswith((".frontier", ".scatter"))}
        if L == 1:
            assert not ran
        elif frontier:
            assert ran == {"full.l%d.%s" % (l, k) for l in range(L - 1) for k in ("frontier", "scatter")}
        else:
            assert ran == {"full.l%d.frontier" % (L - 2)}
        loss = plan.infer_full_loss(g, f, rows)
        ref = plan.full_xent(f, whole[idx], rows=rows)
        assert torch.equal(loss.view(torch.int32), ref.view(torch.int32))        # (bits: a label outside [0, C) gives NaN)
        logits = torch.empty_like(got)
        plan.infer_full_loss(g, f, rows, logits_out=logits)
        assert torch.equal(logits, got)
    assert plan.error_flags() & 1


# ----------------------------------------------------------------------------------------------------------- 3. stale rows
@pytest.mark.parametrize("mode", ["fp32", "fp16"])
def test_stale_hidden_rows_are_never_read(mode):
    """rows of the hidden tables outside a layer's frontier keep what an earlier call left there -- NaN, another list's rows, the rows
    of other weights -- and the result does not change"""
    dims = (20, 16, 16, 3)
    g = _short_graph()
    V = g.num_vertices
    _, _, f = _features(V, dims[0], mode)
    params, flat, plan = _model(dims, mode, V, fanouts=(3, 3, 2))
    whole = plan.infer_full(g, f)
    rng = np.random.default_rng(6)
    a = torch.as_tensor(rng.integers(len(DEGS), V, 16), device="cuda")
    b = torch.as_tensor(rng.integers(len(DEGS), V, 16), device="cuda")
    for t in ("full_h0", "full_h1"):
        plan.tensor(t).fill_(float("nan"))
    assert torch.equal(plan.infer_full(g, f, a), whole[a])
    assert torch.equal(plan.infer_full(g, f, b), whole[b])
    assert torch.equal(plan.infer_full(g, f, a), whole[a])
    # the tables full of another model's rows
    other = torch.randn_like(flat)
    plan.bind_params(other, torch.zeros_like(other))
    plan.infer_full(g, f)
    plan.bind_params(flat, torch.zeros_like(flat))
    assert torch.equal(plan.infer_full(g, f, b), whole[b])
    assert bool(torch.isfinite(whole).all())


# ----------------------------------------------------------------------------------------------------------- 4. training state
def _train_run(mode, with_infer, prefetch):
    rng = np.random.default_rng(6)
    V, E, dims, fan, B = 1500, 9000, (50, 24, 5), (6, 4), 64
    src, dst = rng.integers(0, V, E).astype(np.int64), rng.integers(0, V, E).astype(np.int64)
    g = _graph(V, src, dst, symmetric=True)
    _, _, f = _features(V, dims[0], mode)
    params, flat, plan = _model(dims, mode, V, fanouts=fan, max_seeds=B)
    batches = [torch.as_tensor(rng.permutation(V)[:B], device="cuda") for _ in range(7)]
    short = torch.as_tensor(rng.permutation(V)[:6], device="cuda")
    assert _share(g, short, 1) < SHORT_SHARE
    losses = []
    for i, sd in enumerate(batches):
        per = torch.empty(B, device="cuda")
        if prefetch and i == 3:
            plan.prefetch(g, f, sd)
            if with_infer:
                plan.infer_full(g, f, short)
            plan.step_finish(f, 1.0 / B, per_vertex_out=per)
        else:
            plan.train_step(g, f, sd, loss_scale=1.0 / B, per_vertex_out=per)
            if with_infer and not prefetch and i == 3:
                plan.infer_full_loss(g, f, short)
        losses.append(per)
    torch.cuda.synchronize()
    return torch.stack(losses), flat.clone()


@pytest.mark.parametrize("mode", ["fp16", "tf32"])
@pytest.mark.parametrize("prefetch", [False, True])
def test_frontier_call_leaves_training_bit_identical(mode, prefetch):
    l0, w0 = _train_run(mode, False, prefetch)
    l1, w1 = _train_run(mode, True, prefetch)
    assert torch.equal(l0, l1) and torch.equal(w0, w1)


# ----------------------------------------------------------------------------------------------------------- 5. trainers
def _stream(V, E, F_, C, seed):
    from test_gpu_trainers import _planted, _relabel_first_appearance
    src, dst, x, y = _planted(V, E, F_, C, seed=seed)
    src, dst, x, y = _relabel_first_appearance(src, dst, x, y)
    return src, dst, x, y


@pytest.fixture
def small_buffer():
    from ogl_b200.graph import train_test_graph as ttg
    old = ttg.SIZE_BUFFER
    ttg.SIZE_BUFFER = 1 << 12
    yield
    ttg.SIZE_BUFFER = old


def _seed_all():
    random.seed(1)
    np.random.seed(1)
    torch.manual_seed(1)


def test_pbr_priorities_of_snapshot_lists(small_buffer):
    """PBR with priority_neighbourhood="full": a recompute over one snapshot's new train vertices (the frontier path) leaves the
    sum-tree leaves that the whole-graph losses of those vertices give"""
    import ogl_b200
    from ogl_b200 import config
    from ogl_b200.graph.train_test_graph import TrainTestGraph
    config.set_faithful(False)
    config.set_precision("fp16")
    _seed_all()
    V, E, F_, C, H, snapshots = 3000, 4000, 12, 3, 16, 40
    src, dst, x, y = _stream(V, E, F_, C, seed=5)
    GraphSAGE, _, PrioT, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, -1)
    dyn = ogl_b200.DynamicGraphEdge(snapshots, set(range(len(x))))
    dyn.build(x, y, edge_timestamps={"src": src, "dst": dst})
    gu = TrainTestGraph(dyn, split=0.15, start_prior_alpha=4, end_prior_alpha=50, scale=1, max_priority=10)
    t = PrioT(GraphSAGE(F_, H, C, 1, act, 0, "pool").cuda(), 4, 32, y, 5, ogl_b200.LossPriority(), full_pass=2, cuda=True,
              batch_full=128, n_workers=0, priority_neighbourhood="full")
    t.build_optimizer()
    checked = 0
    for _ in range(snapshots * 2 // 3):
        t.train_timestep(gu)
        gu.evolve()
        new = list(gu.get_new_train_nodes())
        if not new:
            continue
        graph = gu.get_graph()
        ids = torch.as_tensor(np.asarray(gu.get_original_to_subgraph_map()[np.asarray(new)], dtype=np.int64), device="cuda")
        train = list(gu.get_train_set())
        _, stages = _stages(t.graphsage_model.inference_plan(graph), lambda: t.recompute_priorities(gu, new))
        if "full.l0.scatter" not in stages:
            continue
        got = gu.dump_priorities(train)
        whole = t.graphsage_model.inference_loss(graph, torch.arange(graph.native.num_vertices, device="cuda"))
        gu.update_priorities_device(new, whole[ids])
        assert gu.dump_priorities(train) == got
        checked += 1
    assert checked >= 3


def test_next_snapshot_evaluation_rows(small_buffer, tmp_path):
    """evaluate_next_snapshots with eval_neighbourhood="full" writes the row that whole-graph logits give"""
    import ogl_b200
    from ogl_b200 import config
    from ogl_b200.graph.train_test_graph import TrainTestGraph
    config.set_faithful(True)
    config.set_precision("fp16")
    _seed_all()
    V, E, F_, C, H, snapshots, delta = 3000, 4000, 12, 3, 16, 40, 2
    src, dst, x, y = _stream(V, E, F_, C, seed=7)
    GraphSAGE, RandomT, _, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, -1)
    labelled = set(range(len(x)))
    dyn = ogl_b200.DynamicGraphEdge(snapshots, labelled)
    dyn.build(x, y, edge_timestamps={"src": src, "dst": dst})
    dyn_test = ogl_b200.DynamicGraphEdge(snapshots, labelled)
    dyn_test.build(x, y, edge_timestamps={"src": src, "dst": dst})
    for _ in range(delta):
        dyn_test.evolve()
    gu = TrainTestGraph(dyn, split=0.15, start_prior_alpha=4, end_prior_alpha=50, scale=1, max_priority=10)
    t = RandomT(GraphSAGE(F_, H, C, 1, act, 0, "pool").cuda(), 4, 32, y, 5, cuda=True, batch_full=128, n_workers=0,
                eval_neighbourhood="full")
    t.build_optimizer()
    model = t.graphsage_model
    real = model.inference
    paths = []

    def recorded(graph, vertices=None, distributed=False):
        out, stages = _stages(model.inference_plan(graph), lambda: real(graph, vertices, distributed))
        paths.append("full.l0.scatter" in stages)
        return out

    def whole_graph(graph, vertices=None, distributed=False):
        return real(graph, None, distributed)[vertices]

    rows = []
    for _ in range(snapshots // 3):
        t.train_timestep(gu)
        pair = []
        for fn, name in ((recorded, "a.csv"), (whole_graph, "b.csv")):
            out = str(tmp_path / name)
            model.inference = fn
            try:
                t.evaluate_next_snapshots(dyn_test, delta, out, at_least=1)
            finally:
                del model.inference
            pair.append(open(out).read())
        assert pair[0] == pair[1]
        rows.append(pair[0])
        gu.evolve()
        dyn_test.evolve()
    assert any(r for r in rows)
    assert sum(paths) >= 3
