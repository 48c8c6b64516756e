"""Incremental full-neighbourhood inference (inference.StreamingInference): the pieces it is built from -- the row-list pool GEMM, the
out-neighbourhood frontier, the suffix segment max -- against whole-table calls and torch, and the engine's logits torch.equal to the
whole-graph call after every batch of an edge or vertex stream, in every arithmetic mode, whichever path a refresh takes.  The
engine's tables must survive full-inference calls in between, and a refresh must leave training bit-identical."""
import numpy as np
import pytest
import torch

from test_gpu_full_inference import _features, _graph, _model
from test_gpu_full_inference_sharded import DEGS, HUB, _skewed

pytestmark = pytest.mark.gpu
MODES = ["fp32", "tf32", "fp16", "bf16"]
DTYPE = {"fp32": torch.float32, "tf32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}


def _ogl():
    import ogl_b200
    return ogl_b200


def _mode(name):
    o = _ogl()
    return {"fp32": o.OGL_F32, "bf16": o.OGL_BF16, "tf32": o.OGL_TF32, "fp16": o.OGL_FP16}[name]


# ----------------------------------------------------------------------------------------------------------- 0. row-list pool GEMM
@pytest.mark.parametrize("mode", MODES)
def test_pool_rows_are_the_rows_of_the_whole_table(mode):
    """the pool GEMM over m gathered rows gives the bits of the pool GEMM over all V rows, for m = 1, 3, 127, 129 and V, on layer 0
    (the feature table) and a hidden layer"""
    rng = np.random.default_rng(0)
    V, dims = 1000, (50, 24, 24, 5)
    _, _, f = _features(V, dims[0], mode)
    g = _graph(V, rng.integers(0, V, 4000), rng.integers(0, V, 4000))
    _, _, plan = _model(dims, mode, V)
    h = plan.hidden_table(0, V)
    h.copy_(torch.relu(torch.randn(h.shape, device="cuda")).to(h.dtype))
    if mode == "tf32":
        h.copy_(_ogl().native.round_tf32(h))
    for layer, hin in ((0, None), (1, h)):
        whole = plan.pool_table(layer, V)
        plan.pool_rows(g, f, layer, hin, whole, row0=0, n=V)
        for m in (1, 3, 127, 129, V):
            rows = torch.as_tensor(rng.permutation(V)[:m], device="cuda")
            part = plan.pool_table(layer, V)
            plan.pool_rows(g, f, layer, hin, part, rows=rows)
            assert torch.equal(part[rows], whole[rows]), (layer, m)
        tail = plan.pool_table(layer, V)
        plan.pool_rows(g, f, layer, hin, tail, row0=V - 129, n=129)
        assert torch.equal(tail[V - 129:V], whole[V - 129:V]) and not tail[:V - 129].any()


# ----------------------------------------------------------------------------------------------------------- 1. out-frontier
def _ref_out_frontier(g, rows):
    indptr, indices, _ = g.export_csr()
    V = indptr.numel() - 1
    r = rows[(rows >= 0) & (rows < V)]
    deg = indptr[1:] - indptr[:-1]
    dst = torch.repeat_interleave(torch.arange(V, device="cuda"), deg)
    hit = dst[torch.isin(indices, r)]
    ref = torch.unique(torch.cat([r, hit]))
    return ref, int((deg[ref] + 1).sum())


def _check_out(g, rows, what):
    t = torch.as_tensor(rows, dtype=torch.int64, device="cuda")
    got, cost = g.out_frontier(t)
    ref, rcost = _ref_out_frontier(g, t)
    assert torch.equal(got, ref) and cost == rcost, what


def test_out_frontier_matches_torch():
    ogl_b200 = _ogl()
    rng = np.random.default_rng(3)
    g = _skewed()
    V = g.num_vertices
    # an isolated vertex: no in- or out-edges
    indptr, indices, _ = g.export_csr()
    deg = (indptr[1:] - indptr[:-1]).cpu()
    outdeg = torch.bincount(indices.cpu(), minlength=V)
    iso = torch.nonzero((deg == 0) & (outdeg == 0)).flatten().tolist()
    lists = {
        "duplicates, hub": [HUB, 0, 0, 5, HUB, 17, 17, 17] + rng.integers(0, V, 40).tolist(),
        "scattered": rng.permutation(V)[:700].tolist() + [8, 8, 7],
        "every vertex": list(range(V)),
        "isolated": iso[:3] + [0],
        "empty": [],
        "out of range": [-1, V, V + 7, 3, 2**40, 3],
    }
    for what, rows in lists.items():
        _check_out(g, rows, what)
    # asymmetric by construction: u -> v only
    a = _graph(50, np.array([1, 2, 3, 3, 40]), np.array([2, 3, 4, 4, 41]))
    assert a.out_frontier([2])[0].tolist() == [2, 3] and a.in_frontier([2])[0].tolist() == [1, 2]
    _check_out(a, [3, 45], "asymmetric")
    # a vertex-stream prefix
    src, dst = rng.integers(0, 900, 5000), rng.integers(0, 900, 5000)
    from oracle.graph import in_csr
    ip, ix, ei = in_csr(np.concatenate([src, dst]), np.concatenate([dst, src]), 900)
    p = ogl_b200.native.Graph(900, 2 * 5000 + 16)
    p.load_parent(ip, ix, ei)
    p.set_active_prefix(400)
    _check_out(p, rng.integers(0, 900, 30).tolist(), "prefix")


# ----------------------------------------------------------------------------------------------------------- 2. suffix max
def _ref_max(g, x):
    indptr, indices, _ = g.export_csr()
    V = indptr.numel() - 1
    deg = indptr[1:] - indptr[:-1]
    dst = torch.repeat_interleave(torch.arange(V, device="cuda"), deg)
    out = torch.zeros(V, x.shape[1], dtype=x.dtype, device="cuda")
    out = out.scatter_reduce(0, dst[:, None].expand(-1, x.shape[1]), x[indices], "amax", include_self=False)
    return torch.where((deg > 0)[:, None], out, torch.zeros((), dtype=x.dtype, device="cuda"))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_suffix_max_matches_torch(dtype):
    """stored row maxima folded with the edges appended since: rows that had no edges, new vertices, a row gaining 6,000 edges in one
    batch, rows relocated by their growth, and a compaction between batches; each step equals the whole-row max"""
    ogl_b200 = _ogl()
    rng = np.random.default_rng(4)
    V0, V1, W = 3000, 3400, 40
    g = ogl_b200.native.Graph(V1, 200000)
    g.insert_vertices(V0)
    x = torch.randn(V1, W, device="cuda").to(dtype)
    acc = torch.zeros(V1, W, dtype=dtype, device="cuda")
    prev = torch.zeros(V1, dtype=torch.int64, device="cuda")
    for b in range(6):
        if b == 3:
            g.insert_vertices(V1 - V0)
        if b == 4:
            g.compact()
        V = g.num_vertices
        n = 8000
        dst = rng.integers(0, V // 2, n)
        src = rng.integers(0, V, n)
        if b == 2:                       # one row gains > kSegmaxChunk (2048) edges in this batch
            dst[:6000] = 11
        if b == 3:                       # new vertices, some with edges
            dst[:500] = rng.integers(V0, V0 + 200, 500)
        g.insert_edges(torch.as_tensor(src).cuda(), torch.as_tensor(dst).cuda(), symmetric=False)
        deg = g.degrees()
        rows = torch.nonzero(deg != prev[:V]).flatten()
        if b == 3:
            rows = torch.unique(torch.cat([rows, torch.arange(V0, V1, device="cuda")]))
        g.segment_max_suffix(x, acc, rows, prev)
        prev[:V] = deg
        assert torch.equal(acc[:V], _ref_max(g, x[:V])), b
    assert g.stats()["relocations"] > 0 and int(prev[11]) > 6000


# ----------------------------------------------------------------------------------------------------------- 3. the engine
def _init():
    ogl_b200 = _ogl()
    GraphSAGE, _, _, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, -1)
    return GraphSAGE, act


def _engine_setup(mode, n_layers, V_cap=3000, F=20, H=16, C=4, dropout=0.0, seed=0):
    ogl_b200 = _ogl()
    GraphSAGE, act = _init()
    torch.manual_seed(seed)
    model = GraphSAGE(F, H, C, n_layers - 1, act, dropout, "pool").cuda()
    dg = ogl_b200.DeviceGraph(V_cap, 400000, F, mode=_mode(mode))
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((V_cap, F)).astype(np.float32)
    y = rng.integers(0, C, (V_cap, 1)).astype(np.int64)
    return model, dg, x, y, rng


def _add_nodes(dg, x, y, n):
    v0 = dg.number_of_nodes()
    dg.add_nodes(n, {"feat": x[v0:v0 + n], "target": y[v0:v0 + n]})


def _batches(dg, x, y, rng, V_cap):
    """8+ insert batches: symmetric and asymmetric, new vertices with and without edges, a hub that gains thousands of edges at once,
    rows relocated by their growth"""
    _add_nodes(dg, x, y, 1500)
    dg.add_edges(rng.integers(0, 1500, 6000), rng.integers(0, 1500, 6000), symmetric=True)
    yield "initial"
    dg.add_edges(np.array([3, 4]), np.array([5, 5]), symmetric=False)
    yield "two edges"
    dg.add_edges(rng.integers(0, 1500, 3000), np.full(3000, 7), symmetric=False)
    yield "hub gains 3000"
    _add_nodes(dg, x, y, 200)
    yield "new vertices without edges"
    dg.add_edges(rng.integers(0, 1700, 400), rng.integers(1500, 1700, 400), symmetric=True)
    yield "edges of the new vertices"
    _add_nodes(dg, x, y, 300)
    dg.add_edges(rng.integers(1700, 2000, 300), rng.integers(0, 2000, 300), symmetric=False)
    yield "new vertices with out-edges"
    dg.add_edges(rng.integers(0, 2000, 20), rng.integers(0, 2000, 20), symmetric=True)
    yield "a serving request"
    dg.add_edges(rng.integers(0, 2000, 30000), rng.integers(0, 2000, 30000), symmetric=True)
    yield "a batch over the threshold"
    dg.native.compact()
    dg.add_edges(rng.integers(0, 2000, 50), np.full(50, 7), symmetric=False)
    yield "after compaction"
    yield "nothing new"


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("n_layers", [1, 2, 3, 4])
def test_engine_equals_the_whole_graph_call_after_every_batch(mode, n_layers):
    ogl_b200 = _ogl()
    model, dg, x, y, rng = _engine_setup(mode, n_layers)
    eng = ogl_b200.inference.StreamingInference(model, dg)
    plan = model.inference_plan(dg)
    paths = set()
    for what in _batches(dg, x, y, rng, 3000):
        info = eng.refresh()
        paths |= {l["path"] for l in info["layers"]}
        V = dg.number_of_nodes()
        whole = plan.infer_full(dg.native, dg.features)
        assert torch.equal(eng.logits(), whole), what
        T = torch.as_tensor(rng.integers(0, V, 57), device="cuda")
        assert torch.equal(eng.logits(T), model.inference(dg, T)), what
        assert torch.equal(eng.predict(T), whole[T].argmax(1)), what
    assert dg.native.stats()["relocations"] > 0
    assert {"full", "suffix", "all"} <= paths and (n_layers == 1 or "frontier" in paths), paths


def test_engine_with_dropout_uses_eval_semantics():
    ogl_b200 = _ogl()
    model, dg, x, y, rng = _engine_setup("fp16", 2, dropout=0.5)
    eng = ogl_b200.inference.StreamingInference(model, dg)
    for what in _batches(dg, x, y, rng, 3000):
        assert torch.equal(eng.logits(), model.inference(dg)), what


# ----------------------------------------------------------------------------------------------------------- 4. vertex streams
@pytest.mark.parametrize("mode", ["fp32", "fp16"])
def test_vertex_stream_prefix_growth(mode):
    ogl_b200 = _ogl()
    from oracle.graph import in_csr
    model, dg, x, y, rng = _engine_setup(mode, 2, V_cap=1500)
    V, E = 1500, 6000
    src, dst = rng.integers(0, V, E), rng.integers(0, V, E)
    ip, ix, ei = in_csr(np.concatenate([src, dst]), np.concatenate([dst, src]), V)
    dg.native.load_parent(ip, ix, ei)
    dg.features.write(0, torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda())
    eng = ogl_b200.inference.StreamingInference(model, dg)
    paths = []
    for n in (300, 310, 500, 510, 900, 1500):
        dg.native.set_active_prefix(n)
        paths.append(eng.refresh()["layers"][0]["path"] if n > 300 else "full")
        assert torch.equal(eng.logits(), model.inference(dg)), n
    assert "rebuild" in paths, paths


def test_dynamic_graph_vertex_evolve():
    ogl_b200 = _ogl()
    from ogl_b200.graph.dynamic_graph_vertex import DynamicGraphVertex, ParentGraph
    rng = np.random.default_rng(5)
    V, E, F = 1200, 5000, 20
    pg = ParentGraph.from_undirected(rng.integers(0, V, E), rng.integers(0, V, E), V)
    pg.ndata["feat"] = rng.standard_normal((V, F)).astype(np.float32)
    pg.ndata["target"] = rng.integers(0, 4, (V, 1)).astype(np.int64)
    dyn = DynamicGraphVertex(pg, 6, list(range(V)))
    dyn.build(vertex_timestamps={v: int(t) for v, t in enumerate(rng.permutation(V))})
    GraphSAGE, act = _init()
    torch.manual_seed(1)
    model = GraphSAGE(F, 16, 4, 1, act, 0.0, "pool").cuda()
    eng = ogl_b200.inference.StreamingInference(model, dyn.get_graph())
    for _ in range(5):
        assert torch.equal(eng.logits(), model.inference(dyn.get_graph()))
        dyn.evolve()
    assert torch.equal(eng.logits(), model.inference(dyn.get_graph()))


# ----------------------------------------------------------------------------------------------------------- 5. path selection
def _stages(plan, fn):
    plan.profile(True)
    out = fn()
    stages, _, _ = plan.profile_read()
    plan.profile(False)
    return out, {k for k, (_, launches) in stages.items() if launches > 0}


def test_paths_from_the_profile():
    ogl_b200 = _ogl()
    model, dg, x, y, rng = _engine_setup("tf32", 2)
    eng = ogl_b200.inference.StreamingInference(model, dg)
    plan = model.inference_plan(dg)
    _add_nodes(dg, x, y, 1500)
    dg.add_edges(rng.integers(0, 1500, 6000), rng.integers(0, 1500, 6000), symmetric=True)
    assert eng.refresh(full=False)["path"] == "full"

    def check():
        assert torch.equal(eng.logits(), plan.infer_full(dg.native, dg.features))

    dg.add_edges(np.array([1, 2, 3]), np.array([4, 4, 9]), symmetric=False)
    info, st = _stages(plan, eng.refresh)
    assert [l["path"] for l in info["layers"]] == ["suffix", "frontier"], info
    assert {"stream.l0.segmax_suffix", "stream.l0.out_gemm", "stream.l1.frontier", "stream.l1.pool_rows", "stream.l1.segmax",
            "stream.l1.out_gemm", "stream.l1.scatter"} <= st, st
    assert info["layers"][0]["rows"] == 2
    check()
    dg.add_edges(rng.integers(0, 1500, 20000), rng.integers(0, 1500, 20000), symmetric=True)
    info = eng.refresh()
    assert "all" in [l["path"] for l in info["layers"]], info
    check()
    # nothing changed: the degree read is the only launch of the library
    n0 = ogl_b200.kernel_launches()
    info, st = _stages(plan, eng.refresh)
    assert info["path"] == "none" and not st and ogl_b200.kernel_launches() - n0 == 1
    # full=True, a state_dict load, an Adam step of a training plan: full recomputes
    assert eng.refresh(full=True)["path"] == "full"
    check()
    sd = {k: v * 0.5 for k, v in model.state_dict().items()}
    model.load_state_dict(sd)
    assert eng.refresh()["path"] == "full"
    check()
    tp = model.plan_for(dg, [5, 5], 64)
    tp.train_step(dg.native, dg.features, torch.as_tensor(rng.permutation(1500)[:64], device="cuda"), loss_scale=1.0 / 64)
    model.mark_updated(tp)
    dg.add_edges(np.array([5]), np.array([6]), symmetric=False)
    assert eng.refresh()["path"] == "full"
    check()


# ----------------------------------------------------------------------------------------------------------- 6. isolation
def test_tables_survive_full_inference_calls():
    ogl_b200 = _ogl()
    model, dg, x, y, rng = _engine_setup("bf16", 3)
    eng = ogl_b200.inference.StreamingInference(model, dg)
    plan = model.inference_plan(dg)
    for i, what in enumerate(_batches(dg, x, y, rng, 3000)):
        eng.refresh()
        ref = eng.logits()
        V = dg.number_of_nodes()
        for name in ("full_h0", "full_h1"):
            try:
                plan.tensor(name).fill_(float("nan"))
            except RuntimeError:
                pass
        T = torch.as_tensor(rng.integers(0, V, 5), device="cuda")
        model.inference(dg, T)
        model.inference_loss(dg, T)
        assert torch.equal(eng.logits(), ref), what
        assert torch.equal(eng.logits(T), model.inference(dg, T)), what


def _train_run(mode, with_refresh, prefetch):
    ogl_b200 = _ogl()
    model, dg, x, y, rng = _engine_setup(mode, 2, V_cap=1500)
    _add_nodes(dg, x, y, 1500)
    dg.add_edges(rng.integers(0, 1500, 9000), rng.integers(0, 1500, 9000), symmetric=True)
    eng = ogl_b200.inference.StreamingInference(model, dg)
    plan = model.plan_for(dg, [6, 4], 64)
    batches = [torch.as_tensor(rng.permutation(1500)[:64], device="cuda") for _ in range(7)]
    losses = []
    for i, sd in enumerate(batches):
        per = torch.empty(64, device="cuda")
        if prefetch and i == 3:
            plan.prefetch(dg.native, dg.features, sd)
            if with_refresh:
                eng.refresh()
            plan.step_finish(dg.features, 1.0 / 64, per_vertex_out=per)
        else:
            plan.train_step(dg.native, dg.features, sd, loss_scale=1.0 / 64, per_vertex_out=per)
            if with_refresh and i in (2, 3):
                eng.refresh()
        losses.append(per)
    torch.cuda.synchronize()
    return torch.stack(losses), model._flat.clone()


@pytest.mark.parametrize("mode", ["fp16", "tf32"])
@pytest.mark.parametrize("prefetch", [False, True])
def test_refresh_leaves_training_bit_identical(mode, prefetch):
    l0, w0 = _train_run(mode, False, prefetch)
    l1, w1 = _train_run(mode, True, prefetch)
    assert torch.equal(l0, l1) and torch.equal(w0, w1)
