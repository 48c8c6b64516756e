"""Full-neighbourhood inference (DGL's model.inference): the CSR segment max against torch.scatter_reduce, the layer-wise logits
against the edge-list reference full_forward (tests/full_oracle.py), agreement with the sampled path where the two must agree, insertion-order independence,
no side effects on training state, vertex streams, errors, and the trainer / driver surface.

Tolerances as in test_gpu_sage.py: |a - b| <= rtol |b| + rtol max|b|."""
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import sage as osage
from oracle.graph import in_csr
from full_oracle import full_forward

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("fc_pool.weight", "fc_pool.bias", "fc_self.weight", "fc_self.bias", "fc_neigh.weight", "fc_neigh.bias")
DIMS = [((50, 24, 5), (6, 4)), ((166, 64, 2), (9, 9)), ((33, 7), (5,)), ((20, 16, 16, 3), (3, 3, 2))]


def close(a, b, rtol, what=""):
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    assert a.shape == b.shape, (what, a.shape, b.shape)
    scale = b.abs().max().item() if b.numel() else 0.0
    err = (a - b).abs()
    bad = err > rtol * b.abs() + rtol * scale + 1e-30
    assert not bad.any(), "%s: %d / %d elements off, max err %.3e at scale %.3e (rtol %g)" % (
        what, int(bad.sum()), a.numel(), err.max().item(), scale, rtol)


def _mode(name):
    import ogl_b200
    return {"fp32": ogl_b200.OGL_F32, "bf16": ogl_b200.OGL_BF16, "tf32": ogl_b200.OGL_TF32, "fp16": ogl_b200.OGL_FP16}[name]


def _flat(params, L):
    return torch.cat([params[f"layers.{i}.{n}"].reshape(-1).float() for i in range(L) for n in NAMES]).cuda()


def _model(dims, mode, V, seed=3, fanouts=None, max_seeds=8):
    import ogl_b200
    L = len(dims) - 1
    params = osage.xavier_params(dims[0], dims[1], dims[-1], L - 1, seed=seed)
    params = {k: v for k, v in params.items() if int(k.split(".")[1]) < L}      # (xavier_params always draws a head layer)
    flat = _flat(params, L)
    plan = ogl_b200.native.Plan(list(dims), list(fanouts or [2] * L), max_seeds, V, mode=_mode(mode), seed=11)
    plan.bind_params(flat, torch.zeros_like(flat))
    return params, flat, plan


def _features(V, F, mode, seed=5):
    import ogl_b200
    rng = np.random.default_rng(seed)
    x = torch.from_numpy(rng.standard_normal((V, F)).astype(np.float32))
    y = torch.from_numpy(rng.integers(0, 3, V).astype(np.int64))
    f = ogl_b200.native.Features(V, F, _mode(mode))
    f.write(0, x.cuda(), y.cuda())
    return x, y, f


def _graph(V, src, dst, batches=1, symmetric=False):
    import ogl_b200
    g = ogl_b200.native.Graph(V, 2 * len(src) + 16)
    g.insert_vertices(V)
    for s, d in zip(np.array_split(src, batches), np.array_split(dst, batches)):
        g.insert_edges(torch.as_tensor(s).cuda(), torch.as_tensor(d).cuda(), symmetric=symmetric)
    return g


def _ref_segmax(g, x):
    indptr, indices, _ = g.export_csr()
    V = indptr.numel() - 1
    dst = torch.repeat_interleave(torch.arange(V, device="cuda"), indptr[1:] - indptr[:-1])
    ref = torch.zeros(V, x.shape[1], dtype=x.dtype, device="cuda")
    return ref.scatter_reduce(0, dst[:, None].expand(-1, x.shape[1]), x[indices], "amax", include_self=False)


# ----------------------------------------------------------------------------------------------------------- 1. the kernel
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("width", [64, 600])
def test_segment_max_is_exact_on_a_streamed_skewed_graph(dtype, width):
    """in-degrees 0 .. 120000 (the hub takes the chunk-and-combine path), the graph grown by several streaming batches so that rows
    relocated to the pool top and per-snapshot tails are read in place; all rows and a scattered row list with duplicates"""
    rng = np.random.default_rng(1)
    V = 6000
    degs = [0, 1, 31, 32, 33, 255, 256, 1000, 5000, 120000]
    dst = np.concatenate([np.full(d, v) for v, d in enumerate(degs)] + [rng.integers(len(degs), V, 30000)]).astype(np.int64)
    src = rng.integers(0, V, dst.size).astype(np.int64)
    perm = rng.permutation(dst.size)
    g = _graph(V, src[perm], dst[perm], batches=7)
    assert g.stats()["relocations"] > 0
    assert g.degrees()[:len(degs)].tolist() == degs
    x = torch.randn(V, width, device="cuda").to(dtype)
    ref = _ref_segmax(g, x)
    got = g.segment_max(x)
    assert got.shape == ref.shape and bool((got == ref).all())
    rows = torch.as_tensor(np.concatenate([rng.permutation(V)[:700], [9, 9, 8, 0, 0, 7, 9]]), device="cuda")
    rows = rows[torch.randperm(rows.numel(), device="cuda")]
    got_r = g.segment_max(x, rows)
    assert bool((got_r == ref[rows]).all())
    assert torch.equal(g.segment_max(x, rows), got_r)


# ----------------------------------------------------------------------------------------------------------- 2. logits vs the oracle
def _oracle_case(dims, mode, V=1500, E=9000, isolated=40, seed=3):
    rng = np.random.default_rng(seed)
    src = rng.integers(0, V - isolated, E).astype(np.int64)
    dst = rng.integers(0, V - isolated, E).astype(np.int64)
    g = _graph(V, src, dst, symmetric=True)
    ip, ix, _ = in_csr(np.concatenate([src, dst]), np.concatenate([dst, src]), V)
    x, y, f = _features(V, dims[0], mode, seed=seed)
    return g, np.asarray(ip), np.asarray(ix), x, f


@pytest.mark.parametrize("mode", ["fp32", "tf32", "fp16", "bf16"])
@pytest.mark.parametrize("dims,fanouts", DIMS)
def test_logits_match_the_full_oracle(mode, dims, fanouts):
    V = 1500
    g, ip, ix, x, f = _oracle_case(dims, mode, V=V)
    params, flat, plan = _model(dims, mode, V, fanouts=fanouts)
    logits = plan.infer_full(g, f)
    ref = full_forward(params, ip, ix, x.double())
    seeds = torch.as_tensor(np.concatenate([np.random.default_rng(0).permutation(V)[:200], [V - 1, V - 2, 5, 5]]), device="cuda")
    logits_s = plan.infer_full(g, f, seeds)
    sidx = seeds.cpu()
    if mode == "fp32":
        close(logits, ref, 1e-5, "logits")
        close(logits_s, ref[sidx], 1e-5, "seed logits")
    else:
        refq = full_forward(params, ip, ix, x.double(), quant=mode)
        close(logits, refq, 1e-3, "logits vs the quantised oracle")
        close(logits_s, refq[sidx], 1e-3, "seed logits vs the quantised oracle")
        if mode != "bf16":
            close(logits, ref, 1e-3, "logits vs the unquantised oracle")
    assert bool(torch.isfinite(logits).all())


# ----------------------------------------------------------------------------------------------------------- 3. sampled == full
@pytest.mark.parametrize("mode", ["fp32", "tf32", "fp16", "bf16"])
def test_sampled_eval_equals_full_when_every_in_degree_is_0_or_1(mode):
    """with in-degree <= 1 every sampled slot is the one in-neighbour (or none): the sampled and the full neighbourhood coincide"""
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
    sampled = torch.empty(seeds.numel(), dims[-1], device="cuda")
    plan.eval_step(g, f, seeds, logits_out=sampled)
    full = plan.infer_full(g, f, seeds)
    scale = sampled.abs().max().item()
    assert (full - sampled).abs().max().item() <= 1e-6 * scale
    print("%s: sampled and full logits bit-identical: %s" % (mode, torch.equal(full, sampled)))


# ----------------------------------------------------------------------------------------------------------- 4. order independence
@pytest.mark.parametrize("mode", ["fp32", "tf32", "fp16", "bf16"])
def test_logits_are_independent_of_insertion_order_and_reproducible(mode):
    rng = np.random.default_rng(5)
    V, dims = 2000, (40, 32, 32, 6)
    src = np.concatenate([rng.integers(0, V, 20000), rng.integers(0, V, 5000)]).astype(np.int64)
    dst = np.concatenate([rng.integers(0, V - 30, 20000), np.full(5000, 17)]).astype(np.int64)      # vertex 17: a hub
    perm = rng.permutation(src.size)
    streamed = _graph(V, src[perm], dst[perm], batches=50)
    assert streamed.stats()["relocations"] > 0
    once = _graph(V, src, dst)
    _, _, f = _features(V, dims[0], mode)
    _, _, plan = _model(dims, mode, V)
    a = plan.infer_full(streamed, f)
    b = plan.infer_full(once, f)
    assert torch.equal(a, b)
    assert torch.equal(plan.infer_full(streamed, f), a)


# ----------------------------------------------------------------------------------------------------------- 5. no side effects
def _train_run(mode, with_infer, prefetch):
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
            if with_infer:
                plan.infer_full(g, f)
            plan.step_finish(f, 1.0 / B, per_vertex_out=per)
        else:
            plan.train_step(g, f, sd, loss_scale=1.0 / B, per_vertex_out=per)
            if with_infer and not prefetch and i == 3:
                plan.infer_full(g, f, sd)
        losses.append(per)
    torch.cuda.synchronize()
    return torch.stack(losses), flat.clone()


@pytest.mark.parametrize("mode", ["fp16", "tf32"])
@pytest.mark.parametrize("prefetch", [False, True])
def test_infer_full_leaves_training_bit_identical(mode, prefetch):
    """train_step x k -> infer_full -> train_step x k: the per-step losses (Philox sampling, Adam step counter and moments feed them)
    and the final weights equal those of the same run without the call; also with a prefetched minibatch pending across it"""
    l0, w0 = _train_run(mode, False, prefetch)
    l1, w1 = _train_run(mode, True, prefetch)
    assert torch.equal(l0, l1) and torch.equal(w0, w1)


def test_model_inference_tracks_the_updated_weights():
    import ogl_b200
    rng = np.random.default_rng(7)
    V, E, F, H, C = 900, 6000, 12, 16, 3
    src, dst = rng.integers(0, V, E), rng.integers(0, V - 20, E)
    x = rng.standard_normal((V, F)).astype(np.float32)
    y = rng.integers(0, C, (V, 1)).astype(np.int64)
    dg = ogl_b200.DeviceGraph(V, 2 * E, F, mode=ogl_b200.OGL_F32)
    dg.add_nodes(V, {"feat": x, "target": y})
    dg.add_edges(src, dst, symmetric=True)
    GraphSAGE, _, _, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, -1)
    torch.manual_seed(3)
    model = GraphSAGE(F, H, C, 1, act, 0.5, "pool").cuda()
    ip, ix, _ = in_csr(np.concatenate([src, dst]), np.concatenate([dst, src]), V)

    def oracle():
        p = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
        return full_forward(p, np.asarray(ip), np.asarray(ix), torch.from_numpy(x).double())

    before = model.inference(dg)
    close(before, oracle(), 1e-5, "logits at the initial weights")
    plan = model.plan_for(dg, [5, 5], 64)
    for _ in range(3):
        plan.train_step(dg.native, dg.features, torch.as_tensor(rng.permutation(V)[:64], device="cuda"), loss_scale=1.0 / 64)
        model.mark_updated(plan)
    after = model.inference(dg)
    assert not torch.equal(before, after)
    close(after, oracle(), 1e-5, "logits at the trained weights")
    some = torch.as_tensor([3, 0, V - 1, 3], device="cuda")
    assert torch.equal(model.inference(dg, some), after[some])


# ----------------------------------------------------------------------------------------------------------- 6. vertex streams
def test_vertex_stream_prefix():
    import ogl_b200
    rng = np.random.default_rng(8)
    V, E, n_active, dims = 1200, 6000, 700, (20, 16, 4)
    src, dst = rng.integers(0, V, E), rng.integers(0, V, E)
    es, ed = np.concatenate([src, dst]), np.concatenate([dst, src])
    ip, ix, ei = in_csr(es, ed, V)
    g = ogl_b200.native.Graph(V, 2 * E + 16)
    g.load_parent(ip, ix, ei)
    g.set_active_prefix(n_active)
    x, _, f = _features(V, dims[0], "fp32")
    params, _, plan = _model(dims, "fp32", V)
    logits = plan.infer_full(g, f)
    assert logits.shape == (n_active, dims[-1])
    keep = (es < n_active) & (ed < n_active)
    pp, px, _ = in_csr(es[keep], ed[keep], n_active)
    close(logits, full_forward(params, np.asarray(pp), np.asarray(px), x[:n_active].double()), 1e-5, "prefix logits")


# ----------------------------------------------------------------------------------------------------------- 7. errors
def test_errors():
    import ogl_b200
    rng = np.random.default_rng(9)
    V, dims = 500, (20, 16, 4)
    g = _graph(V, rng.integers(0, V, 3000), rng.integers(0, V, 3000), symmetric=True)
    _, _, f = _features(V, dims[0], "fp16")
    _, _, plan = _model(dims, "fp16", V)
    assert plan.error_flags() == 0
    out = plan.infer_full(g, f, torch.as_tensor([1, V + 5, -1, 2], device="cuda"))
    assert plan.error_flags() & 1
    assert bool(torch.isfinite(out).all())
    for bad in (ogl_b200.native.Features(V, dims[0] + 1, ogl_b200.OGL_FP16), ogl_b200.native.Features(V, dims[0], ogl_b200.OGL_BF16)):
        with pytest.raises(ogl_b200.OglError, match="feature store"):
            plan.infer_full(g, bad)
    shard = _graph(V, rng.integers(0, V, 100), rng.integers(0, V, 100))
    shard.set_source_bound(4 * V)
    with pytest.raises(ogl_b200.OglError, match="shard"):
        plan.infer_full(shard, f)
    with pytest.raises(ogl_b200.OglError, match="shard"):
        shard.segment_max(torch.zeros(V, 8, dtype=torch.float16, device="cuda"))


# ----------------------------------------------------------------------------------------------------------- 8. surface
def test_trainer_full_evaluation_writes_rows(tmp_path):
    import ogl_b200
    from ogl_b200 import config
    from ogl_b200.graph import train_test_graph as ttg
    config.set_faithful(True)
    config.set_precision("fp16")
    old = ttg.SIZE_BUFFER
    ttg.SIZE_BUFFER = 1 << 12
    try:
        random.seed(1)
        np.random.seed(1)
        torch.manual_seed(1)
        rng = np.random.default_rng(1)
        V, E, F, C, H, snapshots, delta = 800, 6000, 12, 3, 16, 8, 2
        y = rng.integers(0, C, V)
        src, dst = rng.integers(0, V, E), rng.integers(0, V, E)
        order = {}
        for v in np.stack([src, dst], 1).reshape(-1).tolist():
            order.setdefault(v, len(order))
        perm = np.array(sorted(order, key=order.get), dtype=np.int64)
        m = np.full(V, -1, dtype=np.int64)
        m[perm] = np.arange(len(perm))
        src, dst = m[src], m[dst]
        x = rng.standard_normal((len(perm), F)).astype(np.float32)
        y = y[perm].reshape(-1, 1).astype(np.int64)
        x[np.arange(len(perm)), y[:, 0] % F] += 1.5
        GraphSAGE, RandomT, _, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, -1)
        labelled = set(range(len(perm)))
        dyn = ogl_b200.DynamicGraphEdge(snapshots, labelled)
        dyn.build(x, y, edge_timestamps={"src": src, "dst": dst})
        dyn_test = ogl_b200.DynamicGraphEdge(snapshots, labelled)
        dyn_test.build(x, y, edge_timestamps={"src": src, "dst": dst})
        for _ in range(delta):
            dyn_test.evolve()
        gu = ttg.TrainTestGraph(dyn, split=0.15, start_prior_alpha=4, end_prior_alpha=50, scale=1, max_priority=10)
        t = RandomT(GraphSAGE(F, H, C, 1, act, 0, "pool").cuda(), 10, 32, y, 5, cuda=True, batch_full=128, n_workers=0,
                    eval_neighbourhood="full")
        t.build_optimizer()
        out = str(tmp_path / "full.csv")
        scores = []
        for _ in range(4):
            t.train_timestep(gu)
            scores.append(t.evaluate(gu, out))
            t.evaluate_next_snapshots(dyn_test, delta, out, at_least=1)
            gu.evolve()
            dyn_test.evolve()
        rows = [r for r in open(out).read().strip().split("\n") if r]
        assert len(rows) >= 4 and all(r.split(";")[0] == "random" and len(r.split(";")) == 4 for r in rows)
        assert all(s is not None and 0.0 <= s <= 1.0 for s in scores)
        # the full-neighbourhood F1 is a property of the weights: evaluating twice gives the same score
        assert t.evaluate(gu, None) == t.evaluate(gu, None)
        with pytest.raises(ValueError):
            RandomT(GraphSAGE(F, H, C, 1, act, 0, "pool").cuda(), 1, 32, y, 5, cuda=True, eval_neighbourhood="exact")
    finally:
        ttg.SIZE_BUFFER = old


def test_driver_full_evaluation(tmp_path):
    def run(args):
        r = subprocess.run([sys.executable] + args, cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]

    data = str(tmp_path / "reddit")
    run(["tools/make_synthetic_dataset.py", "reddit", data, "--vertices", "1500", "--edges", "8000", "--feats", "24"])
    out = str(tmp_path / "res.csv")
    run(["train", "reddit", "pytorch", out, str(tmp_path / "tsne"), "--cuda", "--path", data, "--snapshots", "20", "--delta", "2",
         "--eval", "3", "--batch_timestep", "4", "--batch_size", "32", "--embedding_size", "16", "--samples", "5", "--train_offline", "4",
         "--epochs_offline", "1", "--batch_full", "256", "--max_timesteps", "12", "--eval_neighbourhood", "full"])
    rows = [l for l in open(out).read().strip().split("\n") if l]
    assert set(r.split(";")[0] for r in rows) == {"random", "prioritized", "no_rehersal", "offline"}
    assert all(len(r.split(";")) == 4 for r in rows)
    scored = [float(r.split(";")[1]) for r in rows if r.split(";")[1]]
    assert len(scored) >= 8 and all(0.0 <= s <= 1.0 for s in scored)
