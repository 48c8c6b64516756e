"""Host-side logic of the drop-in (no GPU): the TrainTestGraph / PrioritizedReplayBuffer mirrors must
reproduce the REFERENCE's own objects under the same `random` / numpy seeds (fixtures in tests/golden
were produced by /root/reference's code).  The GPU sum tree is replaced by an injected stand-in so that
only the host logic is exercised here; tests/test_gpu_*.py run the same checks on the real kernels."""
import random

import numpy as np
import pytest
import torch

from oracle.sumtree import SumTree as OracleTree
from oracle.graph import EdgeStreamOracle


class _TreeStandIn:
    """same surface as ogl_b200.native.SumTree, CPU arithmetic"""

    def __init__(self, cap):
        self.t = OracleTree(cap)
        self.capacity = cap

    def set(self, idx, val):
        self.t.set(np.asarray(idx, dtype=np.int64), np.asarray(val, dtype=np.float64))

    def values(self):
        return torch.from_numpy(self.t.value)

    def sum(self, lo, hi):
        return torch.tensor([self.t.sum(lo, hi)], dtype=torch.float64)

    def find(self, mass):
        return torch.from_numpy(self.t.find_prefixsum_idx(np.asarray(mass, dtype=np.float64)))

    def sample_stratified(self, u, n_items):
        n = len(u)
        p_total = self.t.sum(0, n_items - 1)
        every = p_total / n
        mass = [u[i] * every + i * every for i in range(n)]
        return self.find(mass)


class _FakeStream:
    """DynamicGraph interface over the oracle's edge stream (no device)"""

    def __init__(self, src, dst, snapshots, labelled):
        self.o = EdgeStreamOracle(src, dst, snapshots)
        self.labelled = labelled
        self.snapshots = snapshots

    @property
    def evolution_index(self):
        return self.o.evolution_index

    def __len__(self):
        return self.snapshots

    def get_graph(self):
        return None

    def evolve(self):
        self.o.evolve()

    def get_added_vertices(self, delta=None):
        v = set(self.o.new_vertices)
        return v, [x in self.labelled for x in v]

    def get_original_to_subgraph_map(self):
        return None

    def get_subgraph_to_original_map(self):
        return None


def test_prioritized_buffer_host_logic(golden):
    from ogl_b200.prioritized_replay.replay_buffer import PrioritizedReplayBuffer
    g = golden("replay_buffer")
    buf = PrioritizedReplayBuffer(int(g["size"]), float(g["alpha"]), float(g["max_p"]), float(g["min_p"]),
                                  tree_backend=_TreeStandIn, verbose=False)
    buf.add_all(dict(zip(g["nodes1"].tolist(), g["pri1"].tolist())))
    assert np.array_equal(buf._it_sum._t.t.value, g["leaves1"])
    buf.update_priorities(dict(zip(g["upd_nodes"].tolist(), g["upd_pri"].tolist())))
    assert np.array_equal(buf._it_sum._t.t.value, g["leaves2"])
    assert [buf.get_min_priority(), buf.get_max_priority(), buf._min_priority, buf._max_priority] == g["minmax"].tolist()
    buf.add_all(dict(zip(g["nodes2"].tolist(), [float(g["p2"])] * len(g["nodes2"]))))
    assert np.array_equal(buf._it_sum._t.t.value, g["leaves3"])
    random.seed(123)
    res = buf._sample_proportional(int(g["draw_n"]))
    assert sorted(res) == g["draw_result"].tolist()
    assert buf.dump_priorities(g["nodes1"][:5].tolist()) == [float(g["leaves3"][buf._it_sum._capacity + i]) for i in range(5)]


def test_train_test_graph_matches_reference(golden):
    from ogl_b200 import config
    from ogl_b200.graph import train_test_graph as ttg
    g = golden("train_test")
    config.set_faithful(True)
    ttg.SIZE_BUFFER = int(g["size_buffer"])
    labelled = set(g["labelled"].tolist())
    np.random.seed(1)
    random.seed(1)
    stream = _FakeStream(g["src"], g["dst"], int(g["snapshots"]), labelled)
    tt = ttg.TrainTestGraph(stream, split=0.15, start_prior_alpha=4, end_prior_alpha=50, scale=1, max_priority=10,
                            tree_backend=_TreeStandIn)
    unpad = lambda row: [int(x) for x in row if x >= 0]
    for k in range(8):
        assert len(tt.get_train_set()) == g["train_len"][k] and len(tt.get_test_set()) == g["test_len"][k]
        assert list(tt.draw_random_train_nodes(16)) == unpad(g["rbr"][k])
        pbr = list(tt.draw_priority_train_nodes(16))
        assert [int(x) for x in pbr] == unpad(g["pbr"][k])
        assert list(tt.get_new_train_nodes(5)) == unpad(g["newn"][k])
        tt.update_priorities({int(v): 0.1 + 0.01 * (int(v) % 37) for v in pbr})
        assert tt.prior_alpha == g["alpha"][k]
        assert [tt.priority_replay_buffer.get_min_priority(), tt.priority_replay_buffer.get_max_priority()] == g["minmax"][k].tolist()
        tt.evolve()
    assert tt.get_train_set() == g["final_train"].tolist() and tt.get_test_set() == g["final_test"].tolist()
    assert tt.dump_priorities(tt.get_train_set()) == g["final_priorities"].tolist()


def test_graphsage_module_surface():
    import ogl_b200
    m = ogl_b200.GraphSAGE(12, 16, 3, 1, torch.nn.functional.relu, 0, "pool", edge_feats=0, pool_feats=32)
    keys = list(m.state_dict().keys())
    assert keys == [f"layers.{i}.{fc}.{p}" for i in range(2) for fc in ("fc_pool", "fc_self", "fc_neigh") for p in ("weight", "bias")]
    assert m.layers[0].fc_pool.weight.shape == (12, 12)       # latent_dim ignored like the reference
    assert m.layers[0].fc_self.weight.shape == (16, 12) and m.layers[1].fc_neigh.weight.shape == (3, 16)
    # parameters are views of one flat buffer in the library's layout
    off = 0
    for p in m._ordered_params():
        assert p.data_ptr() == m._flat.data_ptr() + 4 * off
        off += p.numel()
    sd = {k: torch.randn_like(v) for k, v in m.state_dict().items()}
    m.load_state_dict(sd)
    assert torch.equal(m._flat[:144].view(12, 12), sd["layers.0.fc_pool.weight"])
    with pytest.raises(RuntimeError):
        m.plan_for(None, [5, 5], 8)                              # CPU model: no fallback


def test_utils_init_contract():
    import ogl_b200
    with pytest.raises(RuntimeError):
        ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, GPU=False)
    with pytest.raises(NotImplementedError):
        ogl_b200.init(ogl_b200.Lib_supported.TF, GPU=True)
    t = ogl_b200.utils.to_nn_lib(np.ones((2, 2)), GPU=False)
    assert t.dtype == torch.float32
    m = ogl_b200.utils.sparse1d(5)
    m[np.array([1, 3])] = np.array([7, 9])
    assert m[3] == 9 and m[np.array([1, 0])].tolist() == [7, 0]


def test_priority_strategies_match_reference(golden):
    """TrendPriority / HybridPriority vs the reference's own classes (fixture recorded with np.float restored)"""
    from ogl_b200.prioritized_replay.generate_priority import TrendPriority, HybridPriority, LossPriority
    g = golden("priority_strategies")
    V = int(g["V"])
    trend, hybrid = TrendPriority(V, alpha=0.85), HybridPriority(V, alpha=0.7, loss_contrib=0.4)
    for b, l, rt, rh in zip(g["nodes"], g["losses"], g["trend"], g["hybrid"]):
        assert np.array_equal(trend.get_priorities(b.tolist(), l.copy()), rt)
        assert np.array_equal(hybrid.get_priorities(b.tolist(), l.copy()), rh)
    assert trend.avg == float(g["trend_avg"]) and np.array_equal(trend.values, g["trend_values"])
    x = np.arange(3.0)
    assert LossPriority().get_priorities([0, 1, 2], x) is x


def test_cached_inference_oracle_edge_cases():
    """requests whose vertices are all above the handler's out-degree threshold (empty V0 / P / S), repeated pairs, self pairs"""
    from oracle.inference import CachedInferenceOracle, TH
    rng = np.random.default_rng(0)
    V, F, H, C = 40, 6, 5, 3
    feat = rng.standard_normal((V, F)).astype(np.float32)
    params = {}
    for l, (i, o) in enumerate(((F, H), (H, C))):
        for name, (oo, ii) in (("fc_pool", (i, i)), ("fc_self", (o, i)), ("fc_neigh", (o, i))):
            params["layers.%d.%s.weight" % (l, name)] = rng.standard_normal((oo, ii)).astype(np.float32)
            params["layers.%d.%s.bias" % (l, name)] = rng.standard_normal(oo).astype(np.float32)
    o = CachedInferenceOracle(feat, params)
    # vertex 0 becomes a hub: it is stored as the SOURCE of TH edges (pairs [x, 0] are stored as 0 -> x)
    P, cls = o.request([[x, 0] for x in range(1, TH + 1)])
    assert sorted(P) == [0] and len(cls) == 1                      # every a's only in-neighbour is the hub
    before = {k: v.copy() for k, v in o.cache.items()}
    P, cls = o.request([[0, 0]])                                   # the hub itself: out-degree TH + 1 -> filtered out, nothing to answer
    assert P == [] and cls == []
    for k in before:
        assert np.array_equal(before[k], o.cache[k][:len(before[k])]), k
    P, cls = o.request([[3, 4], [3, 4], [4, 3]])                   # parallel edges count twice in the mean
    assert set(P) == {0, 3, 4} and len(cls) == 3
    assert o.n == TH + 1


def test_pipeline_call_order_single_rank():
    """parallel.Pipeline on one rank: the next minibatch is prefetched BEFORE the current one is finished (that is what lets the
    two overlap), at most two are ever pending, and every minibatch is finished exactly once, in order"""
    import types
    import ogl_b200
    calls = []

    class FakePlan:
        tail_params, n_params = 4, 10

        def prefetch(self, graph, features, seeds):
            calls.append(("prefetch", seeds))

        def step_finish(self, features, scale, do_step=True, per_vertex_out=None, loss_sum_out=None):
            calls.append(("finish", scale, do_step))

    real_stream = ogl_b200.parallel.torch.cuda.current_stream
    real_event = ogl_b200.parallel.torch.cuda.Event
    ogl_b200.parallel.torch.cuda.current_stream = lambda: types.SimpleNamespace(wait_event=lambda e: None)
    ogl_b200.parallel.torch.cuda.Event = lambda *a, **k: types.SimpleNamespace(record=lambda s=None: None)
    try:
        pipe = ogl_b200.parallel.Pipeline(FakePlan(), "g", "f", None, 8)
        pipe.begin("s0")
        for t in range(3):
            pipe.finish("s%d" % (t + 1) if t < 2 else None)
        pipe.flush()
    finally:
        ogl_b200.parallel.torch.cuda.current_stream = real_stream
        ogl_b200.parallel.torch.cuda.Event = real_event
    assert calls == [("prefetch", "s0"), ("prefetch", "s1"), ("finish", 1.0 / 8, True), ("prefetch", "s2"), ("finish", 1.0 / 8, True),
                     ("finish", 1.0 / 8, True)]


def test_package_initialiser_equals_the_oracle_twin():
    """bench.py's two arms start from the same weights: the package's seeded Xavier initialiser and the oracle's are bit-identical"""
    import torch
    from oracle.sage import xavier_params
    from ogl_b200.graphsage.pytorch.graphsage_dgl import xavier_state_dict
    a, b = xavier_params(37, 16, 5, 2, seed=3), xavier_state_dict(37, 16, 5, 2, seed=3)
    assert a.keys() == b.keys()
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_oracle_tf32_rounding_matches_cvt_rna():
    import torch
    from oracle.sage import round_tf32
    x = torch.tensor([1.0, 1.0 + 2 ** -11, 1.0 + 2 ** -11 - 2 ** -20, -1.0 - 2 ** -11, 3.0e-30, 65504.0, 0.1])
    r = round_tf32(x)
    assert r[0] == 1.0 and r[1] == 1.0 + 2 ** -10 and r[2] == 1.0 and r[3] == -1.0 - 2 ** -10      # ties away from zero
    assert bool(((r.view(torch.int32) & 0x1FFF) == 0).all())
    assert float(((r - x).abs() / x.abs()).max()) <= 2 ** -11


def test_fp16_loss_scale_matches_the_oracle_model():
    """mode OGL_FP16 stores activation gradients times a power of two derived from the loss scale (csrc/plan.cu); oracle/sage.py rounds
    its gradients on the same grid: the two formulas must agree for every loss scale a trainer can pass (no device needed)"""
    from ogl_b200._lib import lib
    from oracle import sage as osage
    import random
    rng = random.Random(0)
    cases = [1.0, 0.5, 1.0 / 3, 1.0 / 96, 1.0 / 1024, 1.0 / 8192, 64.0, 65.0, 1e-7, 3e4] + [2.0 ** rng.uniform(-20, 10) for _ in range(500)]
    for a in cases:
        a = float(np.float32(a))
        gs = float(lib.ogl_fp16_grad_scale(a))
        assert gs == osage.grad_scale_for(a), (a, gs, osage.grad_scale_for(a))
        assert 32.0 < a * gs <= 64.0 and np.log2(gs) == int(np.log2(gs)), (a, gs)
    assert float(lib.ogl_fp16_grad_scale(0.0)) == 1.0 and float(lib.ogl_fp16_grad_scale(float("inf"))) == 1.0


def test_graphsage_notices_parameter_writes_outside_the_fused_kernels():
    """torch.optim updates the parameters in place through their views of the flat buffer and leaves the model alone: the model
    must see by itself that its plans' weight shadows are stale (every write bumps the parameter's autograd version)"""
    import torch
    import ogl_b200
    model = ogl_b200.GraphSAGE(6, 4, 3, 1, torch.nn.functional.relu, 0, "pool")
    v0 = model._version
    model._sync_params()
    assert model._version == v0, "nothing was written"
    for p in model.parameters():
        p.grad = torch.ones_like(p)
    torch.optim.Adam(model.parameters()).step()
    model._sync_params()
    assert model._version == v0 + 1, "an optimiser step was not noticed"
    model._sync_params()
    assert model._version == v0 + 1, "one step was counted twice"
    with torch.no_grad():
        model.layers[1].fc_neigh.bias[0] = 5.0
    model._sync_params()
    assert model._version == v0 + 2, "a single in-place write was not noticed"
