"""GraphSAGE('pool') model (mirror of train/graphsage/pytorch/graphsage_dgl.py:6-59 + the DGL
SAGEConv('pool') it imports at :3).

Same constructor, same state_dict keys (`layers.{i}.{fc_pool,fc_self,fc_neigh}.{weight,bias}`,
cf. inference_optimized.py:135-139), but all parameters are views into ONE flat fp32 buffer that the
C library's fused kernels (csrc/plan.cu) read and update in place.  `edge_feats` / `pool_feats` are
accepted and ignored exactly like the reference (graphsage_dgl.py:41-46); `dropout` is SAGEConv's feat_drop.
"""
import math

import torch
import torch.nn as nn

from ... import config, parallel
from ..._native import Plan


class _Affine(nn.Module):
    """weight [out, in] + bias [out]; y = x W^T + b (nn.Linear layout)"""

    def __init__(self, in_feats, out_feats):
        super().__init__()
        self.in_features, self.out_features = in_feats, out_feats
        self.weight = nn.Parameter(torch.empty(out_feats, in_feats))
        self.bias = nn.Parameter(torch.empty(out_feats))
        nn.init.xavier_uniform_(self.weight, gain=nn.init.calculate_gain("relu"))
        bound = 1.0 / math.sqrt(in_feats)
        nn.init.uniform_(self.bias, -bound, bound)


def xavier_state_dict(in_feats, n_hidden, n_classes, n_layers, seed, dtype=torch.float32):
    """seeded state_dict with the initialisation of DGL's SAGEConv.reset_parameters [recalled]: Xavier-uniform weights with
    gain = calculate_gain('relu'), nn.Linear-default biases; keys as the reference's checkpoints (inference_optimized.py:135-139).
    Drawn from one seeded generator in float64 so that CPU and GPU runs (bench.py's two arms) start from the same values."""
    g = torch.Generator().manual_seed(seed)
    dims = [(in_feats, n_hidden)] + [(n_hidden, n_hidden)] * (n_layers - 1) + [(n_hidden, n_classes)]
    p = {}
    for i, (fi, fo) in enumerate(dims):
        for name, (o, k) in (("fc_pool", (fi, fi)), ("fc_self", (fo, fi)), ("fc_neigh", (fo, fi))):
            a = math.sqrt(2.0) * math.sqrt(6.0 / (o + k))
            p["layers.%d.%s.weight" % (i, name)] = ((torch.rand(o, k, generator=g, dtype=torch.float64) * 2 - 1) * a).to(dtype)
            b = 1.0 / math.sqrt(k)
            p["layers.%d.%s.bias" % (i, name)] = ((torch.rand(o, generator=g, dtype=torch.float64) * 2 - 1) * b).to(dtype)
    return p


class SAGEConv(nn.Module):
    """fc_pool: in->in, fc_self / fc_neigh: in->out.  out = fc_self(h_dst) + fc_neigh(max_nbr relu(fc_pool(h_src)))."""

    def __init__(self, in_feats, out_feats, aggregator_type="pool", feat_drop=0.0, activation=None):
        super().__init__()
        if aggregator_type != "pool":
            raise NotImplementedError("the reference driver always passes 'pool' (train/__main__.py:124)")
        self.in_feats, self.out_feats, self.activation, self.feat_drop = in_feats, out_feats, activation, feat_drop
        self.fc_pool = _Affine(in_feats, in_feats)
        self.fc_self = _Affine(in_feats, out_feats)
        self.fc_neigh = _Affine(in_feats, out_feats)


class _SageFn(torch.autograd.Function):
    """autograd bridge for the DGL-style call `model(blocks, x)` followed by loss.backward()"""

    @staticmethod
    def forward(ctx, x, model, plan, *params):
        plan.set_input(x)
        logits = plan.forward(None)
        ctx.model, ctx.plan = model, plan
        ctx.saved = (plan._stamp, plan._forwards)       # the plan keeps ONE set of activations: the ones backward must see
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        if (ctx.plan._stamp, ctx.plan._forwards) != ctx.saved:
            raise RuntimeError("GraphSAGE backward: the plan has run another forward pass or sampled another minibatch since this "
                               "output was computed, and it keeps only the latest activations; call backward before the next "
                               "model(blocks, x) or loader step")
        ctx.plan.backward(dlogits)
        grads = [g.clone() for g in ctx.model._grad_views]
        return (None, None, None) + tuple(grads)


class GraphSAGE(nn.Module):
    def __init__(self, in_feats, n_hidden, n_classes, n_layers, activation, dropout, aggregator_type,
                 edge_feats=None, pool_feats=None):
        super().__init__()
        # `dropout` becomes SAGEConv(feat_drop=dropout) (reference :41-46): dropout of every layer's input in training mode, done by
        # the plan with a Philox-keyed mask (csrc/sage_kernels.cu: k_feat_drop)
        self.dropout = float(dropout or 0.0)
        self.dims = [in_feats] + [n_hidden] * n_layers + [n_classes]
        self.layers = nn.ModuleList()
        for i in range(len(self.dims) - 1):
            last = i == len(self.dims) - 2
            self.layers.append(SAGEConv(self.dims[i], self.dims[i + 1], aggregator_type, feat_drop=dropout,
                                        activation=None if last else activation))
        self._plans = {}
        self._version = 0
        self._seen = ()
        self._flat = self._flat_grad = None
        self._grad_views = []
        self._flatten()

    # ---- flat parameter buffer ------------------------------------------------------------------
    def _ordered_params(self):
        for layer in self.layers:
            for fc in (layer.fc_pool, layer.fc_self, layer.fc_neigh):
                yield fc.weight
                yield fc.bias

    def _flatten(self):
        ps = list(self._ordered_params())
        dev = ps[0].device
        flat = torch.cat([p.detach().reshape(-1).to(torch.float32) for p in ps]).to(dev).contiguous()
        self._flat = flat
        self._flat_grad = torch.zeros_like(flat)
        self._grad_views = []
        off = 0
        for p in ps:
            n = p.numel()
            p.data = flat[off:off + n].view(p.shape)
            self._grad_views.append(self._flat_grad[off:off + n].view(p.shape))
            off += n
        for plan in self._plans.values():
            plan.bind_params(self._flat, self._flat_grad)
        self._version += 1
        self._seen = self._param_versions()

    def _apply(self, fn, *a, **k):
        super()._apply(fn, *a, **k)
        self._plans = {} if not self._flat.is_cuda else self._plans
        self._flatten()
        return self

    def load_state_dict(self, state_dict, strict=True, **kw):
        out = super().load_state_dict(state_dict, strict=strict, **kw)
        self.params_changed()
        return out

    def params_changed(self):
        """mark the parameters as modified outside the fused kernels.  In-place writes to the parameters themselves (a torch optimiser's
        step, p.copy_ under torch.no_grad()) are detected without it (_sync_params); this is for writes that bypass their version
        counters (through p.data or a raw pointer)"""
        self._version += 1

    def _param_versions(self):
        return tuple(p._version for p in self._ordered_params())

    def _sync_params(self):
        """an in-place write to a parameter (a torch optimiser's step, load_state_dict, ...) bumps its autograd version counter:
        if any moved since the last look, every plan's weight shadows are stale"""
        v = self._param_versions()
        if v != self._seen:
            self._seen = v
            self._version += 1

    # ---- plans ------------------------------------------------------------------------------------
    def plan_for(self, graph, hop_fanouts, max_seeds, gemm_impl=0):
        """The fused sampler+model workspace for `graph` (a DeviceGraph), created on first use."""
        if not self._flat.is_cuda:
            raise RuntimeError("ogl_b200 GraphSAGE must live on the GPU: call .cuda() (there is no CPU path)")
        self._sync_params()
        L = len(self.layers)
        hop_fanouts = list(hop_fanouts)[:L]
        if len(hop_fanouts) != L:
            raise ValueError("need one fan-out per layer (%d layers, got %r)" % (L, hop_fanouts))
        key = (id(graph), tuple(hop_fanouts), int(max_seeds), graph.mode, gemm_impl)
        plan = self._plans.get(key)
        if plan is None:
            plan = Plan(self.dims, hop_fanouts, max_seeds, graph.v_cap, mode=graph.mode, seed=config.seed(), gemm_impl=gemm_impl,
                        feat_drop=self.dropout)
            plan.bind_params(self._flat, self._flat_grad)
            plan._version = self._version
            self._plans[key] = plan
        elif plan._version != self._version:
            plan.refresh_params()
            plan._version = self._version
        return plan

    def inference(self, graph, vertices=None, distributed=False):
        """DGL's `model.inference(g, x)`: fp32 logits [n, C] on the device for `vertices` (int64 ids; None: every vertex of `graph`, a
        DeviceGraph) from their WHOLE in-neighbourhoods -- layer by layer over every vertex and every in-edge, no sampling, no
        feat_drop.  Exact max-pooling makes the result bit-reproducible and independent of edge-insertion order.  Runs on a plan of
        this model kept for `graph` (one full-inference workspace per model and graph); no training or sampled-evaluation state
        changes.  Ids outside the graph raise bit 0 of that plan's error_flags() (see inference_plan).
        distributed=True (data-parallel runs, torchrun): every rank computes its share of the rows (parallel.infer_full) and
        receives the others', so each rank returns the same, bit-identical logits.  It is a collective: every rank of the process
        group must make the call, which is why it is never switched on implicitly."""
        plan = self.inference_plan(graph)
        if distributed:
            return parallel.infer_full(plan, graph.native, graph.features, vertices)
        return plan.infer_full(graph.native, graph.features, seeds=vertices)

    def inference_loss(self, graph, vertices=None, distributed=False):
        """per-vertex cross-entropy losses (fp32 [n], on the device) of `inference`'s logits against the graph's labels: what PBR
        ranks its replay buffer by, from exact neighbourhoods.  The arithmetic of the training loss, so equal logits give bit-equal
        losses.  Ids outside the graph raise bit 0 of inference_plan(graph).error_flags(), labels outside [0, C) give NaN and raise
        bit 1.  distributed=True: each rank computes the losses of its share of the vertices and only the losses are exchanged
        (parallel.infer_full_loss); a collective, as for `inference`."""
        plan = self.inference_plan(graph)
        if distributed:
            return parallel.infer_full_loss(plan, graph.native, graph.features, vertices)
        return plan.infer_full_loss(graph.native, graph.features, seeds=vertices)

    def inference_plan(self, graph):
        """the plan `inference` runs on for `graph` (fan-out 1, one seed: only its weights and full-inference workspace are used)"""
        return self.plan_for(graph, [1] * len(self.layers), 1)

    def mark_updated(self, plan):
        """`plan` just ran its fused Adam step: its own shadows are fresh, the other plans' are stale"""
        self._version += 1
        plan._version = self._version

    # ---- DGL-style forward -----------------------------------------------------------------------
    def forward(self, blocks, x):
        plan = blocks[0]._plan
        if plan not in self._plans.values():
            raise RuntimeError("these blocks were not sampled by a plan of this model: build the loader with "
                               "NodeDataLoader(..., plan=model.plan_for(graph, hop_fanouts, batch_size))")
        if blocks[0]._stamp != plan._stamp:
            raise RuntimeError("stale blocks: the plan has sampled another minibatch since")
        self._sync_params()
        if plan._version != self._version:
            plan.refresh_params()
            plan._version = self._version
        plan.set_option("train_mode", int(self.training))      # feat_drop only in training mode, like nn.Dropout
        return _SageFn.apply(x, self, plan, *list(self._ordered_params()))
