"""Streaming inference on the GPU, in two forms.

`StreamingInference` keeps the exact full-neighbourhood logits of every vertex (what `GraphSAGE.inference` computes, bit for bit)
current as edges and vertices arrive: a refresh recomputes only the rows whose inputs changed since the last one (DESIGN.md 3e).

`CachedInference` is the drop-in for the per-request method of the reference's
TorchServe handler (`MNISTDigitClassifier.inference`, /root/reference/inference_optimized.py:144-301; SURVEY 8(f)-3), with its
approximations.

The serving graph lives in one streaming CSR of the C library that stores every edge in both directions (rows [0, V): in-edge
sources, rows [V, 2V): out-edge targets, whose degrees are the out-degrees); the
per-vertex caches h0proj / neigh0 / h1 / h1proj / neigh1 / h2, the feature table and the weights stay resident in HBM; the dense
row updates and the induced-subgraph mean are csrc/infer.cu kernels (fp32, as the reference serves).  The request's vertex sets are
tiny (bounded by the handler's out-degree threshold of 15) and the handler's ANSWER ORDER is CPython's set order, so the sets are
formed on the host from the few adjacency entries the device returns -- exactly as the reference forms them.

Every quirk of the handler is kept (reversed edge storage, mean instead of the training-time max, neigh rewritten for every vertex
of the predecessor set, out-degree filters, answer = cached h2 of the predecessor set); tests/test_gpu_inference.py checks this class
against oracle/inference.py, which is pinned to the reference's own code."""
import json

import numpy as np
import torch

from . import _native as native

TH = 15   # sampling_th (inference_optimized.py:184)


class CachedInference:
    def __init__(self, feat, state_dict, v_cap=None, e_cap=None):
        """feat: [V, F] dataset features (array / tensor); state_dict: `layers.{0,1}.{fc_pool,fc_self,fc_neigh}.{weight,bias}` as
        saved by the reference's export_model.py / GraphSAGE.state_dict()"""
        self.feat = torch.as_tensor(np.asarray(feat, dtype=np.float32) if not isinstance(feat, torch.Tensor) else feat).to("cuda", torch.float32).contiguous()
        V, F = self.feat.shape
        self.v_cap = int(v_cap or V)
        e_cap = int(e_cap or max(16 * self.v_cap, 1 << 16))
        self.w = {k: torch.as_tensor(np.asarray(v) if not isinstance(v, torch.Tensor) else v).detach().to("cuda", torch.float32).contiguous()
                  for k, v in state_dict.items() if k.startswith("layers.")}
        H = self.w["layers.0.fc_self.weight"].shape[0]
        C = self.w["layers.1.fc_self.weight"].shape[0]
        # ONE streaming CSR holds both directions: row v = sources of the stored edges u -> v, row v_cap + u = their targets
        # (degree of row v_cap + u = out-degree of u); a request's edges go in with one insert call
        self.g = native.Graph(2 * self.v_cap, 2 * e_cap)
        self.g.insert_vertices(2 * self.v_cap)
        self.cap_in, self.cap_out = 4096, 1024
        self._q = torch.zeros(5 + 3 * 256 + self.cap_in + 2 * self.cap_out, dtype=torch.int64, device="cuda")
        dims = dict(h0proj=F, neigh0=F, h1=H, h1proj=H, neigh1=H, h2=C)
        self.cache = {k: torch.zeros(self.v_cap, d, device="cuda") for k, d in dims.items()}
        self.member = torch.zeros(self.v_cap, dtype=torch.uint8, device="cuda")
        self.n = 0
        self.requests = 0

    def __len__(self):
        return self.n

    # ---- one request ---------------------------------------------------------------------------------------------
    def request(self, pairs):
        """pairs: [[a, b], ...] -> (P, classes): the vertices answered for (the handler's order) and their predicted classes"""
        vertices, total = set(), set()
        for a, b in pairs:
            vertices.add(a)
            total.add(a)
            total.add(b)
        n_new = max(total) + 1
        assert n_new <= self.v_cap, "vertex id %d beyond the feature table / capacity %d" % (n_new - 1, self.v_cap)
        self.n = max(self.n, n_new)                               # new vertices: zero caches (already), dataset feature rows (resident)
        pr = np.asarray(pairs, dtype=np.int64)
        a, b = pr[:, 0], pr[:, 1]
        # stored reversed, b -> a (:181-182): a's in-row gains b, b's out-row (row v_cap + b) gains a
        self.g.insert_edges(np.concatenate([b, a]), np.concatenate([a, b + self.v_cap]), symmetric=False)
        l_all = np.array(list(vertices), dtype=np.int64)
        v0, pred, succs = self._query(l_all)
        P = list(set(pred))
        S = list(set(succs))
        self.last_sets = (v0, P, S)
        c = self.cache
        for i, (nids, sub, x, proj, neigh, out) in enumerate(((v0, P, self.feat, "h0proj", "neigh0", "h1"), (S, S, c["h1"], "h1proj", "neigh1", "h2"))):
            if not nids:
                continue
            ids = torch.as_tensor(nids, dtype=torch.int64).cuda()
            L = "layers.%d." % i
            native.rows_linear(x, ids, self.w[L + "fc_pool.weight"], self.w[L + "fc_pool.bias"], c[proj], ids, relu=True)
            if sub:
                sub_t = ids if sub is nids else torch.as_tensor(sub, dtype=torch.int64).cuda()
                self.member[sub_t] = 1
                native.induced_mean(self.g, self.member, sub_t, c[proj], c[neigh])
                self.member[sub_t] = 0
            native.rows_linear(x, ids, self.w[L + "fc_self.weight"], self.w[L + "fc_self.bias"], c[out], ids, relu=(i < 1),
                               x2=c[neigh], ids2=ids, w2=self.w[L + "fc_neigh.weight"], b2=self.w[L + "fc_neigh.bias"])
        self.requests += 1
        if not P:
            return P, []
        classes = c["h2"][torch.as_tensor(P, dtype=torch.int64).cuda()].argmax(dim=1).cpu().tolist()
        return P, classes

    def _query(self, l_all):
        """(V0, pred, succs) of the request's vertices (inference_optimized.py:185-211): one launch + one D2H copy; the multi-call
        path takes over when a hub's rows exceed the scratch"""
        n = len(l_all)
        lv = torch.as_tensor(l_all).cuda()
        if n <= 256:
            native.infer_query(self.g, lv, self.v_cap, TH, self.cap_in, self.cap_out, self._q)
            q = self._q.cpu().numpy()
            if q[0] == 0:
                deg = q[3:3 + n]
                keep = l_all[deg < TH]
                base_in = 3 + n + 2 * (n + 1)
                pred = q[base_in:base_in + q[1]].tolist()
                base_out = base_in + self.cap_in
                dst = q[base_out:base_out + q[2]]
                dst_deg = q[base_out + self.cap_out:base_out + self.cap_out + q[2]]
                return list(set(keep.tolist())), pred, dst[dst_deg < TH].tolist()
        out_deg = self.g.row_degrees(lv + self.v_cap).cpu().numpy()
        keep = l_all[out_deg < TH]
        kv = torch.as_tensor(keep).cuda()
        _, succs = self.g.gather_rows(kv + self.v_cap)
        _, pred = self.g.gather_rows(kv)
        if succs.numel():
            succs = succs[self.g.row_degrees(succs + self.v_cap) < TH]
        return list(set(keep.tolist())), pred.cpu().tolist(), succs.cpu().tolist()

    # ---- the handler's call surface (inference_optimized.py:144, :304-318) --------------------------------------------
    def inference(self, data):
        value = json.loads(str(data[0].get("body")))
        _, classes = self.request(value)
        return [str(classes)]


# A layer's changed rows are recomputed on their own while they cost sum(in-degree + 1) <= _THETA * (E + V), the threshold of the
# plan's frontier inference (kFrontierTheta, csrc/plan.cu); above it that layer and every layer above it run over all rows.
_THETA = 0.9


class StreamingInference:
    """Exact full-neighbourhood logits of every vertex of `graph` (a DeviceGraph) under `model` (a GraphSAGE), kept current as the
    graph grows: after any edge / vertex insertions, `logits(T)` is torch.equal to `model.inference(graph, T)`.

    The engine owns per-vertex tables ([v_cap, pitch] each): every layer's pool rows hp_l = relu(h_l Wp + bp), the hidden outputs
    h_l, layer 0's neighbour max neigh0, the fp32 logits and the in-degree of every row at the last refresh.  A refresh finds the rows
    whose in-degree changed plus the new vertices (C_1), and, with frozen weights, recomputes only what depends on them:

    - layer 0: hp0 of the new vertices (an existing vertex's features and hence its hp0 never change); neigh0 of C_1 as the max of
      the stored row and the edges appended since (rows rebuilt by `set_active_prefix` / `load_parent` are recomputed whole), then the
      output rows of C_1;
    - layer l >= 1: hp_l of C_l, then C_{l+1} = C_l u N_out(C_l) (a row changes when its own input or an in-neighbour's did), whose
      segment max and output rows are recomputed.

    Max-pooling is exact and every GEMM row is computed on its own, so the tables hold the bits of the whole-graph call.  A layer
    whose set is too large (_THETA) runs over all rows instead; a weight change (detected through the model's version, as the
    model's plans detect it), a shrinking graph or `refresh(full=True)` recompute everything.

    Edges are assumed append-only and feature rows of existing vertices unchanged: after rewriting an existing vertex's features, call
    `refresh(full=True)`.  Evaluation semantics (no feat_drop).  The engine runs on the model's inference plan for `graph` and uses
    its full-inference workspace as scratch only: `model.inference` calls in between are harmless, and training state is untouched."""

    def __init__(self, model, graph):
        self.model, self.graph = model, graph
        self._n = 0                 # vertices at the last refresh
        self._version = None        # model._version at the last refresh
        self._rebuilds = 0          # graph.native.rebuilds at the last refresh
        self._tabs = False

    def _alloc(self, plan):
        cap, dims = self.graph.v_cap, plan.dims
        rows = (cap + 255) // 256 * 256
        pitch = lambda d: (d + 7) // 8 * 8
        self.hp = [plan.pool_table(l, cap) for l in range(plan.L)]
        self.h = [None] + [torch.zeros(rows, pitch(dims[l]), dtype=plan.dtype, device="cuda") for l in range(1, plan.L)]
        self.neigh0 = plan.pool_table(0, cap)
        self.table = torch.zeros(rows, pitch(dims[-1]), dtype=torch.float32, device="cuda")
        self.deg = torch.zeros(cap, dtype=torch.int64, device="cuda")
        self._tabs = True

    def _out(self, plan, l):
        return self.table if l == plan.L - 1 else self.h[l + 1]

    def _all_rows(self, plan, g, f, l, V, pool=True):
        h = self.h[l]
        if pool:
            plan.pool_rows(g, f, l, h, self.hp[l], row0=0, n=V)
        plan.stream_rows(g, f, l, h, self.hp[l], self._out(plan, l), row0=0, n=V, neigh=self.neigh0 if l == 0 else None)

    def refresh(self, full=False):
        """bring the logits of every vertex up to date with the graph and the weights.  -> dict(path = "none" | "incremental" |
        "full", layers = [dict(rows, edges, path) per layer]): the output rows each layer recomputed, their sum of (in-degree + 1),
        and how ("suffix" / "rebuild": layer 0 over its changed rows, "frontier": a higher layer over C_{l+1}, "all": every row after
        the set grew too large, "full": a full recompute)"""
        plan = self.model.inference_plan(self.graph)           # (brings the plan's weight shadows up to date)
        g, f = self.graph.native, self.graph.features
        if not self._tabs:
            self._alloc(plan)
        V, E, L = g.num_vertices, g.num_edges, plan.L
        deg = g.degrees()
        full = full or self._version != self.model._version or V < self._n or self._n == 0
        layers = []
        if V == 0:
            path = "none"
        elif full:
            if V < self._n:                  # rows past the graph stay zero, as the GEMMs' row tiles expect
                for t in self.hp + self.h[1:] + [self.neigh0, self.table]:
                    t[V:self._n].zero_()
            for l in range(L):
                self._all_rows(plan, g, f, l, V)
                layers.append(dict(rows=V, edges=E + V, path="full"))
            path = "full"
        else:
            Vp = self._n
            C = torch.cat([torch.nonzero(deg[:Vp] != self.deg[:Vp]).squeeze(1), torch.arange(Vp, V, device="cuda")])
            if C.numel() == 0:
                path = "none"
            else:
                path = "incremental"
                budget = _THETA * (E + V)
                if V > Vp:
                    plan.pool_rows(g, f, 0, None, self.hp[0], row0=Vp, n=V - Vp)
                cost = int((deg[C] + 1).sum())
                wide = cost > budget
                if wide:
                    self._all_rows(plan, g, f, 0, V, pool=False)
                    layers.append(dict(rows=V, edges=E + V, path="all"))
                else:
                    suffix = g.rebuilds == self._rebuilds
                    plan.stream_rows(g, f, 0, None, self.hp[0], self._out(plan, 0), rows=C, neigh=self.neigh0,
                                     neigh_mode=plan.NEIGH_SUFFIX if suffix else plan.NEIGH_SEGMAX, deg_prev=self.deg if suffix else None)
                    layers.append(dict(rows=C.numel(), edges=cost, path="suffix" if suffix else "rebuild"))
                for l in range(1, L):
                    if not wide:
                        C2, cost = plan.out_frontier(g, C, layer=l)
                        wide = cost > budget
                    if wide:
                        self._all_rows(plan, g, f, l, V)
                        layers.append(dict(rows=V, edges=E + V, path="all"))
                        continue
                    plan.pool_rows(g, f, l, self.h[l], self.hp[l], rows=C)
                    plan.stream_rows(g, f, l, self.h[l], self.hp[l], self._out(plan, l), rows=C2)
                    layers.append(dict(rows=C2.numel(), edges=cost, path="frontier"))
                    C = C2
        if path != "none" or V != self._n:
            self.deg[:V].copy_(deg)
            self.deg[V:].zero_()
        self._n, self._version, self._rebuilds = V, self.model._version, g.rebuilds
        return dict(path=path, layers=layers)

    def logits(self, vertices=None):
        """refresh, then a new fp32 [n, C] tensor of the logits of `vertices` (int64 ids; None: every vertex in id order)"""
        self.refresh()
        C = self.model.dims[-1]
        if vertices is None:
            return self.table[:self._n, :C].clone()
        v = torch.as_tensor(vertices, dtype=torch.int64).to("cuda").reshape(-1)
        if v.numel() and bool(((v < 0) | (v >= self._n)).any()):
            raise IndexError("StreamingInference.logits: vertex ids outside [0, %d)" % self._n)
        return self.table[v, :C]

    def predict(self, vertices=None):
        """the argmax class of each vertex's logits (int64, on the device)"""
        return self.logits(vertices).argmax(dim=1)
