"""The refresh of inference.StreamingInference restated in torch on the CPU (no GPU): change detection from the in-degrees, the
C_{l+1} = C_l u N_out(C_l) rule, the suffix max of layer 0 and whole-row rebuilds after a prefix change, checked against the
from-scratch full_forward (tests/full_oracle.py) after every batch of a random asymmetric edge stream and of a growing vertex prefix.
Weights and features are small dyadic numbers, so every sum is exact in float64 and any mistake in the set algebra shows as a
mismatch, not as rounding."""
import numpy as np
import torch

from full_oracle import full_forward

THETA = 0.9


def _params(dims, rng):
    p = {}
    for i in range(len(dims) - 1):
        fi, fo = dims[i], dims[i + 1]
        for name, (o, k) in (("fc_pool", (fi, fi)), ("fc_self", (fo, fi)), ("fc_neigh", (fo, fi))):
            p[f"layers.{i}.{name}.weight"] = torch.from_numpy(rng.integers(-4, 5, (o, k)) / 8.0)
            p[f"layers.{i}.{name}.bias"] = torch.from_numpy(rng.integers(-4, 5, o) / 8.0)
    return p


def _csr(adj):
    deg = [len(a) for a in adj]
    indptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64)
    indices = np.array([u for a in adj for u in a], dtype=np.int64)
    return indptr, indices


class HostEngine:
    """the refresh of StreamingInference over python adjacency lists (row v = its in-edge sources in row order)"""

    def __init__(self, params, dims, v_cap):
        self.p, self.L = params, len(dims) - 1
        self.hp = [torch.zeros(v_cap, dims[l], dtype=torch.float64) for l in range(self.L)]
        self.h = [None] + [torch.zeros(v_cap, dims[l], dtype=torch.float64) for l in range(1, self.L)]
        self.neigh0 = torch.zeros(v_cap, dims[0], dtype=torch.float64)
        self.logits = torch.zeros(v_cap, dims[-1], dtype=torch.float64)
        self.deg = np.zeros(v_cap, dtype=np.int64)
        self.n, self.rebuilds = 0, 0
        self.paths = []

    def _w(self, l, name):
        return self.p[f"layers.{l}.{name}"]

    def _pool(self, l, x, rows):
        self.hp[l][rows] = torch.relu(x[rows] @ self._w(l, "fc_pool.weight").t() + self._w(l, "fc_pool.bias"))

    def _max(self, l, adj, v, e0=0, base=None):
        src = adj[v][e0:]
        m = self.hp[l][src].amax(0) if src else None
        if base is None:
            return m if m is not None else torch.zeros(self.hp[l].shape[1], dtype=torch.float64)
        return base if m is None else torch.maximum(base, m)

    def _out(self, l, x, rows, neigh):
        o = x[rows] @ self._w(l, "fc_self.weight").t() + neigh @ self._w(l, "fc_neigh.weight").t() + \
            (self._w(l, "fc_self.bias") + self._w(l, "fc_neigh.bias"))
        if l < self.L - 1:
            self.h[l + 1][rows] = torch.relu(o)
        else:
            self.logits[rows] = o

    def refresh(self, adj, x, rebuilds):
        V = len(adj)
        E = sum(len(a) for a in adj)
        deg = np.array([len(a) for a in adj], dtype=np.int64)
        Vp = self.n
        path = []
        if Vp == 0 or V < Vp:
            C = list(range(V))
            wide = True
            self._pool(0, x, C)
            self.neigh0[C] = torch.stack([self._max(0, adj, v) for v in C])
            path.append("full")
        else:
            C = sorted(set(np.nonzero(deg[:Vp] != self.deg[:Vp])[0].tolist()) | set(range(Vp, V)))
            if not C:
                self.paths.append(["none"])
                return
            self._pool(0, x, list(range(Vp, V)))
            wide = sum(deg[v] + 1 for v in C) > THETA * (E + V)
            if wide:
                C = list(range(V))
                self.neigh0[C] = torch.stack([self._max(0, adj, v) for v in C])
                path.append("all")
            elif rebuilds != self.rebuilds:
                self.neigh0[C] = torch.stack([self._max(0, adj, v) for v in C])
                path.append("rebuild")
            else:                                                # the suffix: edges [deg_prev, deg); deg_prev == 0 replaces
                self.neigh0[C] = torch.stack([self._max(0, adj, v, self.deg[v], self.neigh0[v] if self.deg[v] > 0 else None)
                                              for v in C])
                path.append("suffix")
        self._out(0, x, C, self.neigh0[C])
        for l in range(1, self.L):
            if wide:
                C2 = list(range(V))
            else:
                inC = set(C)
                C2 = sorted(inC | {v for v in range(V) if any(u in inC for u in adj[v])})     # C u N_out(C)
                wide = sum(deg[v] + 1 for v in C2) > THETA * (E + V)
                if wide:
                    C, C2 = list(range(V)), list(range(V))
            self._pool(l, self.h[l], C)
            self._out(l, self.h[l], C2, torch.stack([self._max(l, adj, v) for v in C2]))
            path.append("all" if wide else "frontier")
            C = C2
        self.deg[:V] = deg
        self.deg[V:] = 0
        self.n, self.rebuilds = V, rebuilds
        self.paths.append(path)


def _check(eng, adj, x, params):
    ip, ix = _csr(adj)
    ref = full_forward(params, ip, ix, x[:len(adj)])
    assert torch.equal(eng.logits[:len(adj)], ref)


def test_refresh_of_an_asymmetric_edge_stream():
    rng = np.random.default_rng(0)
    dims, V_cap = (6, 5, 4, 3), 120
    params = _params(dims, rng)
    x = torch.from_numpy(rng.integers(-3, 4, (V_cap, dims[0])).astype(np.float64))
    eng = HostEngine(params, dims, V_cap)
    adj = [[] for _ in range(40)]
    for b in range(14):
        if b in (3, 7):
            adj += [[] for _ in range(20)]                       # new vertices, with and without edges later
        V = len(adj)
        n = [3, 1, 6, 30, 2, 0, 5, 400, 4, 1, 2, 8, 1, 3][b]
        for _ in range(n):
            u, v = rng.integers(0, V), rng.integers(0, V)
            adj[v].append(int(u))                                # appended: the suffix of the row
        if b == 9:
            adj[5] += [int(u) for u in rng.integers(0, V, 50)]   # one row gains many edges at once
        eng.refresh(adj, x, 0)
        _check(eng, adj, x, params)
    flat = {p for ps in eng.paths for p in ps}
    assert {"full", "suffix", "frontier", "all", "none"} <= flat, eng.paths


def test_refresh_of_a_growing_prefix():
    rng = np.random.default_rng(1)
    dims, V = (5, 4, 3), 90
    params = _params(dims, rng)
    x = torch.from_numpy(rng.integers(-3, 4, (V, dims[0])).astype(np.float64))
    parent = [[] for _ in range(V)]
    for _ in range(300):
        u, v = rng.integers(0, V, 2)
        parent[v].append(int(u))
        parent[u].append(int(v))
    eng = HostEngine(params, dims, V)
    for i, n in enumerate((20, 22, 40, 41, 70, 90)):
        adj = [[u for u in parent[v] if u < n] for v in range(n)]     # induced rows, in the parent's edge order
        eng.refresh(adj, x, i + 1)
        _check(eng, adj, x, params)
    assert any("rebuild" in p for p in eng.paths), eng.paths
