#!/usr/bin/env python
"""Benchmark of the streaming GraphSAGE-pool hot path (BASELINE.json metric: train target-vertices/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload reddit|elliptic|arxiv|pubmed]
                    [--dump-outputs DIR]

A "step" is one training minibatch of the workload: sample the 2-hop neighbourhood of B target vertices from the
streaming CSR (Philox, with replacement), compact the frontiers, gather the input feature rows, GraphSAGE-pool
forward, cross-entropy, backward, Adam.  `value` times K such steps with the seeds already in HBM; `e2e` times
the same K steps through the host API (pinned host seeds -> H2D inside the call, loss read back D2H every step).
Default workload = the Reddit-shaped synthetic graph north_star quotes its targets on (232,965 vertices,
~114.6 M directed edges, 602 features, 41 classes, hidden 600, B = 1024, fan-outs 25/10): it fits one B200
(~6 GB resident), so it is also the N = 1 workload; with N > 1 every rank holds a replica and trains its own
B-vertex shard of a global batch of N*B, gradients all-reduced over NCCL (weak scaling).

`--impl reference` times the CPU restatement of the reference's path (oracle/: numpy Philox sampler + to_block,
torch-CPU SAGEConv('pool') fwd/bwd + Adam) on the box's host cores: the reference itself cannot run here
(DGL is un-vendored, un-pinned and absent -- SURVEY 8(c)).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: V, stream edges, F, C, H, B, fanouts (seeds hop first), zipf exponent of the degree weights
    "reddit": dict(V=232965, E=57300000, F=602, C=41, H=600, B=1024, fanouts=[25, 10]),
    "elliptic": dict(V=203769, E=234355, F=166, C=2, H=256, B=32, fanouts=[45, 45]),
    "arxiv": dict(V=169343, E=1166243, F=128, C=40, H=32, B=32, fanouts=[40, 40]),
    "pubmed": dict(V=19717, E=44338, F=500, C=3, H=32, B=32, fanouts=[10, 10]),
}
EXCHANGE = ["peer"]
IMPL = ["ours"]
EXCHANGE_NAME = {"peer": "gradient sum over NVLink peer memory (P2P loads) fused with Adam in one kernel per bucket, no NCCL on the data path",
                 "nccl": "NCCL all-reduce + Adam"}
NAMES = ("fc_pool.weight", "fc_pool.bias", "fc_self.weight", "fc_self.bias", "fc_neigh.weight", "fc_neigh.bias")


# ----------------------------------------------------------------------------------------- synthetic data
def gen_edges(w, device, seed=1):
    """Chung-Lu style power-law stream: endpoints drawn with probability ~ (rank + 50)^-0.83 (degree exponent
    ~2.2), vertex ranks scattered by a fixed permutation.  Returns int64 (src, dst) of length E on `device`."""
    V, E = w["V"], w["E"]
    g = torch.Generator(device=device).manual_seed(seed)
    wt = (torch.arange(V, device=device, dtype=torch.float64) + 50.0) ** -0.83
    cdf = torch.cumsum(wt / wt.sum(), 0).float()
    perm = torch.randperm(V, generator=g, device=device)
    out = []
    for _ in range(2):
        parts = []
        for a in range(0, E, 1 << 24):
            n = min(1 << 24, E - a)
            u = torch.rand(n, generator=g, device=device)
            parts.append(perm[torch.searchsorted(cdf, u).clamp_(max=V - 1)])
        out.append(torch.cat(parts))
    return out[0], out[1]


def gen_features(w, device, seed=2):
    g = torch.Generator(device=device).manual_seed(seed)
    feats = torch.randn(w["V"], w["F"], generator=g, device=device, dtype=torch.float32)
    g3 = torch.Generator(device=device).manual_seed(seed + 1)
    labels = torch.randint(0, w["C"], (w["V"],), generator=g3, device=device, dtype=torch.int64)
    return feats, labels


def init_params(w, seed=0):
    """seeded Xavier init, the same values for both arms (the CPU arm takes the oracle's twin of the package's initialiser;
    tests/test_host_logic.py checks the two are bit-identical)"""
    if IMPL[0] == "reference":
        from oracle.sage import xavier_params
        return xavier_params(w["F"], w["H"], w["C"], 1, seed=seed)
    from ogl_b200.graphsage.pytorch.graphsage_dgl import xavier_state_dict
    return xavier_state_dict(w["F"], w["H"], w["C"], 1, seed=seed)


def seed_batches(w, n_batches, rank, world, seed=4):
    """target-vertex minibatches: uniform B-subsets of the 85 % train split (RBR draw), one per step per rank"""
    rng = np.random.default_rng(seed)
    train = rng.permutation(w["V"])[: int(0.85 * w["V"])]
    out = []
    for _ in range(n_batches):
        glob = rng.choice(train, size=w["B"] * world, replace=False)
        out.append(np.ascontiguousarray(glob[rank * w["B"]:(rank + 1) * w["B"]], dtype=np.int64))
    return out


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock, power and clock-event (throttle) reasons of one GPU, polled through NVML every ~2 ms on a background thread for
    the whole run: the timed region of the default run is ~10-20 ms long, which `nvidia-smi -lms 100` cannot sample at all."""
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake"}

    def __init__(self, index, period=0.002):
        self.rows, self.h, self.nv, self.period, self._stop = [], None, None, period, False
        try:
            import pynvml as nv
            nv.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
                self.h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.nv = nv
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
        except Exception as e:                    # no NVML: the line says so instead of carrying an empty record
            self.err = repr(e)[:200]
            self.h = None

    def _poll(self):
        nv = self.nv
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop:
            try:
                self.rows.append((time.time(), float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)), int(reasons_fn(self.h)),
                                  nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0))
            except Exception:
                pass
            time.sleep(self.period)

    def window(self, t0, t1):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "error": getattr(self, "err", "NVML unavailable")}
        rows = [r for r in self.rows if t0 <= r[0] <= t1]
        reasons = set()
        for r in rows:
            for bit, name in self.BITS.items():
                if r[2] & bit:
                    reasons.add(name)
        return {"sm_mhz": float(np.median([r[1] for r in rows])) if rows else None, "sm_min_mhz": min((r[1] for r in rows), default=None),
                "sm_max_mhz": self.max_mhz, "power_w_max": max((r[3] for r in rows), default=None), "reasons": sorted(reasons),
                "samples": len(rows), "period_ms": 1e3 * self.period, "source": "NVML polled in-process"}

    def stop(self):
        self._stop = True


# ----------------------------------------------------------------------------------------- CPU path (oracle)
class CpuPath:
    """The reference's CPU path restated (oracle/): DGL-style sampling + to_block in numpy, SAGEConv('pool') +
    CrossEntropy + Adam in torch-CPU fp32 (train/graphsage/pytorch/model.py:77-107 with cuda=False)."""

    def __init__(self, w, indptr, indices, feats, labels, params, seed=11):
        from oracle import sampler, sage
        self.w, self.sampler, self.sage = w, sampler, sage
        self.indptr, self.indices = indptr, indices
        self.feats, self.labels = feats, labels
        self.params = {k: v.clone().float().requires_grad_(True) for k, v in params.items()}
        self.opt = torch.optim.Adam(list(self.params.values()), lr=1e-3)
        self.seed, self.step_no = seed, 0

    def step(self, seeds):
        w = self.w
        input_nodes, blocks = self.sampler.sample_blocks(self.indptr, self.indices, self.indices, seeds, w["fanouts"], self.seed,
                                                         self.step_no, fast=True)
        self.step_no += 1
        ob = [dict(n_dst=len(b["dst_nodes"]), edge_src=torch.from_numpy(b["edge_src"]), fanout=b["fanout"]) for b in blocks]
        x = self.feats[torch.from_numpy(input_nodes)]
        self.opt.zero_grad()
        logits, _ = self.sage.forward(self.params, x, ob)
        loss = torch.nn.functional.cross_entropy(logits, self.labels[torch.from_numpy(seeds)])
        loss.backward()
        self.opt.step()
        return float(loss.item())


def cpu_csr(src, dst, V):
    """in-edge CSR (indptr, indices) of the symmetrised stream on the host (torch CPU stable sort)"""
    es = torch.cat([src, dst])
    ed = torch.cat([dst, src])
    order = torch.sort(ed, stable=True).indices
    deg = torch.bincount(ed, minlength=V)
    indptr = torch.zeros(V + 1, dtype=torch.int64)
    torch.cumsum(deg, 0, out=indptr[1:])
    return indptr.numpy(), es[order].numpy()


def time_cpu(path, batches, warmup):
    for b in batches[:warmup]:
        path.step(b)
    t0 = time.perf_counter()
    for b in batches[warmup:]:
        path.step(b)
    return time.perf_counter() - t0


# ----------------------------------------------------------------------------------------- roofline helpers
def stage_flops(stage, w, lv):
    """algorithmic FLOPs of one GEMM stage for per-step mean level counts lv = [B, N1, N0] (SURVEY 8(d))"""
    F, H, C = w["F"], w["H"], w["C"]
    B, N1, N0 = lv
    dims = [F, H, C]
    l = int(stage[1])
    fin, fout = dims[l], dims[l + 1]
    n_src, n_dst = (N0, N1) if l == 0 else (N1, B)
    kind = stage.split(".", 1)[1]
    if kind == "dW_group":     # one launch: fc_self + fc_neigh weight gradients of layer l (+ the fc_pool weight gradient of layer l+1)
        return 4.0 * n_dst * fin * fout + (2.0 * n_dst * fout * fout if l + 1 < 2 else 0.0)
    return {"pool_gemm": 2.0 * n_src * fin * fin, "out_gemm": 4.0 * n_dst * fin * fout, "dW_self": 2.0 * n_dst * fin * fout,
            "dW_neigh": 2.0 * n_dst * fin * fout, "dneigh_gemm": 2.0 * n_dst * fin * fout, "dW_pool": 2.0 * n_src * fin * fin,
            "dx_gemm": 2.0 * n_src * fin * fin + 2.0 * n_dst * fin * fout}.get(kind)


def stage_bytes(stage, w, lv, es=2):
    """algorithmic HBM bytes of the memory-bound stages (SURVEY 8(d)); es = bytes per stored feature element"""
    F, H = w["F"], w["H"]
    B, N1, N0 = lv
    f0, f1 = w["fanouts"]
    if stage == "gather":
        return 2.0 * N0 * F * es + 4.0 * N0
    if stage.startswith("sample.h"):
        h = int(stage[-1])
        D, s = (B, f0) if h == 0 else (N1, f1)
        return D * (4 + 8 + 4) + D * s * (4 + 4) + D * s * (4 + 8)          # row meta + (src,eid) reads + (src,eid) writes
    if stage.endswith(".pool_bwd"):
        l = int(stage[1])
        E, fin, ns = (N1 * f1, F, N0) if l == 0 else (B * f0, H, N1)
        return E * fin * (es + 1) + ns * fin * es + E * 4
    if stage.endswith(".segmax"):
        l = int(stage[1])
        E, fin, nd = (N1 * f1, F, N1) if l == 0 else (B * f0, H, B)
        return E * fin * es + nd * fin * (es + 1) + E * 4
    return None


# ----------------------------------------------------------------------------------------- main arms
def run_reference(args, rank, world):
    if rank != 0:
        return
    # torchrun pins OMP_NUM_THREADS=1 per rank; the other ranks have exited, so rank 0 takes every host core
    torch.set_num_threads(os.cpu_count() or 1)
    w = WORKLOADS[args.workload]
    torch.manual_seed(0)
    t_setup = time.time()
    src, dst = gen_edges(w, "cpu")
    indptr, indices = cpu_csr(src, dst, w["V"])
    del src, dst
    feats, labels = gen_features(w, "cpu")
    path = CpuPath(w, indptr, indices, feats, labels, init_params(w))
    batches = seed_batches(w, args.steps + args.warmup, 0, 1)
    setup_s = time.time() - t_setup
    el = time_cpu(path, batches, args.warmup)
    value = w["B"] * args.steps / el
    cores = torch.get_num_threads()
    line = {"impl": "reference", "metric": "graphsage_train_vertices_per_s", "value": value, "unit": "vertices/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(w, args.workload, 1),
            "cpu_baseline": {"value": value, "unit": "vertices/s", "cores": cores, "kind": "port",
                             "sample": "%d full train steps (B=%d) of the same workload on %d host threads (os.cpu_count=%d); setup %.0f s untimed"
                                       % (args.steps, w["B"], cores, os.cpu_count(), setup_s)},
            "e2e": {"value": value, "unit": "vertices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def first_appearance_relabel(src, dst):
    """dense vertex ids in first-appearance order (precondition of the reference's edge streams, reddit.py:101-113)"""
    inter = np.empty(2 * len(src), dtype=np.int64)
    inter[0::2], inter[1::2] = src, dst
    uniq, first = np.unique(inter, return_index=True)
    rank = np.empty(len(uniq), dtype=np.int64)
    rank[np.argsort(first, kind="stable")] = np.arange(len(uniq))
    lut = dict(zip(uniq.tolist(), rank.tolist())) if len(uniq) < 1000 else None
    pos = np.searchsorted(uniq, inter)
    out = rank[pos]
    return out[0::2].copy(), out[1::2].copy(), uniq[np.argsort(first, kind="stable")]


def aux_elliptic_pbr(n_snapshots=30, faithful=True):
    """configs[1]: Elliptic-shaped edge stream through the drop-in Python API (DynamicGraphEdge + TrainTestGraph + the
    PBR trainer with priority_forward = 2, settings/elliptic.json hyper-parameters): snapshot evolve, priority
    recomputation, 60 minibatches of 32 per timestep.  Reports trained target vertices / s over whole timesteps
    (choose_vertices + train + evolve), wall clock."""
    import random
    import ogl_b200
    from ogl_b200 import config
    from ogl_b200.graph import train_test_graph as ttg
    w = WORKLOADS["elliptic"]
    rng = np.random.default_rng(1)
    src, dst = rng.integers(0, w["V"], w["E"]), rng.integers(0, w["V"], w["E"])
    src, dst, order = first_appearance_relabel(src, dst)
    V = len(order)
    feats = rng.standard_normal((V, w["F"])).astype(np.float32)
    targets = rng.integers(0, w["C"], (V, 1)).astype(np.int64)
    config.set_faithful(faithful)
    config.set_precision("bf16")
    random.seed(1)
    np.random.seed(1)
    old = ttg.SIZE_BUFFER
    ttg.SIZE_BUFFER = 1 << 18
    try:
        GraphSAGE, _, PrioT, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, -1)
        dyn = ogl_b200.DynamicGraphEdge(1000, set(range(V)))
        dyn.build(feats, targets, edge_timestamps={"src": src, "dst": dst}, keep_master=False)
        gu = ttg.TrainTestGraph(dyn, split=0.15, start_prior_alpha=4, end_prior_alpha=50, scale=1, max_priority=10)
        model = GraphSAGE(w["F"], w["H"], w["C"], 1, act, 0, "pool").cuda()
        tr = PrioT(model, 60, 32, targets, 45, ogl_b200.LossPriority(), full_pass=2, cuda=True, batch_full=1024, n_workers=0)
        tr.build_optimizer()
        for _ in range(2):                       # warm-up timesteps (plan creation, graph capture)
            tr.train_timestep(gu)
            gu.evolve()
        torch.cuda.synchronize()
        times = []
        for _ in range(n_snapshots):
            t0 = time.perf_counter()
            tr.train_timestep(gu)
            gu.evolve()
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        med = float(np.median(times))          # (shared host: single timesteps are occasionally several times slower)
        return {"workload": "elliptic-shaped edge stream (V=%d, %d stream edges, F=%d, hidden %d, samples 45, batch 32 x 60 per timestep), "
                            "PBR, priority_forward=2, through the Python drop-in API" % (V, w["E"], w["F"], w["H"]),
                "timesteps": n_snapshots, "vertices_per_s": 60 * 32 / med, "ms_per_timestep_median": 1e3 * med,
                "ms_per_timestep_mean": 1e3 * float(np.mean(times)), "train_set": len(gu.get_train_set())}
    finally:
        ttg.SIZE_BUFFER = old
        config.set_faithful(True)


def aux_sampler_sweep(g, V, n_rows=1 << 20, fanout=25, iters=9):
    """config 5 flavour: the standalone uniform k-neighbour sampler over the resident Reddit-shaped CSR, 2^20 random
    destination rows x 25 picks per launch (indices + edge ids out).  Every call is timed by itself (CUDA events) after 5
    warm-up calls; min and median are reported."""
    from ogl_b200 import native
    gen = torch.Generator(device="cuda").manual_seed(9)
    dst = torch.randint(0, V, (n_rows,), generator=gen, device="cuda", dtype=torch.int64)
    for i in range(5):
        native.sample_neighbors(g, dst, fanout, seed=3, step=i, hop=0)
    torch.cuda.synchronize()
    ms = []
    for i in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        native.sample_neighbors(g, dst, fanout, seed=3, step=10 + i, hop=0)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    picks = n_rows * fanout
    alg = n_rows * (8 + 4 + 8) + picks * 8 + picks * (4 + 8)            # row meta + (eid, src) entry reads + (src, eid) writes
    sect = n_rows * 64 + picks * 32 + picks * 12
    med, best = float(np.median(ms)), float(min(ms))
    return {"rows": n_rows, "fanout": fanout, "ms_median": med, "ms_min": best, "calls": iters, "picks_per_s": picks / (med * 1e-3),
            "algorithmic_gbs": alg / (med * 1e-3) / 1e9, "sector_gbs": sect / (med * 1e-3) / 1e9, "sector_gbs_best": sect / (best * 1e-3) / 1e9,
            "note": "includes the int64->int32 cast of the row list (stream-ordered scratch from a pool that keeps its memory); sector_gbs "
                    "counts every random read as the 32-byte DRAM sector it costs (row start + degree: 2 sectors per row; one 8-byte "
                    "(edge id, source) entry: 1 sector per pick)"}


def aux_snapshot_insert(g, V, n_snap=40, snap_edges=11461):
    """the streaming regime the reference runs (settings/reddit.json: 57.3 M stream edges over 5000 snapshots = 11,461 stream edges
    per evolve(), dynamic_graph_edge.py:190-218): one symmetrised snapshot appended to the LIVE 114.6 M-edge CSR per call.  Launch
    bound, so microseconds per snapshot are reported beside edges/s."""
    import ogl_b200
    gen = torch.Generator(device="cuda").manual_seed(21)
    src = torch.randint(0, V, (n_snap + 5, snap_edges), generator=gen, device="cuda", dtype=torch.int64)
    dst = torch.randint(0, V, (n_snap + 5, snap_edges), generator=gen, device="cuda", dtype=torch.int64)
    for i in range(5):
        g.insert_edges(src[i], dst[i], symmetric=True)
    torch.cuda.synchronize()
    us, l0 = [], ogl_b200.kernel_launches()
    for i in range(5, n_snap + 5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        g.insert_edges(src[i], dst[i], symmetric=True)
        e1.record()
        torch.cuda.synchronize()
        us.append((1e3 * e0.elapsed_time(e1), 1e6 * (time.perf_counter() - t0)))
    dev_us = float(np.median([u[0] for u in us]))
    return {"stream_edges_per_snapshot": snap_edges, "snapshots": n_snap, "us_per_snapshot_device_median": dev_us,
            "us_per_snapshot_wall_median": float(np.median([u[1] for u in us])),
            "launches_per_snapshot": (ogl_b200.kernel_launches() - l0) / n_snap, "stream_edges_per_s": snap_edges / (dev_us * 1e-6),
            "algorithmic_gbs": 2 * snap_edges * 32 / (dev_us * 1e-6) / 1e9}


def aux_arxiv_vertex_stream(n_snapshots=20):
    """configs[2]: ogbn-arxiv-shaped VERTEX stream through the drop-in Python API (DynamicGraphVertex: the active set is a
    prefix of the arrival order, every evolve() re-derives the induced CSR on the GPU) with the RBR trainer and
    settings/arxiv.json hyper-parameters (hidden 32, samples 40, batch 32 x 1 per timestep, 3500 snapshots)."""
    import random
    import ogl_b200
    from ogl_b200 import config
    from ogl_b200.graph import train_test_graph as ttg
    w = WORKLOADS["arxiv"]
    rng = np.random.default_rng(2)
    V = w["V"]
    u, v = rng.integers(0, V, w["E"]), rng.integers(0, V, w["E"])
    feats = rng.standard_normal((V, w["F"])).astype(np.float32)
    targets = rng.integers(0, w["C"], (V, 1)).astype(np.int64)
    config.set_faithful(True)
    config.set_precision("bf16")
    random.seed(1)
    np.random.seed(1)
    old = ttg.SIZE_BUFFER
    ttg.SIZE_BUFFER = 1 << 18
    try:
        GraphSAGE, RandomT, _, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, -1)
        pg = ogl_b200.ParentGraph.from_undirected(u, v, V)
        pg.ndata["feat"], pg.ndata["target"] = feats, targets
        order = rng.permutation(V)
        ts = (np.arange(V), np.empty(V))
        ts[1][order] = np.arange(V, dtype=np.float64)
        t_build = time.perf_counter()
        dyn = ogl_b200.DynamicGraphVertex(pg, 3500, np.ones(V, dtype=bool))
        dyn.build(vertex_timestamps=(ts[0].tolist(), ts[1].tolist()))
        for _ in range(200):                          # start from a graph with ~10 k active vertices
            dyn.evolve()
        torch.cuda.synchronize()
        build_s = time.perf_counter() - t_build
        gu = ttg.TrainTestGraph(dyn, split=0.15, start_prior_alpha=4, end_prior_alpha=50, scale=1, max_priority=10)
        model = GraphSAGE(w["F"], w["H"], w["C"], 1, act, 0, "pool").cuda()
        tr = RandomT(model, 1, 32, targets, 40, cuda=True, batch_full=1024, n_workers=0)
        tr.build_optimizer()
        for _ in range(3):
            tr.train_timestep(gu)
            gu.evolve()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n_snapshots):
            tr.train_timestep(gu)
            gu.evolve()
        torch.cuda.synchronize()
        el = time.perf_counter() - t0
        return {"workload": "arxiv-shaped vertex stream (V=%d, %d directed edges, F=%d, hidden %d, samples 40, batch 32 x 1 per timestep, "
                            "3500 snapshots), RBR, through the Python drop-in API" % (V, 2 * w["E"], w["F"], w["H"]),
                "timesteps": n_snapshots, "vertices_per_s": 32 * n_snapshots / el, "ms_per_timestep_incl_evolve": 1e3 * el / n_snapshots,
                "active_vertices": len(dyn.get_graph()), "build_plus_200_evolves_s": build_s}
    finally:
        ttg.SIZE_BUFFER = old


def aux_cached_inference(n_requests=400, cpu_requests=20):
    """SURVEY 8(f)-3: the reference's streaming-inference request loop (inference_optimized.py:144-301) on an Elliptic-shaped model
    (F=166, hidden 256, 2 classes): requests of 1-5 new edges through ogl_b200.inference.CachedInference, and a bounded sample of the
    same stream through the CPU oracle port (oracle/inference.py), which is pinned to the reference's own method."""
    from ogl_b200.inference import CachedInference
    from oracle.inference import CachedInferenceOracle
    rng = np.random.default_rng(31)
    V, F, H, C = 20000, 166, 256, 2
    feat = rng.standard_normal((V, F)).astype(np.float32)
    params = {}
    for l, (i, o) in enumerate(((F, H), (H, C))):
        for name, (oo, ii) in (("fc_pool", (i, i)), ("fc_self", (o, i)), ("fc_neigh", (o, i))):
            params["layers.%d.%s.weight" % (l, name)] = (rng.standard_normal((oo, ii)) / np.sqrt(ii)).astype(np.float32)
            params["layers.%d.%s.bias" % (l, name)] = (0.1 * rng.standard_normal(oo)).astype(np.float32)
    # the serving graph first grows to ~50 k stored edges through 25 bulk requests (untimed, both arms), then small requests are timed:
    # the device path costs the same per request at any graph size, the handler's host-side graph queries (and this port's) are O(E)
    bulk = [[[int(x), int(y)] for x, y in rng.integers(0, V, (2000, 2))] for _ in range(25)]
    reqs = []
    for r in range(n_requests + 20):
        pairs = []
        for _ in range(int(rng.integers(1, 6))):
            a, b = int(rng.integers(0, V)), int(rng.integers(0, V))
            pairs += [[a, b]] + ([[b, a]] if rng.random() < 0.5 else [])
        reqs.append(pairs)
    d = CachedInference(feat, {k: torch.from_numpy(v) for k, v in params.items()})
    for q in bulk + reqs[:20]:
        d.request(q)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for q in reqs[20:]:
        d.request(q)
    torch.cuda.synchronize()
    gpu_s = time.perf_counter() - t0
    o = CachedInferenceOracle(feat, params)
    for q in bulk + reqs[:20]:
        o.request(q)
    t0 = time.perf_counter()
    for q in reqs[20:20 + cpu_requests]:
        o.request(q)
    cpu_s = time.perf_counter() - t0
    stored = len(o.src)
    return {"workload": "cached streaming inference, Elliptic-shaped model (F=%d, hidden %d, %d classes), %d requests of 1-5 new edges on a serving graph of %d stored edges" % (F, H, C, n_requests, stored),
            "requests_per_s": n_requests / gpu_s, "ms_per_request": 1e3 * gpu_s / n_requests,
            "cpu_port_requests_per_s": cpu_requests / cpu_s, "cpu_port_sample": "%d requests of the same stream, oracle/inference.py" % cpu_requests}


def workload_config(w, name, world):
    return {"workload": "%s-shaped synthetic graph: V=%d, %d stream edges (%d directed), F=%d, C=%d, hidden %d, B=%d per GPU, fan-outs %s, "
                        "2-layer GraphSAGE-pool, Adam" % (name, w["V"], w["E"], 2 * w["E"], w["F"], w["C"], w["H"], w["B"], w["fanouts"]),
            "global_batch": w["B"] * world, "parallelism": ("dp%d (replicated graph+features, two gradient buckets, %s, on a comm stream)" % (world, EXCHANGE_NAME.get(EXCHANGE[0], "?")) if world > 1 else "single GPU") +
                           "; sample+gather of step t+1 prefetched (second buffer set, own stream) under forward/backward of step t",
            "l2": "inputs larger than L2: feature table %.0f MB in the tf32 mode (fp32 storage), %.0f MB in fp16 / bf16, + CSR %.0f MB resident, random "
                  "row gathers; no explicit flush" % (w["V"] * ((w["F"] + 7) // 8 * 8) * 4 / 1e6, w["V"] * ((w["F"] + 7) // 8 * 8) * 2 / 1e6,
                                                      2 * w["E"] * 8 * 1.5 / 1e6)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, params, flat, grad, loss_sum):
    """write what the timed train step hands its caller after its last step, as <out_dir>/<name>.npy in fp32: the updated
    weights under their state-dict names, that step's gradient as grad.<name>, and its loss sum (over this rank's seeds) as
    loss_sum, so that two builds run with the same arguments can be compared output for output"""
    arrays, off = {"loss_sum": loss_sum.reshape(1)}, 0
    for k in (f"layers.{i}.{n}" for i in range(2) for n in NAMES):
        n = params[k].numel()
        arrays[k] = flat[off:off + n].view(params[k].shape)
        arrays["grad." + k] = grad[off:off + n].view(params[k].shape)
        off += n
    assert off == flat.numel(), (off, flat.numel())
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, "outputs of %d bytes exceed the dump limit" % total
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


DTYPES = {"fp16": dict(es=2, note="fp16 storage (ten explicit mantissa bits, as TF32) with static loss scaling: activation gradients are stored times a "
                                  "power of two derived from 1 / global batch and every weight / bias gradient is unscaled exactly where it is "
                                  "written in fp32; tcgen05.mma.kind::f16, fp32 accumulation, fp32 master weights and Adam"),
          "tf32": dict(es=4, note="fp32 storage with every GEMM operand rounded to TF32 where it is produced, tcgen05.mma.kind::tf32, fp32 accumulation"),
          "bf16": dict(es=2, note="bf16 storage, tcgen05.mma.kind::f16, fp32 accumulation: the fast mode, a labelled DEVIATION from north_star's "
                                  "rtol 1e-3 against the reference's fp32 path (see its `parity` block)")}


def measure(dt, headline, args, w, rank, world, dev, dist, g, feats, labels, host, peaks, clocks):
    """everything bench.py measures for one arithmetic mode `dt` on the resident graph: value (inputs in HBM), the stage table
    (headline mode only), e2e (pinned host seeds in, loss out every step), the replica check (N > 1) and the parity leg (N = 1)"""
    import ogl_b200
    from ogl_b200 import native
    V, B, K, W = w["V"], w["B"], args.steps, args.warmup
    es = DTYPES[dt]["es"]
    mode = {"tf32": ogl_b200.OGL_TF32, "bf16": ogl_b200.OGL_BF16, "fp16": ogl_b200.OGL_FP16}[dt]
    fs = native.Features(V, w["F"], mode)
    fs.write(0, feats, labels)
    params = init_params(w)
    flat0 = torch.cat([params[f"layers.{i}.{n}"].reshape(-1).float() for i in range(2) for n in NAMES]).to(dev)
    flat = flat0.clone()
    grad = torch.zeros_like(flat)
    plan = native.Plan([w["F"], w["H"], w["C"]], w["fanouts"], B, V, mode=mode, seed=11)
    plan.bind_params(flat, grad)
    peer = None
    force_split = world == 1 and bool(os.environ.get("OGL_DP_FORCE_SPLIT"))
    if (world > 1 and args.exchange == "peer") or force_split:
        # gradient exchange + Adam as ONE kernel per bucket over NVLink peer memory (csrc/peer.cu); the gradient buffer moves into
        # the peer-visible allocation
        peer = ogl_b200.parallel.make_peer_exchange(plan, flat)
        grad = peer.grads
    n_check = 3 if world > 1 else 0
    batches = seed_batches(w, K + W + n_check, rank, world)
    dev_batches = [torch.as_tensor(b).to(dev) for b in batches]
    pin = [torch.as_tensor(b).pin_memory() for b in batches]
    loss_dev = torch.zeros(1, device=dev)

    def step(seeds):
        # local sample / forward / backward -> (N > 1: one NCCL all-reduce of the flat gradient) -> fused Adam
        ogl_b200.parallel.train_step(plan, g, fs, seeds, B * world, grad, loss_sum_out=loss_dev)

    pipe = ogl_b200.parallel.Pipeline(plan, g, fs, grad, B * world, peer=peer, force_split=force_split) if not args.no_pipeline else None
    # e2e: the step's loss kernel writes the loss sum STRAIGHT into pinned host memory (`loss_sum_out` may be any device-accessible
    # pointer; a 4-byte zero-copy store over PCIe instead of a D2H memcpy node between two graph launches); two slots, so that the
    # host reads step t's loss while step t+1 runs
    loss_host = [torch.zeros(1).pin_memory() for _ in range(2)]
    loss_evs = [torch.cuda.Event(), torch.cuda.Event()]

    def run_steps(inputs, read_back, losses):
        """pipelined loop (ogl_b200.parallel.Pipeline): sample + gather of step t+1 (ogl_plan_prefetch, the plan's second buffer
        set) overlap forward / backward of step t; N > 1 adds the bucketed gradient exchange + Adam on a comm stream.
        --no-pipeline: one fused (graph-replayed) ogl_plan_train_step per step."""
        if pipe is None:
            for s in inputs:
                step(s)
                if read_back:
                    losses.append(float(loss_dev.item()))      # D2H read of the step's loss (synchronises)
            return
        pipe.begin(inputs[0])
        n = len(inputs)
        for i in range(n):
            slot = i & 1
            pipe.finish(inputs[i + 1] if i + 1 < n else None, loss_sum_out=loss_host[slot] if read_back else loss_dev)
            if read_back:
                # every step's loss goes device -> pinned host memory inside the timed region (written by the step itself); the host
                # consumes it one step later, so that the read-back of step t does not stall the launch of step t+1
                loss_evs[slot].record()
                if i > 0:
                    loss_evs[slot ^ 1].synchronize()
                    losses.append(float(loss_host[slot ^ 1]))
        if read_back and n > 0:
            loss_evs[(n - 1) & 1].synchronize()
            losses.append(float(loss_host[(n - 1) & 1]))
        pipe.flush()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    host_ms = [0.0]

    def timed(inputs, read_back):
        """K steps bracketed by barrier + synchronize; device time by CUDA events, max over ranks"""
        barrier()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        wall0 = time.time()
        t0.record()
        losses = []
        h0 = time.perf_counter()
        run_steps(inputs, read_back, losses)
        host_ms[0] = (time.perf_counter() - h0) * 1e3      # host time to ENQUEUE the steps (well below the device time = not host-bound)
        t1.record()
        barrier()
        wall1 = time.time()
        ms = t0.elapsed_time(t1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, wall0, wall1, losses

    # ---- N > 1: replicas stay bit-identical, and the N-rank run equals the same global batches trained on ONE rank
    replicas = None
    if world > 1:
        chk = dev_batches[K + W:]
        run_steps(chk, False, [])
        torch.cuda.synchronize()
        # 64-bit checksum of the raw parameter bits, compared across the ranks
        cs = flat.view(torch.int32).to(torch.int64).sum().reshape(1)
        every = [torch.zeros_like(cs) for _ in range(world)]
        dist.all_gather(every, cs)
        same = all(int(e.item()) == int(every[0].item()) for e in every)
        # rank 0 replays the n_check steps alone: for every step the shards of all ranks one after the other (same Philox step and
        # row positions as rank r used), gradients summed in rank order, one Adam step -- with a plan of its own
        all_seeds = [torch.zeros(B, dtype=torch.int64, device=dev) for _ in range(world)]
        replay_err = None
        trained = flat.clone()
        step_seeds = []
        for sd in chk:
            dist.all_gather(all_seeds, sd)
            step_seeds.append([t.clone() for t in all_seeds])
        if rank == 0:
            f2, g2 = flat0.clone(), torch.zeros_like(flat0)
            p2 = native.Plan([w["F"], w["H"], w["C"]], w["fanouts"], B, V, mode=mode, seed=11)
            p2.bind_params(f2, g2)
            acc = torch.zeros_like(g2)
            for t, shards in enumerate(step_seeds):
                acc.zero_()
                for sd in shards:
                    p2.set_step(t)
                    p2.sample(g, sd)
                    p2.forward(fs, want_logits=False)
                    p2.loss_backward(fs, 1.0 / (B * world), want_per_vertex=False)
                    acc += g2
                g2.copy_(acc)
                p2.adam_step()
            torch.cuda.synchronize()
            replay_err = float((f2 - trained).abs().max().item() / trained.abs().max().item())
            del p2
        replicas = {"replicas_bit_identical": bool(same), "checked_after_steps": n_check, "checksum": int(every[0].item()),
                    "one_rank_replay_max_err_of_scale": replay_err,
                    "note": "rank 0 replays the same global batches alone (all shards in rank order, summed gradients, one Adam step per step)"}
        assert same, "data-parallel replicas diverged: %r" % [int(e.item()) for e in every]
        # back to the initial state for the measurement
        flat.copy_(flat0)
        plan.refresh_params()
        plan.reset_optimizer(0)
        barrier()

    run_steps(dev_batches[:W], False, [])
    # ---- value: inputs resident in HBM (the step's launch sequence is replayed as CUDA graphs)
    gs0 = plan.graph_stats()
    l0 = ogl_b200.kernel_launches()
    ms_dev, wall0, wall1, _ = timed(dev_batches[W:W + K], read_back=False)
    host_enqueue_ms = host_ms[0]
    gs1 = plan.graph_stats()
    if headline and args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, params, flat, grad, loss_dev)
    out = {"dtype": dt, "arithmetic": DTYPES[dt]["note"], "value": B * world * K / (ms_dev / 1e3), "ms_per_step": ms_dev / K,
           "host_enqueue_ms_per_step": host_enqueue_ms / K, "replicas": replicas,
           "cuda_graph": {"replays_in_timed_region": gs1["replays"] - gs0["replays"], "captures_in_timed_region": gs1["captures"] - gs0["captures"]},
           "clocks": clocks.window(wall0, wall1) if clocks else None}
    # ---- the same K steps once more with the library's per-stage CUDA events on (direct launches, no graph, no overlap):
    #      stage shares + the roofline of the dominant kernel
    stages = None
    if headline:
        plan.profile(True)
        l0 = ogl_b200.kernel_launches()
        ms_prof, _, _, _ = timed(dev_batches[W:W + K], read_back=False)
        launches = ogl_b200.kernel_launches() - l0          # kernels per K steps (a graph replay launches the same kernels)
        stages, level_sums, n_prof = plan.profile_read()
        plan.profile(False)
        out["gpu_launches"] = launches
        out["cuda_graph"]["ms_per_step_direct_launch_profiled"] = ms_prof / K
    # ---- e2e: pinned host seeds -> H2D inside the call, loss D2H every step
    run_steps(pin[:W], False, [])
    ms_e2e, wall2, wall3, losses = timed(pin[W:W + K], read_back=True)
    last_loss = None
    if losses:
        t = torch.tensor([losses[-1]], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t)                              # the loss sum of the GLOBAL batch of the last step
        last_loss = float(t.item()) / (B * world)
    out["e2e"] = {"value": B * world * K / (ms_e2e / 1e3), "unit": "vertices/s", "h2d_bytes_per_step": 8 * B, "d2h_bytes_per_step": 4,
                  "ms_per_step": ms_e2e / K,
                  "api": "ogl_plan_prefetch(pinned host seeds of step t+1) + ogl_plan_step_finish(step t, loss_sum_out = pinned host memory: the step's loss kernel stores its 4 bytes there itself, every step; the host consumes them one step later)",
                  "last_loss": last_loss, "clocks": clocks.window(wall2, wall3) if clocks else None}
    if rank != 0:
        return out

    # ---- roofline of the dominant kernel (headline mode)
    if headline:
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        tc_sus, tc_burst = peaks.get("bf16_tflops_sustained", 1400.0), peaks.get("bf16_tflops", 1650.0)
        peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        if dt == "tf32":                                    # tcgen05 kind::tf32 issues at half the kind::f16 rate (1.125 vs 2.25 PFLOP/s nominal)
            tc_sus, tc_burst, tc_nom = tc_sus / 2, tc_burst / 2, 1125.0
            peak_src += ", bf16 figures / 2 for kind::tf32"
        else:
            tc_nom = 2250.0
        lv = [x / max(n_prof, 1) for x in level_sums]                 # mean [B, N1, N0] per step
        per = {k: v[0] / max(n_prof, 1) for k, v in stages.items()}   # ms per step per stage
        total_stage_ms = sum(per.values())
        # dominant kernel = the kernel family with the largest total share of the step; the roofline is quoted on its
        # largest launch (FLOPs / bytes of that launch from the per-step node counts, duration from the stage events)
        is_layer = lambda k: len(k) > 3 and k[0] == "l" and k[1].isdigit() and k[2] == "."

        def family(k):
            kind = k.split(".", 1)[1] if is_layer(k) else k.split(".")[0]
            if kind in ("pool_gemm", "out_gemm", "dneigh_gemm", "dx_gemm"):
                return "k_gemm_nt_tc"
            if kind in ("dW_self", "dW_neigh", "dW_pool", "dW_group"):
                return "k_gemm_tn_tc"
            return {"pool_bwd": "k_pool_bwd", "segmax": "k_segmax_fwd", "gather": "k_gather_rows", "sample": "k_sample",
                    "to_block": "k_tb_*", "rev_edges": "k_rev_*", "db_out": "k_colsum_*", "db_pool": "k_colsum_*"}.get(kind, kind)
        fam = {}
        for k in per:
            fam.setdefault(family(k), []).append(k)
        fam_ms = {f: sum(per[k] for k in ks) for f, ks in fam.items()}
        top_family = max(fam_ms, key=fam_ms.get)
        top = max(fam[top_family], key=per.get)
        fl = stage_flops(top, w, lv) if is_layer(top) else None
        by = stage_bytes(top, w, lv, es)
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(dt, {}).get(top)
            if tr:
                traffic = tr["dram_read_bytes"] + tr["dram_write_bytes"]
        except Exception:
            pass
        common = {"kernel": top_family, "launch": top, "kernel_share_of_step": fam_ms[top_family] / total_stage_ms,
                  "kernel_ms_per_step": fam_ms[top_family], "kernel_launches_per_step": len(fam[top_family]), "traffic": traffic,
                  "ms_per_launch": per[top], "timed_by": "CUDA events recorded by the library around the launch, on the launch stream, "
                                                         "kernel alone on the device (stages_mode)"}
        if fl:
            ach = fl / (per[top] * 1e-3) / 1e12
            # a single ~0.1 ms kernel timed by itself runs in the burst regime (1965 MHz): `frac` is against the burst peak; the
            # sustained figure (long back-to-back GEMMs, clocks settled ~1.3 GHz) and the data-sheet one are printed beside it
            roof = dict(common, bound="tensor", achieved=ach, peak=tc_burst, unit="TFLOP/s", frac=ach / tc_burst, peak_source=peak_src + ", burst",
                        peak_burst=tc_burst, frac_burst=ach / tc_burst, peak_sustained=tc_sus, frac_sustained=ach / tc_sus,
                        flops_per_launch=fl, peak_nominal=tc_nom, frac_nominal=ach / tc_nom)
            fam_fl = sum(stage_flops(k, w, lv) or 0.0 for k in fam[top_family])
            roof["kernel_avg_tflops"] = fam_fl / (fam_ms[top_family] * 1e-3) / 1e12
        elif by:
            ach = by / (per[top] * 1e-3) / 1e9
            roof = dict(common, bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s", frac=ach / hbm_peak, peak_source=peak_src,
                        bytes_per_launch=by, peak_nominal=8000.0, frac_nominal=ach / 8000.0)
        else:
            roof = dict(common, bound="hbm", achieved=None, peak=hbm_peak, unit="GB/s", frac=None)
        stage_table = {}
        for k in sorted(per, key=per.get, reverse=True):
            ent = {"ms": round(per[k], 4), "share": round(per[k] / total_stage_ms, 4)}
            f_, b_ = (stage_flops(k, w, lv) if is_layer(k) else None), stage_bytes(k, w, lv, es)
            if f_:
                ent["tflops"] = round(f_ / (per[k] * 1e-3) / 1e12, 1)
            if b_:
                ent["gbs"] = round(b_ / (per[k] * 1e-3) / 1e9, 1)
            stage_table[k] = ent
        out["roofline"] = roof
        out["stages"] = stage_table
        out["stages_mode"] = ("direct launches with CUDA events around every stage, no CUDA graph, no side-stream / prefetch overlap: %.3f ms per "
                              "step against %.3f ms for the graph-replayed, overlapped step that `value` times; shares and per-kernel rates come "
                              "from this mode" % (ms_prof / K, ms_dev / K))
        out["mean_level_counts"] = {"B": lv[0], "N1": lv[1], "N0": lv[2]}

    # ---- parity leg (N = 1, untimed): ONE step of this mode at the trained weights against the unquantised fp64 oracle on the
    #      same sampled blocks (oracle/parity.py; the oracle is the checker here, never the thing measured)
    if host is not None and not args.no_parity:
        from oracle import parity as opar
        seeds = batches[W]
        sd = torch.as_tensor(seeds).to(dev)
        trained = flat.clone()

        def parity_at(weights, label):
            t0 = time.time()
            flat.copy_(weights)
            plan.refresh_params()
            plan.sample(g, sd)
            logits = plan.forward(fs)
            per_v, _ = plan.loss_backward(fs, 1.0 / B)
            torch.cuda.synchronize()
            cur = opar.dict_from_flat(flat.detach().cpu(), [w["F"], w["H"], w["C"]])
            m = opar.compare_step(plan, cur, host["feats"], host["labels"], seeds, logits, per_v, grad,
                                  {"tf32": 2.0 ** -10, "fp16": 2.0 ** -10, "bf16": 2.0 ** -8}[dt])
            r = opar.summary(m)
            r["weights"] = label
            r["logits_scale"] = m["logits"]["scale"]
            r["seconds"] = round(time.time() - t0, 1)
            r["meets_rtol_1e-3"] = {"logits_and_losses": bool(m["logits"]["frac_outside"] == 0.0 and m["per_vertex_loss"]["frac_outside"] == 0.0),
                                    "gradients_pinned": bool(m["grad_frac_outside_pinned_max"] == 0.0)}
            return r
        # at the initial weights (the state tests/test_gpu_parity_reddit.py asserts on) and at the weights the timed steps left behind:
        # cross-entropy turns an ABSOLUTE logit error e into a RELATIVE error ~e of d(loss)/d(logits), so every gradient inherits a
        # common relative error that grows with the scale of the logits as training proceeds
        out["parity"] = parity_at(flat0, "initial (Xavier, seed 0)")
        out["parity_trained"] = parity_at(trained, "after the %d warm-up + timed steps of this run" % (2 * (K + W) + (K if headline else 0)))
    del pipe, plan, fs
    torch.cuda.empty_cache()
    return out


def run_ours(args, rank, world, local_rank):
    import ogl_b200
    from ogl_b200 import native
    w = WORKLOADS[args.workload]
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    clocks = ClockSampler(local_rank) if rank == 0 else None

    # ---- build the streaming graph by inserting the edge stream in snapshot batches (timed: edge inserts/s)
    src, dst = gen_edges(w, dev)
    V, E = w["V"], w["E"]
    g = native.Graph(V, 2 * E + (1 << 20))               # (+ room for the snapshot-insert aux leg)
    g.insert_vertices(V)
    chunk = max(1 << 14, min(1 << 21, E // 16))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = ogl_b200.kernel_launches()
    e0.record()
    for a in range(0, E, chunk):
        g.insert_edges(src[a:a + chunk], dst[a:a + chunk], symmetric=True)
    e1.record()
    torch.cuda.synchronize()
    insert_ms = e0.elapsed_time(e1)
    insert_launches = ogl_b200.kernel_launches() - launches0
    assert g.num_edges == 2 * E
    feats, labels = gen_features(w, dev)
    host = None
    if rank == 0 and world == 1 and not (args.no_cpu_baseline and args.no_parity):
        ip, ix, _ = g.export_csr(with_eids=False)
        host = {"csr": (ip.cpu().numpy(), ix.cpu().numpy()), "feats": feats.cpu(), "labels": labels.cpu()}
        del ip, ix
    del src, dst
    torch.cuda.empty_cache()

    dts = [args.dtype]
    if world == 1 and not args.no_alt:
        dts += [d for d in ("fp16", "tf32", "bf16") if d != args.dtype]
    res = {}
    for i, dt in enumerate(dts):
        res[dt] = measure(dt, i == 0, args, w, rank, world, dev, dist, g, feats, labels, host, peaks, clocks)
    if clocks:
        clocks.stop()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    B, K, W = w["B"], args.steps, args.warmup
    head = res[args.dtype]

    cpu = None
    if host is not None and not args.no_cpu_baseline:
        IMPL[0] = "reference"
        torch.set_num_threads(os.cpu_count() or 1)
        path = CpuPath(w, host["csr"][0], host["csr"][1], host["feats"], host["labels"], init_params(w))
        IMPL[0] = "ours"
        cb = seed_batches(w, args.cpu_steps + 1, 0, 1, seed=5)
        el = time_cpu(path, cb, 1)
        cpu = {"value": B * args.cpu_steps / el, "unit": "vertices/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": "%d full train steps (B=%d) of the same workload, oracle port (numpy sampler + torch-CPU fp32 SAGE-pool + Adam), %.1f s"
                         % (args.cpu_steps, B, el)}
    del feats
    aux, snap = None, None
    if world == 1 and not args.no_aux:
        try:
            sweep = aux_sampler_sweep(g, V)
            # the regime the reference runs: one snapshot of settings/reddit.json = 11,461 stream edges appended to the LIVE graph
            snap = aux_snapshot_insert(g, V)
        except Exception as e:
            sweep = {"error": repr(e)[:300]}
        del g
        torch.cuda.empty_cache()
        try:
            aux = {"elliptic_pbr": aux_elliptic_pbr(faithful=True)}
            aux["elliptic_pbr"]["mode"] = "faithful (reference choosers: host shuffles, per-batch loss read-back into the Python priority dict)"
            aux["elliptic_pbr_device"] = aux_elliptic_pbr(faithful=False)
            aux["elliptic_pbr_device"]["mode"] = "device (counter-RNG draws, stratified proportional sampling and priority updates on the GPU sum tree)"
            aux["sampler_sweep"] = sweep
            aux["arxiv_rbr"] = aux_arxiv_vertex_stream()
            aux["cached_inference"] = aux_cached_inference()
        except Exception as e:                       # the aux leg must never take the headline line with it
            aux = {"elliptic_pbr": {"error": repr(e)[:300]}}
    alt = []
    for dt in dts[1:]:
        r = res[dt]
        alt.append({k: r[k] for k in ("dtype", "arithmetic", "value", "ms_per_step", "e2e", "parity", "parity_trained", "clocks") if k in r})
    line = {"metric": "graphsage_train_vertices_per_s", "value": head["value"], "unit": "vertices/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": head["dtype"],
            "arithmetic": head["arithmetic"], "data": "synthetic", "config": workload_config(w, args.workload, world),
            "e2e": head["e2e"], "parity": head.get("parity"), "parity_trained": head.get("parity_trained"), "replicas": head.get("replicas"),
            "host_enqueue_ms_per_step": head["host_enqueue_ms_per_step"], "gpu_launches": head.get("gpu_launches"),
            "cuda_graph": head["cuda_graph"], "clocks": head["clocks"], "roofline": head.get("roofline"), "cpu_baseline": cpu,
            "mean_level_counts": head.get("mean_level_counts"), "stages": head.get("stages"), "stages_mode": head.get("stages_mode"),
            "alt": alt or None, "aux": aux,
            "edge_insert": {"stream_edges_per_s": E / (insert_ms / 1e3), "ms": insert_ms, "batch_stream_edges": chunk, "launches": insert_launches,
                            "algorithmic_gbs": 2 * E * (16 + 8 + 8) / (insert_ms / 1e3) / 1e9, "snapshot": snap}}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="reddit", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-steps", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: gradient exchange + Adam fused in one kernel over NVLink peer memory, or NCCL all-reduce + Adam")
    ap.add_argument("--no-pipeline", action="store_true", help="one fused ogl_plan_train_step per step instead of the prefetch pipeline")
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "tf32", "bf16"],
                    help="arithmetic of the headline line: fp16 (loss-scaled) and tf32 meet north_star's rtol 1e-3 against the reference's fp32 "
                         "path -- fp16 stores half the bytes and issues at twice the tensor rate; bf16 is as fast as fp16 but a labelled deviation "
                         "(N = 1 prints the other modes too, under `alt`)")
    ap.add_argument("--no-alt", action="store_true", help="N = 1: do not measure the other arithmetic modes")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity leg (one step against the fp64 oracle, untimed)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of the headline mode, write what their last step returned (updated weights, gradient, "
                         "loss sum; rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    EXCHANGE[0] = args.exchange
    IMPL[0] = args.impl
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a B200: the product path has no CPU fallback")
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
