#!/usr/bin/env python
"""Full-neighbourhood inference of short vertex lists: the frontier path of ogl_plan_infer_full against the whole-graph hidden layer.

    python tools/frontier_bench.py [--reps 10] [--warmup 2] [--out FILE]

On bench.py's Reddit-shaped graph (lists of 39, 200, 1,000, 5,000 and 34,945 = the 15 % split, fp16 and tf32) and arxiv-shaped
graph (39, 1,000, 5,000, fp16 and tf32), 2-layer models with bench.py's weights, per list:
  - rows and edge share of each layer: S_1 = the list (the last layer), S_0 = S_1 u N_in(S_1) (Graph.in_frontier); the edge share
    is sum over the rows of (in-degree + 1) over E + V, the quantity the plan compares with its threshold;
  - "new": plan.infer_full(g, f, T), the path the plan chooses (frontier when S_0's share is at most the threshold);
  - "old": the path before the frontier, rebuilt from public calls: layer 0 over [0, V), then the last layer over T;
  - "frontier": the frontier path at any share, rebuilt from public calls: layer 0 over S_0 (precomputed), its rows scattered into
    the [V, pitch] table (torch index_copy_), the last layer over T; plus the frontier kernel's time from the profile of "new" (its
    expansion runs whichever path is chosen).  The crossover of "frontier" and "old" is the threshold the plan should use;
  - the per-stage times of one profiled "new" call, and whether its logits are torch.equal to "old".
Times: CUDA events around the call, median / min / max of --reps calls after --warmup calls.  Prints one JSON line with the GPU
and its power limit."""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from full_inference_bench import BATCH_FULL, emit, gpu_info, timed  # noqa: E402

CASES = {"reddit": [39, 200, 1000, 5000, 34945], "arxiv": [39, 1000, 5000]}


def setup(name, dev):
    from ogl_b200 import native
    w = bench.WORKLOADS[name]
    V, E = w["V"], w["E"]
    src, dst = bench.gen_edges(w, dev)
    g = native.Graph(V, 2 * E)
    g.insert_vertices(V)
    chunk = max(1 << 14, min(1 << 21, E // 16))
    for a in range(0, E, chunk):
        g.insert_edges(src[a:a + chunk], dst[a:a + chunk], symmetric=True)
    del src, dst
    feats, labels = bench.gen_features(w, dev)
    params = bench.init_params(w)
    flat0 = torch.cat([params["layers.%d.%s" % (i, n)].reshape(-1).float() for i in range(2) for n in bench.NAMES]).to(dev)
    return w, g, feats, labels, flat0


def run_workload(name, args, dev, modes):
    from ogl_b200 import native
    w, g, feats, labels, flat0 = setup(name, dev)
    V, C = w["V"], w["C"]
    E = g.num_edges
    deg = g.degrees()
    rng = np.random.default_rng(5)
    lists = {n: torch.as_tensor(rng.permutation(V)[:n], dtype=torch.int64, device=dev) for n in CASES[name]}
    res = {"workload": "%s-shaped synthetic graph of bench.py: V=%d, %d directed edges, F=%d, hidden %d, C=%d, 2 layers, max-pool" % (
        name, V, E, w["F"], w["H"], C), "lists": {}}
    fronts = {}
    for n, T in lists.items():
        s0, cost0 = g.in_frontier(T)
        fronts[n] = s0
        cost1 = int((deg[T] + 1).sum())
        res["lists"][str(n)] = {"layers": {"l0": {"rows": int(s0.numel()), "row_share": s0.numel() / V, "edge_share": cost0 / (E + V)},
                                           "l1": {"rows": n, "row_share": n / V, "edge_share": cost1 / (E + V)}}, "modes": {}}
    for mname, mode in modes:
        fs = native.Features(V, w["F"], mode)
        fs.write(0, feats, labels)
        plan = native.Plan([w["F"], w["H"], C], w["fanouts"], BATCH_FULL, V, mode=mode, seed=5)
        flat = flat0.clone()
        plan.bind_params(flat, torch.zeros_like(flat))
        table = plan.hidden_table(0, V)
        for n, T in lists.items():
            s0 = fronts[n]
            compact = plan.hidden_table(0, s0.numel())
            new_l = torch.empty(n, C, device=dev)
            old_l = torch.empty(n, C, device=dev)
            fr_l = torch.empty(n, C, device=dev)

            def new():
                plan.infer_full(g, fs, T, logits_out=new_l)

            def old():
                plan.infer_full_layer(g, fs, 0, None, out=table)
                plan.infer_full_layer(g, fs, 1, table, rows=T, out=old_l)

            def frontier():
                plan.infer_full_layer(g, fs, 0, None, rows=s0, out=compact)
                table.index_copy_(0, s0, compact[:s0.numel()])
                plan.infer_full_layer(g, fs, 1, table, rows=T, out=fr_l)

            r = {"new": timed(new, args.reps, args.warmup), "old": timed(old, args.reps, args.warmup),
                 "frontier_from_public_calls": timed(frontier, args.reps, args.warmup)}
            new()
            old()
            frontier()
            torch.cuda.synchronize()
            r["new_equal_old"] = bool(torch.equal(new_l, old_l))
            r["frontier_equal_old"] = bool(torch.equal(fr_l, old_l))
            plan.profile(True)
            new()
            stages, _, _ = plan.profile_read()
            plan.profile(False)
            stages = {k: v for k, v in stages.items() if v[1] > 0}       # (the plan keeps the names of stages of earlier calls)
            r["stages_ms"] = {k: round(v[0], 4) for k, v in stages.items()}
            r["path"] = "frontier" if "full.l0.scatter" in stages else "all_rows"
            fk = stages.get("full.l0.frontier", (0.0, 0))[0]
            r["frontier_kernel_ms"] = fk
            r["frontier_total_median_ms"] = r["frontier_from_public_calls"]["median_ms"] + fk
            res["lists"][str(n)]["modes"][mname] = r
            del compact
        del plan, fs, table
        torch.cuda.empty_cache()
    del g
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="reddit,arxiv")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "frontier_bench needs a GPU"
    import ogl_b200
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    modes = (("fp16", ogl_b200.OGL_FP16), ("tf32", ogl_b200.OGL_TF32))
    out = {"gpu": gpu_info(), "workloads": {}}
    for name in args.workloads.split(","):
        out["workloads"][name] = run_workload(name, args, dev, modes)
    emit(out, args.out)


if __name__ == "__main__":
    main()
