#!/usr/bin/env python
"""Incremental full-neighbourhood inference: StreamingInference.refresh() after an insert batch against the whole-graph call
model.inference(graph) at the same state.

    python tools/streaming_inference_bench.py [--reps 10] [--warmup 2] [--workloads reddit,arxiv] [--out FILE]

bench.py's Reddit-shaped and arxiv-shaped graphs (symmetric edge streams), features and weights, 2-layer models in fp16 and tf32.
The graph is built without the last edges of its stream; those arrive in batches of increasing size (a serving request, one
snapshot, ten snapshots, and one batch whose frontier crosses the threshold), each applied once.  Per batch and mode:
  - refresh(): CUDA events around the call, median / min / max of --reps calls after --warmup calls.  Every call starts from the
    state before the batch (the engine's stored degrees are reset outside the timed window), so it repeats the same work: the suffix
    max is idempotent and every recomputed row is computed on its own;
  - whole: model.inference(graph), timed the same way;
  - per layer: the output rows the refresh recomputed, their edge share (sum of in-degree + 1 over E + V), the path taken, and the
    per-stage times of one profiled refresh;
  - whether the refreshed logits are torch.equal to the whole-graph call (asserted).
Prints one JSON line with the GPU and its power limit."""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from full_inference_bench import emit, gpu_info, timed  # noqa: E402

SNAPSHOT = 11461                 # stream edges per snapshot of settings/reddit.json (57.3 M over 5,000 snapshots)
BATCHES = {"reddit": [10, SNAPSHOT, 10 * SNAPSHOT, 1000000], "arxiv": [10, SNAPSHOT, 10 * SNAPSHOT, 400000]}


def run_workload(name, args, dev, modes):
    import ogl_b200
    w = bench.WORKLOADS[name]
    V, E = w["V"], w["E"]
    batches = BATCHES[name]
    src, dst = bench.gen_edges(w, dev)
    feats, labels = bench.gen_features(w, dev)
    params = bench.init_params(w)
    GraphSAGE, _, _, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, -1)
    res = {"workload": "%s-shaped synthetic graph of bench.py: V=%d, %d undirected stream edges (inserted in both directions), F=%d, "
                       "hidden %d, C=%d, 2 layers, max-pool; the last %d stream edges arrive in batches of %s" % (
                           name, V, E, w["F"], w["H"], w["C"], sum(batches), batches), "modes": {}}
    for mname, mode in modes:
        dg = ogl_b200.DeviceGraph(V, 2 * E, w["F"], mode=mode, keep_master=False)
        dg.add_nodes(V, {"feat": feats, "target": labels})
        head = E - sum(batches)
        chunk = max(1 << 14, min(1 << 21, E // 16))
        for a in range(0, head, chunk):
            dg.native.insert_edges(src[a:min(a + chunk, head)], dst[a:min(a + chunk, head)], symmetric=True)
        model = GraphSAGE(w["F"], w["H"], w["C"], 1, act, 0.0, "pool").cuda()
        model.load_state_dict({k: v.float() for k, v in params.items()})
        eng = ogl_b200.inference.StreamingInference(model, dg)
        plan = model.inference_plan(dg)
        eng.refresh()
        out, a = {}, head
        for b in batches:
            prev_deg, prev_n = eng.deg.clone(), eng._n
            dg.native.insert_edges(src[a:a + b], dst[a:a + b], symmetric=True)
            a += b
            Vg, Eg = dg.native.num_vertices, dg.native.num_edges

            def reset():
                eng.deg.copy_(prev_deg)
                eng._n = prev_n

            for _ in range(args.warmup):
                reset()
                eng.refresh()
            ms = []
            for _ in range(args.reps):
                reset()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                info = eng.refresh()
                e1.record()
                torch.cuda.synchronize()
                ms.append(e0.elapsed_time(e1))
            r = {"refresh": {"median_ms": float(np.median(ms)), "min_ms": float(min(ms)), "max_ms": float(max(ms)), "reps": args.reps},
                 "whole": timed(lambda: model.inference(dg), args.reps, args.warmup)}
            r["speedup_median"] = r["whole"]["median_ms"] / r["refresh"]["median_ms"]
            r["layers"] = [dict(rows=l["rows"], row_share=l["rows"] / Vg, edge_share=l["edges"] / (Eg + Vg), path=l["path"])
                           for l in info["layers"]]
            reset()
            plan.profile(True)
            eng.refresh()
            stages, _, _ = plan.profile_read()
            plan.profile(False)
            r["stages_ms"] = {k: round(v[0], 4) for k, v in stages.items() if v[1] > 0 and k.startswith("stream.")}
            equal = bool(torch.equal(eng.logits(), model.inference(dg)))
            assert equal, (name, mname, b)
            r["equal_to_whole"] = equal
            out[str(b)] = r
            print(name, mname, b, r["refresh"]["median_ms"], r["whole"]["median_ms"], [l["path"] for l in r["layers"]], file=sys.stderr)
        res["modes"][mname] = out
        del eng, plan, model, dg
        torch.cuda.empty_cache()
    del src, dst, feats, labels
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--workloads", default="reddit,arxiv")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "streaming_inference_bench needs a GPU"
    import ogl_b200
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    modes = (("fp16", ogl_b200.OGL_FP16), ("tf32", ogl_b200.OGL_TF32))
    out = {"gpu": gpu_info(), "theta": 0.9, "workloads": {}}
    for name in args.workloads.split(","):
        out["workloads"][name] = run_workload(name, args, dev, modes)
    emit(out, args.out)


if __name__ == "__main__":
    main()
