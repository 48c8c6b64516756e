#!/usr/bin/env python
"""Full-neighbourhood inference (GraphSAGE.inference / ogl_plan_infer_full) on the Reddit-shaped workload of bench.py.

    python tools/full_inference_bench.py [--reps 10] [--warmup 2] [--sampled-reps 3] [--out FILE]
    torchrun --nproc-per-node N tools/full_inference_bench.py --gpus N [--reps 10] [--warmup 2] [--out FILE]

Prints one JSON line: the GPU and its power limit, then per arithmetic mode (fp16 = the headline mode, tf32, bf16) the time of
inference over all vertices and over a 15 % test split (CUDA events, median / min / max of --reps calls after --warmup), the
per-stage times of one profiled call, the segment max's algorithmic bytes and rate against the measured HBM copy peak, the GEMMs'
TFLOP/s, and the sampled evaluation the trainers run by default (ogl_plan_eval_step in batch_full = 512 chunks) over the same
vertex sets.  The graph, features and weights are bench.py's (same generators and seeds).
With --gpus N: the data-parallel call (parallel.infer_full) in fp16 and tf32, per rank (see sharded()).
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

HBM_COPY_GBS = 6556.8        # measured HBM copy bandwidth of a B200 (BASELINE.md, section 3)
BATCH_FULL = 512             # the trainers' default evaluation chunk


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        pl, clk = (x.strip() for x in r.stdout.strip().split(","))
        info.update(power_limit=pl, max_sm_clock=clk)
    except Exception as e:                     # (the numbers below still stand; the card's limit is then unknown)
        info.update(power_limit="unknown (%s)" % e)
    return info


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median_ms": float(np.median(ms)), "min_ms": float(min(ms)), "max_ms": float(max(ms)), "reps": reps}


def sharded(args):
    """--gpus N under torchrun: parallel.infer_full, every rank computing its edge-balanced share of the rows, in fp16 and tf32.
    Per rank: the call over all vertices and over the 15 % split, the time spent in the row exchange (allgather_rows: NCCL
    broadcasts, CUDA events around each exchange), and the per-stage times of one profiled call (its segment max covers only the
    rank's rows, the pool GEMMs every row)."""
    import torch.distributed as dist
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    assert dist.get_world_size() == args.gpus, "run --gpus N under torchrun --nproc-per-node N"
    import ogl_b200
    from ogl_b200 import parallel
    w, g, feats, labels, flat0, test, E_dir = setup(dev)
    V, F, C, H = w["V"], w["F"], w["C"], w["H"]
    bounds = parallel.edge_balanced_bounds(g.degrees())
    me = {"rank": parallel.rank(), "rows": bounds[parallel.rank() + 1] - bounds[parallel.rank()], "modes": {}}
    ex_ms = []

    def exchange(table, b):
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        parallel.allgather_rows(table, b)
        e.record()
        ex_ms.append((a, e))

    for name, mode in (("fp16", ogl_b200.OGL_FP16), ("tf32", ogl_b200.OGL_TF32)):
        fs, plan = make_plan(w, mode, feats, labels, flat0)
        ref = plan.infer_full(g, fs)
        got = parallel.infer_full(plan, g, fs, exchange=exchange)
        r = {"equal_to_one_rank": bool(torch.equal(got, ref))}
        del ref, got
        for key, ids in (("all_vertices", None), ("test_split_15pct", test)):
            ex_ms.clear()
            r[key] = timed(lambda: parallel.infer_full(plan, g, fs, ids, exchange=exchange), args.reps, args.warmup)
            torch.cuda.synchronize()
            per_call = np.array([a.elapsed_time(e) for a, e in ex_ms]).reshape(args.reps + args.warmup, -1)[args.warmup:].sum(1)
            r[key]["allgather_rows_median_ms"] = float(np.median(per_call))
        r["all_vertices"]["vertices_per_s"] = V / (r["all_vertices"]["median_ms"] / 1e3)
        dist.barrier()
        plan.profile(True)
        parallel.infer_full(plan, g, fs, exchange=parallel.allgather_rows)
        stages, _, _ = plan.profile_read()
        plan.profile(False)
        r["stages_ms"] = {k: round(v[0], 4) for k, v in stages.items()}
        me["modes"][name] = r
        del plan, fs
        torch.cuda.empty_cache()
    every = [None] * dist.get_world_size()
    dist.all_gather_object(every, me)
    if dist.get_rank() == 0:
        out = {"workload": "reddit-shaped synthetic graph of bench.py: V=%d, %d directed edges, F=%d, hidden %d, C=%d, 2 layers, max-pool; "
                           "data-parallel full inference (parallel.infer_full) on %d GPUs" % (V, E_dir, F, H, C, args.gpus),
               "gpu": gpu_info(), "gpus": args.gpus, "bounds": bounds, "ranks": every}
        emit(out, args.out)
    dist.destroy_process_group()


def setup(dev):
    """bench.py's Reddit-shaped graph (streamed in), features, weights and the 15 % test split"""
    from ogl_b200 import native
    w = bench.WORKLOADS["reddit"]
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
    test = torch.as_tensor(np.random.default_rng(5).permutation(V)[: int(0.15 * V)], dtype=torch.int64, device=dev)
    return w, g, feats, labels, flat0, test, g.num_edges


def make_plan(w, mode, feats, labels, flat0):
    from ogl_b200 import native
    fs = native.Features(w["V"], w["F"], mode)
    fs.write(0, feats, labels)
    plan = native.Plan([w["F"], w["H"], w["C"]], w["fanouts"], BATCH_FULL, w["V"], mode=mode, seed=5)
    flat = flat0.clone()
    plan.bind_params(flat, torch.zeros_like(flat))
    return fs, plan


def emit(out, path):
    line = json.dumps(out)
    print(line)
    if path:
        with open(path, "w") as f:
            f.write(line + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sampled-reps", type=int, default=3)
    ap.add_argument("--gpus", type=int, default=0,
                    help="N: data-parallel inference under torchrun --nproc-per-node N (default: the one-GPU call and its stages)")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "full_inference_bench needs a GPU"
    if args.gpus:
        return sharded(args)
    import ogl_b200

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    w, g, feats, labels, flat0, test, E_dir = setup(dev)
    V, F, C, H = w["V"], w["F"], w["C"], w["H"]
    dims = [F, H, C]
    pitch = [(d + 7) // 8 * 8 for d in dims]
    out = {"workload": "reddit-shaped synthetic graph of bench.py: V=%d, %d directed edges (mean in-degree %.0f), F=%d, hidden %d, C=%d, "
                       "2 layers, max-pool" % (V, E_dir, E_dir / V, F, H, C),
           "gpu": gpu_info(), "hbm_copy_peak_gbs": HBM_COPY_GBS, "modes": {}}
    deg = g.degrees()
    out["degrees"] = {"max": int(deg.max()), "zero": int((deg == 0).sum()), "above_chunk_2048": int((deg > 2048).sum())}
    for name, mode in (("fp16", ogl_b200.OGL_FP16), ("tf32", ogl_b200.OGL_TF32), ("bf16", ogl_b200.OGL_BF16)):
        es = 4 if mode == ogl_b200.OGL_TF32 else 2
        fs, plan = make_plan(w, mode, feats, labels, flat0)
        logits = torch.empty(V, C, device=dev)
        logits_t = torch.empty(test.numel(), C, device=dev)
        r = {"all_vertices": timed(lambda: plan.infer_full(g, fs, logits_out=logits), args.reps, args.warmup),
             "test_split_15pct": timed(lambda: plan.infer_full(g, fs, test, logits_out=logits_t), args.reps, args.warmup)}
        r["all_vertices"]["vertices_per_s"] = V / (r["all_vertices"]["median_ms"] / 1e3)
        assert bool(torch.isfinite(logits).all())
        # per-stage times of one call over all vertices (every stage alone on the device, CUDA events around it)
        plan.profile(True)
        plan.infer_full(g, fs, logits_out=logits)
        stages, _, _ = plan.profile_read()
        plan.profile(False)
        r["stages_ms"] = {k: round(v[0], 4) for k, v in stages.items()}
        roof = {}
        for l in range(2):
            fin, fout = dims[l], dims[l + 1]
            seg_bytes = E_dir * pitch[l] * es + E_dir * 8 + V * pitch[l] * es
            ms = stages["full.l%d.segmax" % l][0]
            frac = seg_bytes / ms / 1e6 / HBM_COPY_GBS
            roof["l%d.segmax" % l] = {"bytes": seg_bytes, "ms": ms, "gbs": seg_bytes / ms / 1e6, "of_hbm_copy_peak": frac,
                                      "bound": "memory: one [%d] row of x per edge from a %.0f MB table (L2: 126 MB)%s" % (
                                          pitch[l], V * pitch[l] * es / 1e6,
                                          "; the algorithmic rate is above the HBM copy peak, so part of the row reads are L2 hits "
                                          "(power-law sources are read many times)" if frac > 1 else "")}
            for st, flops in (("pool_gemm", 2.0 * V * fin * fin), ("out_gemm", 2.0 * V * 2 * fin * fout)):
                ms = stages["full.l%d.%s" % (l, st)][0]
                roof["l%d.%s" % (l, st)] = {"flops": flops, "ms": ms, "tflops": flops / ms / 1e9}
        r["roofline"] = roof
        # the trainers' default evaluation over the same vertex sets: sampled 2-hop neighbourhoods, batch_full chunks
        every = torch.arange(V, dtype=torch.int64, device=dev)

        def sampled(ids, outl):
            for i in range(0, ids.numel(), BATCH_FULL):
                plan.eval_step(g, fs, ids[i:i + BATCH_FULL], logits_out=outl[i:i + BATCH_FULL])

        r["sampled_eval_all_vertices"] = timed(lambda: sampled(every, logits), args.sampled_reps, 1)
        r["sampled_eval_test_split_15pct"] = timed(lambda: sampled(test, logits_t), args.sampled_reps, 1)
        out["modes"][name] = r
        del plan, fs
        torch.cuda.empty_cache()
    emit(out, args.out)


if __name__ == "__main__":
    main()
