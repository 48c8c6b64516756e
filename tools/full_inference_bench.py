#!/usr/bin/env python
"""Full-neighbourhood inference (GraphSAGE.inference / ogl_plan_infer_full) on the Reddit-shaped workload of bench.py.

    python tools/full_inference_bench.py [--reps 10] [--warmup 2] [--sampled-reps 3] [--out FILE]

Prints one JSON line: the GPU and its power limit, then per arithmetic mode (fp16 = the headline mode, tf32, bf16) the time of
inference over all vertices and over a 15 % test split (CUDA events, median / min / max of --reps calls after --warmup), the
per-stage times of one profiled call, the segment max's algorithmic bytes and rate against the measured HBM copy peak, the GEMMs'
TFLOP/s, and the sampled evaluation the trainers run by default (ogl_plan_eval_step in batch_full = 512 chunks) over the same
vertex sets.  The graph, features and weights are bench.py's (same generators and seeds).
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--sampled-reps", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "full_inference_bench needs a GPU"
    import ogl_b200
    from ogl_b200 import native

    w = bench.WORKLOADS["reddit"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    V, E, F, C, H = w["V"], w["E"], w["F"], w["C"], w["H"]
    src, dst = bench.gen_edges(w, dev)
    g = native.Graph(V, 2 * E)
    g.insert_vertices(V)
    chunk = max(1 << 14, min(1 << 21, E // 16))
    for a in range(0, E, chunk):
        g.insert_edges(src[a:a + chunk], dst[a:a + chunk], symmetric=True)
    del src, dst
    E_dir = g.num_edges
    feats, labels = bench.gen_features(w, dev)
    params = bench.init_params(w)
    flat0 = torch.cat([params["layers.%d.%s" % (i, n)].reshape(-1).float() for i in range(2) for n in bench.NAMES]).to(dev)
    test = torch.as_tensor(np.random.default_rng(5).permutation(V)[: int(0.15 * V)], dtype=torch.int64, device=dev)
    dims = [F, H, C]
    pitch = [(d + 7) // 8 * 8 for d in dims]
    out = {"workload": "reddit-shaped synthetic graph of bench.py: V=%d, %d directed edges (mean in-degree %.0f), F=%d, hidden %d, C=%d, "
                       "2 layers, max-pool" % (V, E_dir, E_dir / V, F, H, C),
           "gpu": gpu_info(), "hbm_copy_peak_gbs": HBM_COPY_GBS, "modes": {}}
    deg = g.degrees()
    out["degrees"] = {"max": int(deg.max()), "zero": int((deg == 0).sum()), "above_chunk_2048": int((deg > 2048).sum())}
    for name, mode in (("fp16", ogl_b200.OGL_FP16), ("tf32", ogl_b200.OGL_TF32), ("bf16", ogl_b200.OGL_BF16)):
        es = 4 if mode == ogl_b200.OGL_TF32 else 2
        fs = native.Features(V, F, mode)
        fs.write(0, feats, labels)
        plan = native.Plan(dims, w["fanouts"], BATCH_FULL, V, mode=mode, seed=5)
        flat = flat0.clone()
        plan.bind_params(flat, torch.zeros_like(flat))
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
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
