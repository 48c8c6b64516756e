#!/usr/bin/env python
"""PBR priority recomputation (PrioritizedPytorchSupervisedGraphSage.recompute_priorities) on the Reddit-shaped workload of bench.py,
with priority_neighbourhood="sampled" (eval_step over batch_full chunks of sampled neighbourhoods) and "full" (GraphSAGE.inference_loss).

    python tools/priority_bench.py [--reps 10] [--warmup 2] [--out FILE]
    torchrun --nproc-per-node N tools/priority_bench.py --gpus N [--reps 10] [--warmup 2] [--out FILE]

The graph and features are bench.py's (same generators and seeds), the weights the model's initialisation; the trainer takes settings/reddit.json's batch_full,
samples and embedding size, fp16 arithmetic and the on-device priority route (LossPriority, fast choosers).  The train split is the
driver's: 85 % of the vertices.  Two cases, each the median of --reps calls after --warmup calls (CUDA events around the call, which
includes building the id lists and pushing the losses into the sum tree; "losses_only" times the loss computation alone):
  (a) train_set:       every train vertex -- the priority_forward timestep;
  (b) new_train_nodes: one snapshot's new train vertices (85 % of V / snapshots) -- the other timesteps.
Also the per-stage times of one call of each option, and with --gpus N (full option only; the sampled one is not sharded) the time
each rank spends in the exchanges of parallel.infer_full_loss.  Prints one JSON line."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
from full_inference_bench import emit, gpu_info, timed  # noqa: E402


class _Graph:
    """the DeviceGraph surface the trainer and the model use: the native graph, the feature store, capacity and mode"""

    def __init__(self, g, fs, V, mode):
        self.native, self.features, self.v_cap, self.mode = g, fs, V, mode


def _graph_util(graph, train, V):
    """TrainTestGraph's priority surface over a fixed graph and train split (no temporal graph behind it)"""
    from ogl_b200.graph.train_test_graph import TrainTestGraph

    class GU(TrainTestGraph):
        def __init__(self):
            self.prior_alpha, self.max_priority, self.min_priority = 4, 10, 0.0000001
            self._tree_backend, self._verbose = None, False
            self.train_set, self.train_set_list = set(train), list(train)
            self.priority_replay_buffer = self._new_buffer()
            self.priority_replay_buffer.add_all({v: 2 for v in train})

        def get_graph(self):
            return graph

        def get_original_to_subgraph_map(self):
            return np.arange(V)

    return GU()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--gpus", type=int, default=0, help="N: data-parallel under torchrun --nproc-per-node N")
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "priority_bench needs a GPU"
    dist = None
    if args.gpus:
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0"))
        dev = torch.device("cuda", local)
        torch.cuda.set_device(dev)
        dist.init_process_group("nccl", device_id=dev)
        assert dist.get_world_size() == args.gpus, "run --gpus N under torchrun --nproc-per-node N"
    else:
        dev = torch.device("cuda", 0)
        torch.cuda.set_device(dev)
    import ogl_b200
    from ogl_b200 import config, native, parallel
    from ogl_b200.graph import train_test_graph as ttg
    settings = json.load(open(os.path.join(ROOT, "settings", "reddit.json")))
    config.set_precision("fp16")
    config.set_faithful(False)
    w = bench.WORKLOADS["reddit"]
    V, E, F, C, H = w["V"], w["E"], w["F"], w["C"], settings["embedding_size"]
    src, dst = bench.gen_edges(w, dev)
    g = native.Graph(V, 2 * E)
    g.insert_vertices(V)
    chunk = max(1 << 14, min(1 << 21, E // 16))
    for a in range(0, E, chunk):
        g.insert_edges(src[a:a + chunk], dst[a:a + chunk], symmetric=True)
    del src, dst
    feats, labels = bench.gen_features(w, dev)
    fs = native.Features(V, F, ogl_b200.OGL_FP16)
    fs.write(0, feats, labels)
    del feats
    graph = _Graph(g, fs, V, ogl_b200.OGL_FP16)
    # the driver's split (train_test_split, test_size 0.15) and one snapshot's share of it
    perm = np.random.default_rng(5).permutation(V)
    train = perm[int(0.15 * V):].tolist()
    new_train = train[:max(2, len(train) // settings["snapshots"])]
    ttg.SIZE_BUFFER = 1 << 18
    GraphSAGE, _, PrioT, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, dev.index)
    torch.manual_seed(1)
    model = GraphSAGE(F, H, C, 1, act, 0, "pool").cuda()
    out = {"workload": "reddit-shaped synthetic graph of bench.py: V=%d, %d directed edges, F=%d, hidden %d, C=%d, 2 layers, max-pool; "
                       "fp16; recompute_priorities with batch_full=%d, samples=%d (settings/reddit.json)"
                       % (V, g.num_edges, F, H, C, settings["batch_full"], settings["samples"]),
           "gpu": gpu_info(), "gpus": max(args.gpus, 1), "train_vertices": len(train), "new_train_vertices": len(new_train),
           "options": {}}
    for option in ("sampled", "full"):
        t = PrioT(model, settings["batch_timestep"], settings["batch_size"], labels, settings["samples"], ogl_b200.LossPriority(),
                  full_pass=settings["priority_forward"], cuda=True, batch_full=settings["batch_full"], n_workers=0,
                  priority_neighbourhood=option)
        gu = _graph_util(graph, train, V)
        r = {}
        plan = model.inference_plan(graph) if option == "full" else t._eval_plan(graph)

        def losses_only(ids):
            """the loss computation of recompute_priorities alone, without the sum-tree push and the host-side id lists"""
            if option == "full":
                return model.inference_loss(graph, ids, distributed=parallel.world() > 1)
            out = torch.empty(ids.numel(), device=dev)
            for i in range(0, ids.numel(), t.batch_full):
                plan.eval_step(g, fs, ids[i:i + t.batch_full], per_vertex_out=out[i:i + t.batch_full])
            return out

        for key, vs in (("a_train_set", train), ("b_new_train_nodes", new_train)):
            r[key] = timed(lambda: t.recompute_priorities(gu, vs), args.reps, args.warmup)
            r[key]["vertices_per_s"] = len(vs) / (r[key]["median_ms"] / 1e3)
            ids = torch.as_tensor(vs, dtype=torch.int64, device=dev)
            r[key]["losses_only"] = timed(lambda: losses_only(ids), args.reps, args.warmup)
        for key, vs in (("a_train_set", train), ("b_new_train_nodes", new_train)):
            plan.profile(True)
            t.recompute_priorities(gu, vs)
            stages, _, _ = plan.profile_read()
            plan.profile(False)
            r[key]["stages_ms"] = {k: round(v[0], 4) for k, v in stages.items()}
        if option == "full" and dist is not None:
            # per rank: the time spent in the exchanges of one sharded call (hidden table + losses), CUDA events around each
            ev = []

            def exchange(table, b):
                a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                parallel.allgather_rows(table, b)
                e.record()
                ev.append((a, e))

            for key, vs in (("a_train_set", train), ("b_new_train_nodes", new_train)):
                ids = torch.as_tensor(vs, dtype=torch.int64, device=dev)
                ev.clear()
                timed(lambda: parallel.infer_full_loss(plan, g, fs, ids, exchange=exchange), args.reps, args.warmup)
                torch.cuda.synchronize()
                per_call = np.array([a.elapsed_time(e) for a, e in ev]).reshape(args.reps + args.warmup, -1)[args.warmup:]
                r[key]["exchange_ms_per_call"] = {"hidden_table": float(np.median(per_call[:, :-1].sum(1))),
                                                  "losses": float(np.median(per_call[:, -1]))}
        if dist is not None:
            every = [None] * dist.get_world_size()
            dist.all_gather_object(every, r)
            r = {"ranks": every}
        elif option == "sampled":
            r["note"] = "not sharded: every rank of a torchrun job recomputes every priority by itself"
        out["options"][option] = r
    if dist is None or dist.get_rank() == 0:
        emit(out, args.out)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
