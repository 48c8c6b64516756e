"""`python train <dataset> pytorch <result.csv> <tsne_dir> --cuda [...]` -- the reference's command line
(train/__main__.py:14-49,97-207 of MassimoPerini/online-gnn-learning) over the B200 path (SURVEY 8(f)-1).

Same positional / optional arguments, same overlay of the command line on settings/<dataset>.json, same loop: four
models (random / prioritized / no_rehersal / offline rehearsal policies) trained in lock-step on one TrainTestGraph,
evaluated every `eval` snapshots on the current test set and on the graph `delta` snapshots ahead, rows appended to
the result CSV as `model;f1;delay;confusion`.  Only the pytorch backend with --cuda exists here (no CPU fallback);
TSNE plotting is not built (the reference's only call site is commented out, :188-189).
"""
import argparse
import gc
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

START_PRIOR_ALPHA = 4
END_PRIOR_ALPHA = 50
SCALE = 1


def parse(argv=None):
    ap = argparse.ArgumentParser(prog="train")
    ap.add_argument("dataset", choices=["elliptic", "pubmed", "reddit", "arxiv"], help="Dataset")
    ap.add_argument("backend", choices=["pytorch"], help="Framework (only the pytorch/CUDA path is built here)")
    ap.add_argument("save_result", help="output file (.csv)")
    ap.add_argument("save_tsne", help="path tsne plots (unused)")
    ap.add_argument("--cuda", action="store_true", help="Enable CUDA (required)")
    ap.add_argument("--gpu", type=int, default=-1, help="Use a specific GPU")
    for name, typ in (("snapshots", int), ("embedding_size", int), ("latent_dim", int), ("depth", int), ("samples", int),
                      ("batch_timestep", int), ("eval", int), ("batch_size", int), ("batch_full", int), ("epochs_offline", int),
                      ("train_offline", int), ("priority_forward", int), ("plot_tsne", int), ("dropout", float), ("delta", int)):
        ap.add_argument("--" + name, type=typ)
    ap.add_argument("--n_sampling_workers", type=int, default=0, help="accepted and ignored: sampling runs on the GPU")
    ap.add_argument("--copy_dataset_gpu", action="store_true", help="accepted: the dataset always lives on the GPU here")
    # extensions (not in the reference)
    ap.add_argument("--path", help="dataset directory (overrides settings/<dataset>.json)")
    ap.add_argument("--max_timesteps", type=int, help="stop after N snapshots")
    ap.add_argument("--precision", choices=["bf16", "tf32", "fp16", "fp32"], default="tf32",
                    help="arithmetic of the dense path: tf32 (default: tensor cores, rtol 1e-3 vs the reference's fp32, fp32 range), bf16 (fastest, ~5e-3), "
                         "fp16 (tf32's error at bf16's speed; loss-scaled, standardised features), fp32 (exact, SIMT)")
    ap.add_argument("--fast_choosers", action="store_true", help="on-GPU counter-RNG draws / proportional PBR instead of the literal reference choosers")
    ap.add_argument("--eval_neighbourhood", choices=["sampled", "full"], default="sampled",
                    help="neighbourhoods the F1 evaluation scores vertices from: sampled (the reference's fan-outs) or full (every in-edge, "
                         "GraphSAGE.inference: exact and independent of the sampler)")
    ap.add_argument("--priority_neighbourhood", choices=["sampled", "full"], default="sampled",
                    help="neighbourhoods the prioritized model's priority recomputation scores the train vertices from: sampled (the "
                         "reference's fan-outs) or full (every in-edge, GraphSAGE.inference_loss: exact, no sampling noise)")
    args = ap.parse_args(argv)
    custom = {k: v for k, v in vars(args).items() if v is not None}
    with open(os.path.join(ROOT, "settings", args.dataset + ".json")) as f:
        data = json.load(f)
    data.update(custom)                      # the command line wins (reference :45-49)
    return args, data


def run(args, data):
    import numpy as np
    import ogl_b200
    from ogl_b200 import config, dataset_utils
    from ogl_b200.graph.train_test_graph import TrainTestGraph

    if not data["cuda"]:
        raise SystemExit("ogl_b200 is the `--cuda` path of the reference; pass --cuda (there is no CPU fallback)")
    # data-parallel run: `torchrun --nproc-per-node N train ...` -- one process per GPU, replicated graph / model / choosers (same
    # seeds on every rank), every minibatch sharded over the ranks, gradients summed over NCCL (ogl_b200.parallel, SURVEY 8(e))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        import torch
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        data["gpu"] = local
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        torch.manual_seed(1)                 # torch.randperm of the offline / no-rehearsal policies must agree across the ranks
        if dist.get_rank() != 0:
            data["save_result"] = None       # rank 0 writes the CSV; the replicas evaluate the same numbers
    config.set_precision(data["precision"])
    config.set_faithful(not data["fast_choosers"])
    print("init")
    GraphSAGE, RandomT, PrioritizedT, NoRehT, FullT, activation = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, data["cuda"], data["gpu"])
    print("load data")
    feat_size, labels, graph, n_classes, dynamic_graph_test = dataset_utils.LOADERS[args.dataset](
        data["path"], snapshots=data["snapshots"], cuda=data["cuda"], copy_to_gpu=data["copy_dataset_gpu"])
    for _ in range(data["delta"]):
        dynamic_graph_test.evolve()
    print("train test init")
    graph_util = TrainTestGraph(graph, split=0.15, start_prior_alpha=START_PRIOR_ALPHA, end_prior_alpha=END_PRIOR_ALPHA, scale=SCALE,
                                max_priority=10)
    print("create graphsage")
    mk = lambda: GraphSAGE(feat_size, data["embedding_size"], n_classes, data["depth"] - 1, activation, data["dropout"], "pool",
                           edge_feats=data["edge_feats"], pool_feats=data["latent_dim"]).cuda()
    kw = dict(cuda=data["cuda"], batch_full=data["batch_full"], n_workers=data["n_sampling_workers"],
              eval_neighbourhood=data["eval_neighbourhood"])
    t_random = RandomT(mk(), data["batch_timestep"], data["batch_size"], labels, data["samples"], **kw)
    t_priority = PrioritizedT(mk(), data["batch_timestep"], data["batch_size"], labels, data["samples"], ogl_b200.LossPriority(),
                              full_pass=data["priority_forward"], priority_neighbourhood=data["priority_neighbourhood"], **kw)
    t_no_reh = NoRehT(mk(), data["batch_timestep"], data["batch_size"], labels, data["samples"], **kw)
    t_full = FullT(mk(), data["epochs_offline"], data["batch_size"], labels, data["samples"], **kw)
    trainers = [t_random, t_priority, t_no_reh, t_full]
    for t in trainers:
        t.build_optimizer()
    size_evolution = len(graph_util)
    if data.get("max_timesteps"):
        size_evolution = min(size_evolution, data["max_timesteps"])
    print(size_evolution)
    for time_step in range(size_evolution):
        print("processing time step: ", time_step)
        t_random.train_timestep(graph_util)
        t_priority.train_timestep(graph_util)
        t_no_reh.train_timestep(graph_util)
        if time_step % data["train_offline"] == 0:
            print("train offline")
            t_full.train_timestep(graph_util)
        if time_step % data["eval"] == 0:
            for t in trainers:
                t.evaluate(graph_util, data["save_result"])
            for t in trainers:
                t.evaluate_next_snapshots(dynamic_graph_test, data["delta"], data["save_result"])
        if time_step + data["delta"] + 1 < len(graph_util):
            print("evolving...")
            graph_util.evolve()
            dynamic_graph_test.evolve()
            gc.collect()
    return trainers


if __name__ == "__main__":
    import numpy as np
    _args, _data = parse()
    print(_args)
    np.random.seed(1)              # the reference seeds numpy and `random` only (:211-212)
    random.seed(1)
    run(_args, _data)
