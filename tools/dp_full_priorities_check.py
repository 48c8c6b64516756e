"""torchrun --nproc-per-node N tools/dp_full_priorities_check.py -- the PBR trainer with priority_neighbourhood="full" in data-parallel
mode, where recompute_priorities shares the full-inference rows between the ranks and exchanges only the losses
(parallel.infer_full_loss).  After every timestep each rank recomputes the priorities of the whole train set twice on the same
weights: sharded over the ranks, and alone (Plan.infer_full_loss on this rank).  Checks:
  trees_equal:  the priorities of the train set after the two recomputes are identical;
  losses_equal: GraphSAGE.inference_loss(distributed=True) is torch.equal to the one-rank call;
  ranks_equal:  every rank holds the same priorities and losses.
Prints one JSON line on rank 0."""
import json
import os
import random
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _same_on_every_rank(t):
    cs = t.contiguous().view(torch.int32).to(torch.int64).sum().reshape(1)
    every = [torch.zeros_like(cs) for _ in range(dist.get_world_size())]
    dist.all_gather(every, cs)
    return all(int(e) == int(every[0]) for e in every)


def main():
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import ogl_b200
    from ogl_b200 import config, parallel
    from ogl_b200.graph import train_test_graph as ttg
    from test_gpu_trainers import _planted, _relabel_first_appearance
    config.set_faithful(False)
    config.set_precision("fp16")
    ttg.SIZE_BUFFER = 1 << 12
    random.seed(1); np.random.seed(1); torch.manual_seed(1)
    V, E, F, C, H = 1200, 9000, 12, 3, 16
    src, dst, x, y = _planted(V, E, F, C, seed=5)
    src, dst, x, y = _relabel_first_appearance(src, dst, x, y)
    GraphSAGE, _, PrioT, _, _, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, local)
    dyn = ogl_b200.DynamicGraphEdge(12, set(range(len(x))))
    dyn.build(x, y, edge_timestamps={"src": src, "dst": dst})
    gu = ttg.TrainTestGraph(dyn, split=0.15, start_prior_alpha=4, end_prior_alpha=50, scale=1, max_priority=10)
    t = PrioT(GraphSAGE(F, H, C, 1, act, 0, "pool").cuda(), 25, 32, y, 5, ogl_b200.LossPriority(), full_pass=2, cuda=True,
              batch_full=128, n_workers=0, priority_neighbourhood="full")
    t.build_optimizer()
    world = parallel.world
    trees_equal = losses_equal = ranks_equal = True
    steps = 6
    for step in range(steps):
        t.train_timestep(gu)                     # (its recompute_priorities runs sharded on even timesteps)
        train = list(gu.get_train_set())
        t.recompute_priorities(gu, train)
        sharded = torch.tensor(gu.dump_priorities(train), dtype=torch.float64, device="cuda")
        parallel.world = lambda: 1               # the same recompute on this rank alone (the trainer asks parallel.world())
        try:
            t.recompute_priorities(gu, train)
        finally:
            parallel.world = world
        alone = torch.tensor(gu.dump_priorities(train), dtype=torch.float64, device="cuda")
        graph = gu.get_graph()
        sub = torch.as_tensor(np.asarray(gu.get_original_to_subgraph_map()[np.array(train)], dtype=np.int64), device="cuda")
        m = t.graphsage_model
        d = m.inference_loss(graph, sub, distributed=True)
        one = m.inference_plan(graph).infer_full_loss(graph.native, graph.features, seeds=sub)
        trees_equal = trees_equal and torch.equal(sharded, alone)
        losses_equal = losses_equal and torch.equal(d, one)
        same_tree, same_loss = _same_on_every_rank(sharded), _same_on_every_rank(d)      # (collectives: every rank calls them)
        ranks_equal = ranks_equal and same_tree and same_loss
        if step + 1 < len(gu):
            gu.evolve()
    ok = torch.tensor([int(trees_equal), int(losses_equal), int(ranks_equal)], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if dist.get_rank() == 0:
        print(json.dumps({"world": dist.get_world_size(), "trees_equal": bool(ok[0]), "losses_equal": bool(ok[1]),
                          "ranks_equal": bool(ok[2]), "timesteps": steps, "train_vertices": len(gu.get_train_set())}))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
