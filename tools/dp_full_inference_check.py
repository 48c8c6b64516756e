"""torchrun --nproc-per-node N tools/dp_full_inference_check.py -- the four drop-in trainers with eval_neighbourhood="full" in
data-parallel mode, where evaluation shares the full-inference rows between the ranks (parallel.infer_full).  After every timestep
each rank evaluates twice on the same weights: sharded over the ranks, and alone (Plan.infer_full on this rank).  Checks:
  rows_equal:   the CSV rows of the two evaluations are identical (F1, confusion matrix, the timestep's delay);
  logits_equal: GraphSAGE.inference(distributed=True) is torch.equal to the one-rank call, for every vertex and for the test set;
  ranks_equal:  every rank holds the same logits.
Prints one JSON line on rank 0."""
import json
import os
import random
import sys
import tempfile

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
    config.set_faithful(True)
    config.set_precision("fp16")
    ttg.SIZE_BUFFER = 1 << 12
    random.seed(1); np.random.seed(1); torch.manual_seed(1)
    V, E, F, C, H = 1200, 9000, 12, 3, 16
    src, dst, x, y = _planted(V, E, F, C, seed=5)
    src, dst, x, y = _relabel_first_appearance(src, dst, x, y)
    GraphSAGE, RandomT, PrioT, NoRehT, FullT, act = ogl_b200.init(ogl_b200.Lib_supported.PYTORCH, True, local)
    dyn = ogl_b200.DynamicGraphEdge(12, set(range(len(x))))
    dyn.build(x, y, edge_timestamps={"src": src, "dst": dst})
    gu = ttg.TrainTestGraph(dyn, split=0.15, start_prior_alpha=4, end_prior_alpha=50, scale=1, max_priority=10)
    mk = lambda: GraphSAGE(F, H, C, 1, act, 0, "pool").cuda()
    kw = dict(cuda=True, batch_full=128, n_workers=0, eval_neighbourhood="full")
    trainers = [RandomT(mk(), 25, 32, y, 5, **kw), PrioT(mk(), 25, 32, y, 5, ogl_b200.LossPriority(), full_pass=2, **kw),
                NoRehT(mk(), 25, 32, y, 5, **kw), FullT(mk(), 1, 32, y, 5, **kw)]
    for t in trainers:
        t.build_optimizer()
    out = tempfile.mkdtemp()
    sharded, alone = os.path.join(out, "sharded.csv"), os.path.join(out, "alone.csv")
    world = parallel.world
    logits_equal = ranks_equal = True
    for step in range(6):
        for t in trainers:
            t.train_timestep(gu)
        for t in trainers:
            t.evaluate(gu, sharded)
            parallel.world = lambda: 1           # the same evaluation on this rank alone (the trainers ask parallel.world())
            try:
                t.evaluate(gu, alone)
            finally:
                parallel.world = world
        graph = gu.get_graph()
        test = torch.as_tensor(np.asarray(gu.get_original_to_subgraph_map()[np.array(gu.get_test_set())], dtype=np.int64), device="cuda")
        for t in trainers:
            m = t.graphsage_model
            for v in (None, test):
                d = m.inference(graph, v, distributed=True)
                one = m.inference_plan(graph).infer_full(graph.native, graph.features, seeds=v)
                same = _same_on_every_rank(d)          # (a collective: every rank makes the call)
                logits_equal = logits_equal and torch.equal(d, one)
                ranks_equal = ranks_equal and same
        if step + 1 < len(gu):
            gu.evolve()
    rows_s, rows_a = open(sharded).read().splitlines(), open(alone).read().splitlines()
    ok = torch.tensor([int(rows_s == rows_a and len(rows_s) > 0), int(logits_equal), int(ranks_equal)], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if dist.get_rank() == 0:
        print(json.dumps({"world": dist.get_world_size(), "rows_equal": bool(ok[0]), "logits_equal": bool(ok[1]),
                          "ranks_equal": bool(ok[2]), "rows": len(rows_s), "f1": [r.split(";")[1] for r in rows_s[-len(trainers):]]}))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
