"""The four training policies on the B200 path (mirror of train/graphsage/pytorch/model.py:12-323).

Where the reference builds a DGL sampler + DataLoader per call, gathers features on the CPU, copies
them over PCIe and runs DGL/cuBLAS kernels (:77-107), every minibatch here is ONE C call
(`ogl_plan_train_step`): seeds go host->device (8 bytes each), everything else -- sampling, to_block,
feature gather, the GraphSAGE-pool forward/backward, CE loss, Adam -- stays on the GPU with no host
synchronisation.  Per-vertex losses for PBR come back only in faithful mode.
"""
import numpy as np
import torch

from ... import config, parallel, utils
from ...sampling import MultiLayerNeighborSampler, NodeDataLoader
from ..model import SupervisedGraphSage


class _FusedAdam:
    """`trainer.optimizer` look-alike: Adam(lr=1e-3) state lives in the training plan (pytorch/model.py:25)."""

    def __init__(self, trainer):
        self._t = trainer

    def zero_grad(self):
        pass

    def step(self):
        plan = self._t._last_plan
        plan.adam_step()
        self._t.graphsage_model.mark_updated(plan)


class PytorchSupervisedGraphSage(SupervisedGraphSage):
    def __init__(self, graphsage_model, batch_per_timestep, batch_size, labels, samples, reduction="mean", n_workers=1,
                 cuda=False, batch_full=512, fanouts=None, eval_neighbourhood="sampled"):
        if not cuda:
            raise RuntimeError("ogl_b200 trainers are the `--cuda` path; there is no CPU fallback")
        if eval_neighbourhood not in ("sampled", "full"):
            raise ValueError("eval_neighbourhood must be 'sampled' or 'full', got %r" % (eval_neighbourhood,))
        # "full": evaluate / evaluate_next_snapshots score every vertex from its whole in-neighbourhood (GraphSAGE.inference), which makes
        # the F1 columns independent of the sampler; "sampled" (the reference's behaviour): fan-out-sampled neighbourhoods
        self.eval_neighbourhood = eval_neighbourhood
        super().__init__(graphsage_model, batch_per_timestep, batch_size, labels, samples, n_workers, cuda, batch_full)
        self.reduction = reduction
        n_layers = len(graphsage_model.layers)
        # the reference samples [samples]*2 (one int for both hops); per-hop fan-outs are an opt-in extension
        self.hop_fanouts = list(fanouts) if fanouts is not None else [samples] * n_layers
        self.optimizer = None
        self._last_plan = None
        self._pin = None
        self._pin_busy = None          # event recorded after the last launch that reads the pinned seed buffer

    def build_optimizer(self):
        self.optimizer = _FusedAdam(self)

    def get_model(self):
        return "base_model"

    # ---- plans / staging ---------------------------------------------------------------------------
    def _train_plan(self, graph):
        return self.graphsage_model.plan_for(graph, self.hop_fanouts, max(self.batch_size, 1))

    def _eval_plan(self, graph):
        return self.graphsage_model.plan_for(graph, self.hop_fanouts, max(self.batch_full, 1))

    def _host_seeds(self, vertices):
        """pinned int64 staging buffer for the seed ids (the only per-step host->device payload)"""
        if isinstance(vertices, torch.Tensor) and vertices.is_cuda:
            return vertices.to(torch.int64).contiguous()
        v = torch.as_tensor(np.asarray(vertices, dtype=np.int64))
        if self._pin_busy is not None:
            self._pin_busy.synchronize()                # an earlier async H2D copy may still be reading the buffer
            self._pin_busy = None
        if self._pin is None or self._pin.numel() < v.numel():
            self._pin = torch.empty(max(v.numel(), 1024), dtype=torch.int64).pin_memory()
        self._pin[:v.numel()].copy_(v)
        return self._pin[:v.numel()]

    # ---- evaluation (reference :39-71) -------------------------------------------------------------
    def _eval_logits_device(self, graph, test_vertices):
        """eval-mode forward over `test_vertices` in batch_full chunks (or, with eval_neighbourhood="full", over their whole
        neighbourhoods); logits [n, C] stay on the device"""
        self.graphsage_model.eval()
        if self.eval_neighbourhood == "full":
            v = torch.as_tensor(np.asarray(test_vertices, dtype=np.int64)).cuda()
            if v.numel() == 0:
                return None
            # under torchrun every rank evaluates in lock-step on the same graph and weights: the ranks share the rows
            out = self.graphsage_model.inference(graph, v, distributed=parallel.world() > 1)
            if self.graphsage_model.inference_plan(graph).error_flags() & 1:
                raise IndexError("a vertex id outside the graph was evaluated (DGL's NodeDataLoader raises on such ids)")
            return out
        seeds = self._host_seeds(test_vertices)
        n = seeds.numel()
        if n == 0:
            return None
        plan = self._eval_plan(graph)
        C = self.graphsage_model.dims[-1]
        out = torch.empty(n, C, dtype=torch.float32, device="cuda")
        for i in range(0, n, self.batch_full):
            chunk = seeds[i:i + self.batch_full]
            plan.eval_step(graph.native, graph.features, chunk, logits_out=out[i:i + chunk.numel()])
        self._mark_pin_busy(seeds)
        if plan.error_flags() & 1:                       # (synchronises: evaluation reads its result back right after anyway)
            raise IndexError("a vertex id outside the graph was evaluated (DGL's NodeDataLoader raises on such ids)")
        return out

    def _run_custom_eval(self, graph, subgraph_to_id, id_to_subgraph, test_vertices):
        """the reference's hook (:39-71): a list of host arrays [<= batch_full, C].  _evaluate_vertices itself uses
        _eval_logits_device + the on-GPU confusion matrix and only falls back to this hook when a subclass overrides it."""
        out = self._eval_logits_device(graph, test_vertices)
        if out is None:
            return []
        host = out.cpu().numpy()
        return [host[i:i + self.batch_full] for i in range(0, host.shape[0], self.batch_full)]

    _base_run_custom_eval = _run_custom_eval

    # ---- one minibatch -----------------------------------------------------------------------------
    def _fused_step(self, graph, seeds, per_vertex_out=None, loss_sum_out=None):
        plan = self._train_plan(graph)
        if parallel.world() > 1:
            return self._dp_steps(graph, plan, seeds, seeds.numel(), per_vertex_out)
        plan.train_step(graph.native, graph.features, seeds, loss_scale=1.0 / seeds.numel(), do_step=True,
                        per_vertex_out=per_vertex_out, loss_sum_out=loss_sum_out)
        self.graphsage_model.mark_updated(plan)
        self._last_plan = plan
        self._mark_pin_busy(seeds)

    def _mark_pin_busy(self, seeds):
        if not seeds.is_cuda:
            self._pin_busy = torch.cuda.Event()
            self._pin_busy.record()

    def _fused_steps(self, graph, seeds, batch, per_vertex_out=None):
        """all full minibatches of `batch` seeds in ONE C call (no host round trip between steps), then the ragged tail"""
        batch = max(int(batch), 1)
        n = seeds.numel()
        n_full = n // batch
        plan = self._train_plan(graph)
        if parallel.world() > 1:
            return self._dp_steps(graph, plan, seeds, batch, per_vertex_out)
        if n_full:
            plan.train_steps(graph.native, graph.features, seeds[:n_full * batch], batch, loss_scale=1.0 / batch, do_step=True,
                             per_vertex_out=None if per_vertex_out is None else per_vertex_out[:n_full * batch])
            self.graphsage_model.mark_updated(plan)
            self._last_plan = plan
            self._mark_pin_busy(seeds)
        if n > n_full * batch:
            tail = seeds[n_full * batch:]
            self._fused_step(graph, tail, per_vertex_out=None if per_vertex_out is None else per_vertex_out[n_full * batch:])

    def _dp_steps(self, graph, plan, seeds, batch, per_vertex_out):
        """data-parallel twin of the loop above (one process per GPU, torchrun; SURVEY 8(e)): every rank holds the same graph, model
        and -- because the choosers run on identically seeded RNGs -- the same `seeds`; of each minibatch a rank trains its
        contiguous shard (parallel.shard) with the loss scaled by 1 / global minibatch size, the flat gradients are summed over
        the ranks (NCCL all-reduce, bucketed and overlapped by parallel.Pipeline) and every replica takes the same Adam step.
        Per-vertex losses (PBR) are all-gathered so that every rank applies identical priority updates."""
        w = parallel.world()
        if getattr(self, "_dp_pipe_plan", None) is not plan:
            self._dp_pipe = parallel.Pipeline(plan, graph.native, graph.features, self.graphsage_model._flat_grad, batch)
            self._dp_pipe_plan = plan
        pipe = self._dp_pipe
        n = seeds.numel()
        jobs = []                                                  # (global lo, global hi, local lo, local hi)
        for lo in range(0, n, batch):
            hi = min(lo + batch, n)
            if hi - lo >= w:
                sl = parallel.shard(range(lo, hi))
                jobs.append((lo, hi, sl[0], sl[-1] + 1))
            else:                                                  # fewer seeds than ranks: every rank trains all of them, scaled by 1 / w
                jobs.append((lo, hi, lo, hi))
        per_local = None
        if per_vertex_out is not None:
            per_local = torch.empty(sum(j[3] - j[2] for j in jobs), dtype=torch.float32, device="cuda")
        pipe.begin(seeds[jobs[0][2]:jobs[0][3]])
        off = 0
        for i, (lo, hi, a, b) in enumerate(jobs):
            nxt = seeds[jobs[i + 1][2]:jobs[i + 1][3]] if i + 1 < len(jobs) else None
            scale = 1.0 / (hi - lo) if hi - lo >= w else 1.0 / ((hi - lo) * w)
            pipe.finish(nxt, per_vertex_out=None if per_local is None else per_local[off:off + b - a], scale=scale)
            off += b - a
        pipe.flush()
        self.graphsage_model.mark_updated(plan)
        self._last_plan = plan
        self._mark_pin_busy(seeds)
        if per_vertex_out is not None:
            pos = torch.cat([torch.arange(a, b, device="cuda") for (_, _, a, b) in jobs])
            all_pos, all_loss = parallel.allgather_losses(pos, per_local)
            per_vertex_out[all_pos] = all_loss

    def train_step(self, graph, blocks, input_nodes, seeds, subgraph_to_id):
        """DGL-style signature of the reference (:77-107): one optimiser step on the minibatch `blocks` describes.  Blocks that were
        sampled by this trainer's own train plan and are still current (NodeDataLoader(..., plan=self._train_plan(graph))) are
        trained AS GIVEN -- forward, loss, backward and Adam run over the neighbourhoods those blocks hold; any other blocks
        (another plan's, or stale ones) cannot be replayed, so a fresh minibatch is sampled for `seeds` and the call says so."""
        plan = self._train_plan(graph)
        seeds = seeds.to("cuda", torch.int64).contiguous()
        blk = blocks[0] if blocks else None
        if blk is not None and getattr(blk, "_plan", None) is plan and getattr(blk, "_stamp", None) == plan._stamp and \
                plan.n_seeds == seeds.numel():
            plan.set_option("train_mode", 1)
            plan.forward(graph.features, want_logits=False)
            plan.loss_backward(graph.features, 1.0 / seeds.numel(), want_per_vertex=False)
            plan.set_option("train_mode", 0)
            plan.adam_step()
            self.graphsage_model.mark_updated(plan)
            self._last_plan = plan
            return "trained on the given blocks"
        self._fused_step(graph, seeds)
        return "resampled"

    def _batches(self, vertices, batch):
        seeds = self._host_seeds(vertices)
        batch = max(int(batch), 1)
        return [seeds[i:i + batch] for i in range(0, seeds.numel(), batch)]


class RandomPytorchSupervisedGraphSage(PytorchSupervisedGraphSage):
    """RBR: rehearsal on uniformly drawn train vertices (reference :110-138)."""

    def __init__(self, model, batch_per_timestep, batch_size, labels, samples, cuda=False, batch_full=512, n_workers=0, fanouts=None,
                 eval_neighbourhood="sampled"):
        super().__init__(model, batch_per_timestep, batch_size, labels, samples, n_workers=n_workers, cuda=cuda,
                         batch_full=batch_full, fanouts=fanouts, eval_neighbourhood=eval_neighbourhood)

    def choose_vertices(self, graph_util):
        draws = [graph_util.draw_random_train_nodes(self.batch_size) for _ in range(self.batch_per_timestep)]
        if draws and isinstance(draws[0], torch.Tensor):
            return torch.cat(draws)
        return [v for d in draws for v in d]

    def _run_custom_train(self, graph, subgraph_to_id, id_to_subgraph, train_vertices, graph_util):
        self.graphsage_model.train()
        n = len(train_vertices)
        if n == 0:
            return
        self._fused_steps(graph, self._host_seeds(train_vertices), n // self.batch_per_timestep)

    def get_model(self):
        return "random"


class PrioritizedPytorchSupervisedGraphSage(PytorchSupervisedGraphSage):
    """PBR: loss-prioritised rehearsal (reference :141-257)."""

    def __init__(self, model, batch_per_timestep, batch_size, labels, samples, priority_strategy, full_pass=2, cuda=False,
                 batch_full=512, n_workers=0, fanouts=None, eval_neighbourhood="sampled", priority_neighbourhood="sampled"):
        if priority_neighbourhood not in ("sampled", "full"):
            raise ValueError("priority_neighbourhood must be 'sampled' or 'full', got %r" % (priority_neighbourhood,))
        # neighbourhoods recompute_priorities scores the train vertices from, independent of eval_neighbourhood: "sampled" (the
        # reference's fan-outs) or "full" (every in-edge, GraphSAGE.inference_loss)
        self.priority_neighbourhood = priority_neighbourhood
        super().__init__(model, batch_per_timestep, batch_size, labels, samples, reduction="none", n_workers=n_workers,
                         cuda=cuda, batch_full=batch_full, fanouts=fanouts, eval_neighbourhood=eval_neighbourhood)
        self.time_step = 0
        self._per_buf = None
        self.pass_var = 0
        self.full_pass = full_pass
        self.priority_strategy = priority_strategy

    def choose_vertices(self, graph_util):
        if self.time_step % self.full_pass == 0:
            self.pass_var += 1
            self.recompute_priorities(graph_util, graph_util.get_train_set())
        elif len(graph_util.get_new_train_nodes()) > 1:
            self.recompute_priorities(graph_util, graph_util.get_new_train_nodes())
        draws = [graph_util.draw_priority_train_nodes(self.batch_size) for _ in range(self.batch_per_timestep)]
        return [v for d in draws for v in d]

    def _device_priorities(self):
        """the on-GPU priority update feeds the raw per-vertex losses to the sum tree, which is what LossPriority computes
        (generate_priority.py:7-9); Trend / Hybrid priorities keep per-vertex history on the host, so they always take the
        reference's route through priority_strategy.get_priorities (pytorch/model.py:203-206, 250-253)"""
        from ...prioritized_replay.generate_priority import LossPriority
        return (not config.faithful()) and type(self.priority_strategy) is LossPriority

    def _push_priorities(self, graph_util, nodes, losses_dev):
        if not self._device_priorities():
            pri = self.priority_strategy.get_priorities(nodes, losses_dev.cpu().numpy())
            graph_util.update_priorities(dict(zip(nodes, pri)))
        else:
            graph_util.update_priorities_device(list(nodes), losses_dev)

    def _run_custom_train(self, graph, subgraph_to_id, id_to_subgraph, train_vertices, graph_util):
        self.graphsage_model.train()
        n = len(train_vertices)
        if n:
            # every minibatch of the timestep runs back to back on the GPU; the per-vertex losses are pushed into the
            # priority structure afterwards, in batch order (a vertex trained twice keeps the loss of its last batch,
            # exactly what the reference's per-batch dict updates leave behind, pytorch/model.py:203-206)
            seeds = self._host_seeds(train_vertices)
            if self._per_buf is None or self._per_buf.numel() < n:
                self._per_buf = torch.empty(max(n, self.batch_size), dtype=torch.float32, device="cuda")
            per = self._per_buf[:n]
            batch = max(n // self.batch_per_timestep, 1)
            self._fused_steps(graph, seeds, batch, per_vertex_out=per)
            nodes = np.asarray(subgraph_to_id[np.asarray(train_vertices, dtype=np.int64)]).tolist()
            if not self._device_priorities():
                # one read-back, then the reference's sequence of per-batch dict updates (the running min / max of the
                # priority transform advances batch by batch, replay_buffer.py:110-130)
                host = per.cpu().numpy()
                for i in range(0, n, batch):
                    pri = self.priority_strategy.get_priorities(nodes[i:i + batch], host[i:i + batch])
                    graph_util.update_priorities(dict(zip(nodes[i:i + batch], pri)))
            else:
                last = {v: i for i, v in enumerate(nodes)}               # a vertex trained twice keeps its last loss
                idx = torch.as_tensor(list(last.values()), dtype=torch.int64, device="cuda")
                graph_util.update_priorities_device(list(last.keys()), per[idx])
        self.time_step += 1

    def recompute_priorities(self, graph_util, train_set):
        """eval-mode forward over `train_set`; per-vertex CE loss -> priorities (reference :210-254).  priority_neighbourhood="sampled":
        batch_full chunks of sampled neighbourhoods (each chunk advances the evaluation plan's Philox step).  "full": one
        GraphSAGE.inference_loss over the whole in-neighbourhoods, shared between the ranks under torchrun; it advances no Philox
        step.  The losses of training steps (_run_custom_train) are training losses and stay sampled either way."""
        self.graphsage_model.eval()
        id_to_subgraph = graph_util.get_original_to_subgraph_map()
        graph = graph_util.get_graph()
        sub = np.asarray(id_to_subgraph[train_set], dtype=np.int64)
        n = len(sub)
        if n == 0:
            return
        if self.priority_neighbourhood == "full":
            m = self.graphsage_model
            losses = m.inference_loss(graph, torch.as_tensor(sub).cuda(), distributed=parallel.world() > 1)
            flags = m.inference_plan(graph).error_flags()
            if flags & 1:
                raise IndexError("a vertex id outside the graph was evaluated (DGL's NodeDataLoader raises on such ids)")
            if flags & 2:
                raise ValueError("a train vertex has a label outside [0, %d) (torch's cross_entropy raises on such labels)" % m.dims[-1])
            self._push_priorities(graph_util, list(train_set), losses)
            return
        seeds = self._host_seeds(sub)
        plan = self._eval_plan(graph)
        losses = torch.empty(n, dtype=torch.float32, device="cuda")
        for i in range(0, n, self.batch_full):
            chunk = seeds[i:i + self.batch_full]
            plan.eval_step(graph.native, graph.features, chunk, per_vertex_out=losses[i:i + chunk.numel()])
        self._mark_pin_busy(seeds)
        self._push_priorities(graph_util, list(train_set), losses)

    def get_model(self):
        return "prioritized"


class FullPytorchSupervisedGraphSage(PytorchSupervisedGraphSage):
    """offline baseline: `batch_per_timestep` epochs over the whole train set (reference :260-290)."""

    def __init__(self, model, batch_per_timestep, batch_size, labels, samples, cuda=False, batch_full=512, n_workers=0, fanouts=None,
                 eval_neighbourhood="sampled"):
        super().__init__(model, batch_per_timestep, batch_size, labels, samples, n_workers=n_workers, cuda=cuda,
                         batch_full=batch_full, fanouts=fanouts, eval_neighbourhood=eval_neighbourhood)

    def choose_vertices(self, graph_util):
        return list(graph_util.get_train_set())

    def _run_custom_train(self, graph, subgraph_to_id, id_to_subgraph, batch_nodes, graph_util):
        self.graphsage_model.train()
        train_set = torch.as_tensor(np.asarray(batch_nodes, dtype=np.int64))
        for _ in range(self.batch_per_timestep):
            train_set = train_set[torch.randperm(train_set.numel())]
            self._fused_steps(graph, self._host_seeds(train_set), self.batch_size)

    def get_model(self):
        return "offline"


class NoRehPytorchSupervisedGraphSage(PytorchSupervisedGraphSage):
    """no rehearsal: train on the newest vertices only (reference :293-323)."""

    def __init__(self, model, batch_per_timestep, batch_size, labels, samples, cuda=False, batch_full=512, n_workers=0, fanouts=None,
                 eval_neighbourhood="sampled"):
        super().__init__(model, batch_per_timestep, batch_size, labels, samples, n_workers=n_workers, cuda=cuda,
                         batch_full=batch_full, fanouts=fanouts, eval_neighbourhood=eval_neighbourhood)

    def choose_vertices(self, graph_util):
        return []

    def _run_custom_train(self, graph, subgraph_to_id, id_to_subgraph, batch_nodes, graph_util):
        self.graphsage_model.train()
        for _ in range(self.batch_per_timestep):
            idxs = graph_util.get_new_train_nodes(self.batch_size)
            if len(idxs) < 2:
                return
            sub = torch.as_tensor(np.asarray(id_to_subgraph[idxs], dtype=np.int64))
            sub = sub[torch.randperm(sub.numel())]          # NodeDataLoader(shuffle=True) of the reference
            self._fused_step(graph, self._host_seeds(sub))

    def get_model(self):
        return "no_rehersal"
