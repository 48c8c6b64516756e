"""Data-parallel training over the GPUs of one box (SURVEY 8(e)): one process per GPU (torchrun), replicated
streaming graph + feature store + weights, every rank trains its own shard of the global target-vertex batch, the
flat fp32 gradient buffer is summed with ONE NCCL all-reduce (loss_scale = 1 / global batch makes the sum the mean
gradient) before the replicated fused Adam step.  PBR keeps its sum trees identical on all ranks by all-gathering the
(vertex id, loss) pairs.  The reference has no multi-GPU path (single process, SURVEY 2.1)."""
import torch
import torch.distributed as dist


def world():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def rank():
    return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0


def shard(seeds, r=None, w=None):
    """rank r's contiguous slice of a global seed list (equal sizes up to the remainder, order preserved)"""
    r = rank() if r is None else r
    b = shard_bounds(len(seeds), w)
    return seeds[b[r]:b[r + 1]]


def shard_bounds(n, w=None):
    """the w + 1 boundaries of shard()'s slices of an n-element list"""
    w = world() if w is None else w
    base, rem = divmod(n, w)
    return [r * base + min(r, rem) for r in range(w + 1)]


def edge_balanced_bounds(degrees, w=None):
    """w + 1 row boundaries 0 = b_0 <= ... <= b_w = V that split the cost sum(deg + 1) of full inference's segment max (one source row
    read per in-edge, one output row per vertex) evenly: b_r is the first row whose cost prefix reaches r / w of the total, so a
    shard's cost is off the even share by less than one row's.  degrees: the [V] in-degrees (Graph.degrees()); the graph is
    replicated, so every rank computes the same bounds."""
    w = world() if w is None else w
    cost = degrees.to(torch.int64) + 1
    prefix = torch.cat([torch.zeros(1, dtype=torch.int64, device=cost.device), torch.cumsum(cost, 0)])
    total = int(prefix[-1])
    targets = torch.tensor([(r * total + w - 1) // w for r in range(w + 1)], dtype=torch.int64, device=cost.device)
    return torch.searchsorted(prefix, targets).tolist()


def allgather_rows(table, bounds, group=None):
    """rank r's rows table[bounds[r]:bounds[r + 1]] go to every rank, in place: one broadcast per non-empty slice from its owner (rows
    are contiguous, nothing is staged); no-op on one rank"""
    if world() == 1:
        return table
    for r in range(len(bounds) - 1):
        if bounds[r + 1] > bounds[r]:
            src = r if group is None else dist.get_global_rank(group, r)
            dist.broadcast(table[bounds[r]:bounds[r + 1]], src=src, group=group)
    return table


def infer_full(plan, graph, features, vertices=None, exchange=allgather_rows, r=None, w=None):
    """Plan.infer_full split over the ranks: fp32 logits [n, C] of `vertices` (int64 ids; None: every vertex), the full result on
    every rank and bit-identical to the one-rank call.  Every hidden layer runs on this rank's edge_balanced_bounds range of rows,
    then exchange(table, bounds) fills in the other ranks' rows of its [V, pitch] output table; the last layer runs on this rank's
    shard() of `vertices` (or its range of rows) and its logits are exchanged the same way.  Every rank must call it (the exchange
    is collective).  r, w: this rank and the number of ranks (default: the process group's; a test runs every rank of a world in
    one process with them and an exchange of its own)."""
    r = rank() if r is None else r
    w = world() if w is None else w
    h, v, bounds = _hidden_layers(plan, graph, features, vertices, exchange, r, w)
    lo, hi = bounds[r], bounds[r + 1]
    logits = torch.empty(graph.num_vertices if v is None else v.numel(), plan.dims[-1], dtype=torch.float32, device="cuda")
    _last_layer(plan, graph, features, h, v, lo, hi, logits[lo:hi])
    exchange(logits, bounds)
    return logits


def infer_full_loss(plan, graph, features, vertices=None, exchange=allgather_rows, r=None, w=None):
    """Plan.infer_full_loss split over the ranks: fp32 per-vertex cross-entropy losses [n] of `vertices` (None: every vertex), the full
    vector on every rank and bit-identical to the one-rank call.  The hidden layers run and are exchanged exactly as in infer_full;
    the last layer and the loss run on this rank's share of the vertices, and only the losses (4 bytes per vertex, not 4 C) are
    exchanged.  A collective, like infer_full; ids outside the graph raise bit 0 of plan.error_flags(), labels outside [0, C) bit 1."""
    r = rank() if r is None else r
    w = world() if w is None else w
    h, v, bounds = _hidden_layers(plan, graph, features, vertices, exchange, r, w)
    lo, hi = bounds[r], bounds[r + 1]
    losses = torch.empty(graph.num_vertices if v is None else v.numel(), dtype=torch.float32, device="cuda")
    if hi > lo:
        logits = _last_layer(plan, graph, features, h, v, lo, hi, None)
        if v is None:
            plan.full_xent(features, logits, row0=lo, out=losses[lo:hi])
        else:
            # the label of an id outside the graph is vertex 0's, as in the one-rank call (the last layer has raised bit 0)
            rows = v[lo:hi]
            rows = torch.where((rows < 0) | (rows >= graph.num_vertices), torch.zeros_like(rows), rows)
            plan.full_xent(features, logits, rows=rows, out=losses[lo:hi])
    exchange(losses, bounds)
    return losses


def _hidden_layers(plan, graph, features, vertices, exchange, r, w):
    """the hidden layers of infer_full / infer_full_loss, each on this rank's edge_balanced_bounds range of rows and exchanged into a
    [V, pitch] table -> (the last hidden table, or None for a one-layer model; the vertices as a device int64 tensor, or None; the
    bounds of the last layer's shards: the row ranges for every vertex, shard_bounds of the list otherwise)"""
    V = graph.num_vertices
    bounds = edge_balanced_bounds(graph.degrees(), w)
    lo, hi = bounds[r], bounds[r + 1]
    h = None
    tables = [None, None]
    for l in range(plan.L - 1):
        if tables[l & 1] is None:
            tables[l & 1] = plan.hidden_table(l, V)
        out = tables[l & 1]
        plan.infer_full_layer(graph, features, l, h, row0=lo, n=hi - lo, out=out[lo:hi])
        exchange(out, bounds)
        h = out
    if vertices is None:
        return h, None, bounds
    v = vertices.to(device="cuda", dtype=torch.int64) if isinstance(vertices, torch.Tensor) else \
        torch.as_tensor(vertices, dtype=torch.int64, device="cuda")
    return h, v, shard_bounds(v.numel(), w)


def _last_layer(plan, graph, features, h, v, lo, hi, out):
    """the last layer on rows [lo, hi) of the vertices (v None: of the graph) -> fp32 logits [hi - lo, C] (into out if given)"""
    if v is None:
        return plan.infer_full_layer(graph, features, plan.L - 1, h, row0=lo, n=hi - lo, out=out)
    return plan.infer_full_layer(graph, features, plan.L - 1, h, rows=v[lo:hi], out=out)


def allreduce_grads(flat_grad, group=None):
    """sum the flat gradient buffer over the ranks (in place); no-op on one rank"""
    if world() > 1:
        dist.all_reduce(flat_grad, op=dist.ReduceOp.SUM, group=group)
    return flat_grad


def allgather_losses(vertex_ids, losses, group=None):
    """every rank receives all (vertex id, per-vertex loss) pairs of the step, in rank order (PBR priority updates
    must be applied identically on every replica)"""
    if world() == 1:
        return vertex_ids, losses
    w = world()
    n = torch.tensor([vertex_ids.numel()], dtype=torch.int64, device=vertex_ids.device)
    sizes = [torch.zeros_like(n) for _ in range(w)]
    dist.all_gather(sizes, n, group=group)
    m = int(max(int(s.item()) for s in sizes))
    pad_v = torch.full((m,), -1, dtype=vertex_ids.dtype, device=vertex_ids.device)
    pad_l = torch.zeros(m, dtype=losses.dtype, device=losses.device)
    pad_v[:vertex_ids.numel()] = vertex_ids
    pad_l[:losses.numel()] = losses
    vs = [torch.empty_like(pad_v) for _ in range(w)]
    ls = [torch.empty_like(pad_l) for _ in range(w)]
    dist.all_gather(vs, pad_v, group=group)
    dist.all_gather(ls, pad_l, group=group)
    keep = [int(s.item()) for s in sizes]
    return torch.cat([v[:k] for v, k in zip(vs, keep)]), torch.cat([l[:k] for l, k in zip(ls, keep)])


def train_step(plan, graph, features, local_seeds, global_batch, flat_grad, per_vertex_out=None, loss_sum_out=None):
    """one data-parallel step: local sample/forward/backward -> gradient all-reduce -> replicated Adam"""
    w = world()
    plan.train_step(graph, features, local_seeds, loss_scale=1.0 / float(global_batch), do_step=(w == 1),
                    per_vertex_out=per_vertex_out, loss_sum_out=loss_sum_out)
    if w > 1:
        allreduce_grads(flat_grad)
        plan.adam_step()


def make_peer_exchange(plan, flat_params, group=None):
    """NVLink peer-memory gradient exchange for `plan` (csrc/peer.cu): allocates the rank's peer-visible gradient buffer, binds it
    as the plan's gradient buffer, exchanges the CUDA IPC handles over the process group and maps the peers.  Returns the
    native.Peer (its `.grads` is the new flat gradient tensor).  One rank: a plain local buffer, no peers."""
    from . import _native as native
    w, r = world(), rank()
    peer = native.Peer(r, w, plan.n_params)
    if w > 1:
        mine = torch.frombuffer(bytearray(peer.handle()), dtype=torch.uint8).cuda()
        every = [torch.empty_like(mine) for _ in range(w)]
        dist.all_gather(every, mine, group=group)
        peer.connect(b"".join(bytes(t.cpu().numpy().tobytes()) for t in every))
        dist.barrier(group=group)
    plan.bind_params(flat_params, peer.grads)
    return peer


class Pipeline:
    """Train loop with everything that does not need fresh weights off the critical path (any number of GPUs).

    A step is split at the only point where it needs fresh weights: `begin` = sample + gather (reads the graph and the
    feature store only), `finish` = forward .. backward (.. Adam).  `begin` of step t+1 is a prefetch (Plan.prefetch: the
    plan's own stream and second buffer set), so it overlaps forward / backward of step t -- the job NodeDataLoader's worker
    processes do in the reference (pytorch/model.py:128-131).  With more than one rank the gradient exchange is bucketed:
    the exchange of everything but layer 0's fc_pool.weight overlaps the last weight-gradient GEMM.  With a peer group both
    exchanges and Adam are nodes of the step's own launch sequence (Plan.step_finish_dp); with NCCL the all-reduces, the small
    second bucket and Adam run on a communication stream and forward(t+1) waits for Adam(t).  Same arithmetic as the
    unpipelined loop (no stale gradients, same Philox step per minibatch)."""

    def __init__(self, plan, graph, features, flat_grad, global_batch, peer=None, force_split=False):
        """peer: a native.Peer from make_peer_exchange -> the gradient exchange + Adam is ONE kernel per bucket over NVLink peer
        memory (no NCCL on the data path); None -> NCCL all-reduce + ogl_plan_adam_step"""
        self.plan, self.graph, self.features, self.flat_grad = plan, graph, features, flat_grad
        self.peer = peer
        if peer is not None:
            assert flat_grad.data_ptr() == peer.grads.data_ptr(), "the plan must be bound to the peer group's gradient buffer"
        self.scale = 1.0 / float(global_batch)
        # force_split (experiments; needs `peer`): run the one-graph data-parallel finish (Plan.step_finish_dp) on ONE rank with a
        # one-rank peer group -- what its launch structure costs, without NVLink traffic or waiting for other ranks
        self.w = max(world(), 2) if force_split else world()
        self.comm = torch.cuda.Stream() if self.w > 1 else None
        self.ev_bwd = torch.cuda.Event()
        self.ev_head = torch.cuda.Event()
        self.ev_adam = torch.cuda.Event()
        self._begun = 0
        self._adam_pending = False

    def begin(self, seeds):
        self.plan.prefetch(self.graph, self.features, seeds)
        self._begun += 1

    def finish(self, next_seeds=None, per_vertex_out=None, loss_sum_out=None, scale=None):
        """scale: loss scale of THIS step (1 / its global batch) when it differs from the pipeline's (a ragged last minibatch)"""
        assert self._begun > 0, "Pipeline.finish() without begin()"
        if next_seeds is not None and self._begun < 2:
            self.begin(next_seeds)                       # enqueued first: overlaps this step's forward / backward
        self._begun -= 1
        main = torch.cuda.current_stream()
        keep_scale = self.scale
        if scale is not None:
            self.scale = float(scale)
        try:
            self._finish(main, per_vertex_out, loss_sum_out)
        finally:
            self.scale = keep_scale

    def _finish(self, main, per_vertex_out, loss_sum_out):
        if self.w == 1:
            self.plan.step_finish(self.features, self.scale, do_step=True, per_vertex_out=per_vertex_out, loss_sum_out=loss_sum_out)
            return
        if self.peer is not None:
            # one launch sequence (one CUDA graph) per step, the exchanges inside it (ogl_plan_step_finish_dp)
            self.plan.step_finish_dp(self.peer, self.features, self.scale, per_vertex_out=per_vertex_out, loss_sum_out=loss_sum_out)
            return
        if self._adam_pending:
            main.wait_event(self.ev_adam)                # weights (and the gradient buffer) of the previous step are settled
        # two gradient buckets: everything except layer 0's fc_pool.weight is final before the last weight-gradient GEMM
        # runs, so its all-reduce overlaps that GEMM; the small second bucket + Adam overlap the next step's start
        n0 = self.plan.tail_params
        self.plan.step_finish_head(self.features, self.scale, per_vertex_out=per_vertex_out, loss_sum_out=loss_sum_out)
        self.ev_head.record(main)
        with torch.cuda.stream(self.comm):
            self.comm.wait_event(self.ev_head)
            allreduce_grads(self.flat_grad[n0:])
        self.plan.step_finish_tail(self.features)
        self.ev_bwd.record(main)
        with torch.cuda.stream(self.comm):
            self.comm.wait_event(self.ev_bwd)
            allreduce_grads(self.flat_grad[:n0])
            self.plan.adam_step()
            self.ev_adam.record(self.comm)
        self._adam_pending = True

    def flush(self):
        if self._adam_pending:
            torch.cuda.current_stream().wait_event(self.ev_adam)
            self._adam_pending = False
