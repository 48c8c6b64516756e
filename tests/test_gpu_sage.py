"""GraphSAGE-pool forward / backward / loss / Adam on the GPU vs the oracle (oracle/sage.py).

Tolerances (north_star): fp32 mode rtol 1e-5, bf16 mode rtol 1e-3 -- both taken relative to the
tensor's scale (|a-b| <= rtol*|b| + rtol*max|b|), because single elements of a length-600 dot
product can cancel to ~0.  Tensors the product STORES in bf16 (hp, neigh, hidden activations) are
compared at one bf16 ulp (2^-8) since a last-bit difference in the fp32 accumulation order may flip
the rounding of a stored value.  The argmax slots of the max-pool are compared exactly in fp32 mode.
"""
import numpy as np
import pytest
import torch

from oracle.graph import in_csr
from oracle import sage as osage

pytestmark = pytest.mark.gpu

NAMES = ("fc_pool.weight", "fc_pool.bias", "fc_self.weight", "fc_self.bias", "fc_neigh.weight", "fc_neigh.bias")


def close(a, b, rtol, what=""):
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    assert a.shape == b.shape, (what, a.shape, b.shape)
    scale = b.abs().max().item() if b.numel() else 0.0
    err = (a - b).abs()
    bound = rtol * b.abs() + rtol * scale + 1e-30
    bad = err > bound
    assert not bad.any(), "%s: %d / %d elements off, max err %.3e at scale %.3e (rtol %g)" % (
        what, int(bad.sum()), a.numel(), err.max().item(), scale, rtol)


def close_bf16_grad(a, b, what=""):
    """gradients of the bf16 pipeline vs the bf16-operand oracle: relative Frobenius error <= 1e-2 (about two bf16 ulps), >= 99.5 % of the
    elements within 3e-3 (of |b| + scale) and none further than 5e-2 * scale.  (A hidden activation that rounds to
    +0 on one side and to a tiny positive value on the other flips its ReLU mask: a whole term, not an ulp, for a
    handful of elements.)"""
    a = torch.as_tensor(a).double().cpu()
    b = torch.as_tensor(b).double().cpu()
    assert a.shape == b.shape, (what, a.shape, b.shape)
    scale = b.abs().max().item()
    err = (a - b).abs()
    fro = (err.pow(2).sum().sqrt() / b.pow(2).sum().sqrt().clamp(min=1e-30)).item()
    frac_bad = (err > 3e-3 * b.abs() + 3e-3 * scale).double().mean().item()
    assert fro <= 1e-2 and frac_bad <= 5e-3 and err.max().item() <= 5e-2 * scale, \
        "%s: rel. Frobenius err %.2e, %.3f %% of elements off, max err %.2e at scale %.2e" % (what, fro, 100 * frac_bad, err.max().item(), scale)


def flat_from_dict(params, n_layers):
    return torch.cat([params[f"layers.{i}.{n}"].reshape(-1).float() for i in range(n_layers) for n in NAMES])


def dict_from_flat(flat, dims):
    out, off = {}, 0
    for i in range(len(dims) - 1):
        fi, fo = dims[i], dims[i + 1]
        for n, shape in zip(NAMES, ((fi, fi), (fi,), (fo, fi), (fo,), (fo, fi), (fo,))):
            k = int(np.prod(shape))
            out[f"layers.{i}.{n}"] = flat[off:off + k].view(shape)
            off += k
    assert off == flat.numel()
    return out


def pin_device_argmax(plan, blocks, inter, ulp):
    """route the oracle's max-pool gradient through the slots the device picked (sets blocks[l]["arg"]), after checking that every
    device slot attains the free-running oracle's max (`inter`) within one ulp of the mode: in a rounded arithmetic two neighbours
    often tie, and which of them wins is decided by the last bit of the fp32 accumulation order"""
    L = len(blocks)
    for l in range(L):
        n_dst, fanout = blocks[l]["n_dst"], blocks[l]["fanout"]
        dim = inter[l]["hp"].shape[1]
        arg = plan.tensor(f"arg{l}", rows=n_dst)[:, :dim].long().cpu()
        arg[arg == 255] = -1
        assert torch.equal(arg < 0, inter[l]["arg"] < 0)
        es = blocks[l]["edge_src"].view(n_dst, fanout)
        src_row = torch.gather(es, 1, arg.clamp(min=0))                      # [n_dst, F] local src row of the device's slot
        assert bool((src_row[arg >= 0] >= 0).all()), "device argmax points at an empty slot"
        hp_o = inter[l]["hp"].detach()
        picked = hp_o[src_row.clamp(min=0), torch.arange(dim)[None, :].expand_as(src_row)]
        mx = inter[l]["neigh"].detach()
        # one ulp of the value + the fp32 accumulation-order noise of a cancelling dot product (relative to the scale)
        # (same tolerance as the comparison of the stored hp itself: layer >= 1 inherits rounding flips of its input)
        ok = (picked >= mx - 2 * ulp * mx.abs() - ulp * hp_o.abs().max()) | (arg < 0)
        assert bool(ok.all()), "device argmax slot is not a maximum within one ulp of the mode: %d bad" % int((~ok).sum())
        blocks[l]["arg"] = arg
    return blocks


class Case:
    def __init__(self, V=1500, E=9000, dims=(50, 24, 5), fanouts=(6, 4), n_seeds=96, mode="fp32", seed=3, gemm_impl=1,
                 isolated=40):
        import ogl_b200
        self.ogl = ogl_b200
        rng = np.random.default_rng(seed)
        src = rng.integers(0, V - isolated, E).astype(np.int64)
        dst = rng.integers(0, V - isolated, E).astype(np.int64)
        self.V, self.dims, self.fanouts, self.L = V, list(dims), list(fanouts), len(fanouts)
        self.mode = {"bf16": ogl_b200.OGL_BF16, "tf32": ogl_b200.OGL_TF32, "fp16": ogl_b200.OGL_FP16}.get(mode, ogl_b200.OGL_F32)
        self.quant = mode if mode in ("bf16", "tf32", "fp16") else None
        self.g = ogl_b200.native.Graph(V, 2 * E)
        self.g.insert_vertices(V)
        self.g.insert_edges(torch.as_tensor(src).cuda(), torch.as_tensor(dst).cuda(), symmetric=True)
        self.feats = torch.from_numpy(rng.standard_normal((V, dims[0])).astype(np.float32))
        self.labels = torch.from_numpy(rng.integers(0, dims[-1], V).astype(np.int64))
        self.f = ogl_b200.native.Features(V, dims[0], self.mode)
        self.f.write(0, self.feats.cuda(), self.labels.cuda())
        self.params = osage.xavier_params(dims[0], dims[1], dims[-1], self.L - 1, seed=seed)
        self.flat = flat_from_dict(self.params, self.L).cuda()
        self.grad = torch.zeros_like(self.flat)
        self.plan = ogl_b200.native.Plan(self.dims, self.fanouts, max(n_seeds, 8), V, mode=self.mode, seed=11, gemm_impl=gemm_impl)
        assert self.plan.n_params == self.flat.numel()
        self.plan.bind_params(self.flat, self.grad)
        # seeds include isolated vertices (zero in-degree rows -> neigh = 0)
        self.seeds = np.concatenate([rng.permutation(V - isolated)[:n_seeds - 3], np.arange(V - 3, V)]).astype(np.int64)

    def oracle_blocks(self):
        L = self.L
        blocks = []
        for hop in reversed(range(L)):                     # input layer first
            lid, _, _, f = self.plan.block_edges(hop)
            blocks.append(dict(n_dst=self.plan.level_nodes(hop).numel(), edge_src=lid.long().cpu(), fanout=f))
        x_in = self.feats[self.plan.level_nodes(L).long().cpu()]
        return x_in, blocks

    def run_oracle(self, dtype=torch.float64):
        x_in, blocks = self.oracle_blocks()
        labels = self.labels[torch.as_tensor(self.seeds)]
        return osage.loss_and_grads(self.params, x_in, blocks, labels, quant=self.quant, dtype=dtype)


@pytest.mark.parametrize("mode,rtol,rtol_store", [("fp32", 1e-5, 1e-5), ("bf16", 1e-3, 2 ** -8), ("tf32", 2e-4, 2 ** -10), ("fp16", 2e-4, 2 ** -10)])
@pytest.mark.parametrize("dims,fanouts", [((50, 24, 5), (6, 4)), ((166, 64, 2), (9, 9)), ((33, 7), (5,)), ((20, 16, 16, 3), (3, 3, 2))])
def test_forward_backward_parity_simt(mode, rtol, rtol_store, dims, fanouts):
    c = Case(dims=dims, fanouts=fanouts, mode=mode, gemm_impl=1)
    c.plan.sample(c.g, torch.as_tensor(c.seeds).cuda())
    logits = c.plan.forward(c.f)
    per, tot = c.plan.loss_backward(c.f, 1.0 / len(c.seeds))
    loss, per_ref, logits_ref, grads_ref, inter = c.run_oracle()
    close(logits, logits_ref, rtol, "logits")
    close(per, per_ref, max(rtol, 1e-5), "per-vertex loss")
    close(tot, per_ref.sum().reshape(1), max(rtol, 1e-5), "loss sum")
    L = c.L
    for l in range(L):
        h = L - 1 - l
        n_src, n_dst = c.plan.level_nodes(h + 1).numel(), c.plan.level_nodes(h).numel()
        hp = c.plan.tensor(f"hp{l}", rows=n_src)[:, :dims[l]].float()
        close(hp, inter[l]["hp"], rtol_store, f"hp{l}")
        ng = c.plan.tensor(f"neigh{l}", rows=n_dst)[:, :dims[l]].float()
        close(ng, inter[l]["neigh"], rtol_store, f"neigh{l}")
        if mode == "fp32":
            arg = c.plan.tensor(f"arg{l}", rows=n_dst)[:, :dims[l]].long().cpu()
            ref = inter[l]["arg"].clone()
            ref[ref < 0] = 255
            # argmax slot may legitimately differ only where two slots tie within fp32 rounding; demand >= 99.9 % equal
            assert (arg == ref).double().mean().item() > 0.999
    got = dict_from_flat(c.grad, dims)
    for k, v in grads_ref.items():
        if k in got:                                       # (the 1-layer case leaves the oracle's unused head without grads)
            close(got[k], v, rtol * (3 if mode != "fp32" else 1), "grad " + k)


@pytest.mark.parametrize("mode", ["bf16", "tf32", "fp16"])
@pytest.mark.parametrize("dims,fanouts,n_seeds", [((50, 24, 5), (6, 4), 96), ((166, 256, 2), (9, 9), 64), ((602, 600, 41), (10, 5), 300),
                                                  ((33, 7), (5,), 40), ((128, 32, 32, 40), (4, 3, 2), 50)])
def test_forward_backward_parity_tcgen05(dims, fanouts, n_seeds, mode):
    """the tensor-core paths: every GEMM on the tcgen05 kernels (gemm_impl=0), vs the oracle that rounds its operands where the
    product does (bf16 / tf32) AND vs the SIMT implementation of the same arithmetic.  (What these arithmetics cost against the
    UNQUANTISED oracle is measured at the benchmarked shape in tests/test_gpu_parity_reddit.py.)"""
    ulp = 2 ** -8 if mode == "bf16" else 2 ** -11
    c = Case(V=3000, E=20000, dims=dims, fanouts=fanouts, n_seeds=n_seeds, mode=mode, gemm_impl=0)
    seeds_dev = torch.as_tensor(c.seeds).cuda()
    c.plan.sample(c.g, seeds_dev)
    logits = c.plan.forward(c.f)
    per, tot = c.plan.loss_backward(c.f, 1.0 / len(c.seeds))
    L = c.L
    # pass 1: free-running oracle -> forward tensors; the device's argmax slots must attain the oracle's max
    _, per_ref, logits_ref, _, inter = c.run_oracle()
    close(logits, logits_ref, 1e-3, "logits")
    close(per, per_ref, 1e-3, "per-vertex loss")
    x_in, blocks = c.oracle_blocks()
    for l in range(L):
        h = L - 1 - l
        n_src, n_dst = c.plan.level_nodes(h + 1).numel(), c.plan.level_nodes(h).numel()
        close(c.plan.tensor(f"hp{l}", rows=n_src)[:, :dims[l]].float(), inter[l]["hp"], ulp, f"hp{l}")
        close(c.plan.tensor(f"neigh{l}", rows=n_dst)[:, :dims[l]].float(), inter[l]["neigh"], ulp, f"neigh{l}")
    pin_device_argmax(c.plan, blocks, inter, ulp)
    # pass 2: gradients with the device's routing through the max-pool
    labels = c.labels[torch.as_tensor(c.seeds)]
    _, _, _, grads_ref, _ = osage.loss_and_grads(c.params, x_in, blocks, labels, quant=mode, dtype=torch.float64)
    got = dict_from_flat(c.grad, dims)
    for k, v in grads_ref.items():
        if k in got:
            close_bf16_grad(got[k], v, "grad " + k)
    # same arithmetic on the SIMT kernels: same minibatch (same Philox step), tighter agreement
    g_tc = c.grad.clone()
    simt = c.ogl.native.Plan(c.dims, c.fanouts, max(n_seeds, 8), c.V, mode=c.mode, seed=11, gemm_impl=1)
    g2 = torch.zeros_like(c.flat)
    simt.bind_params(c.flat, g2)
    simt.sample(c.g, seeds_dev)
    logits2 = simt.forward(c.f)
    simt.loss_backward(c.f, 1.0 / len(c.seeds))
    close(logits, logits2, 1e-3, "tc vs simt logits")
    close_bf16_grad(g_tc, g2, "tc vs simt grads")


def test_zero_degree_rows_and_tail_padding():
    """all seeds isolated: neigh = 0 everywhere, out = fc_self(h) + biases; nothing leaks from stale workspace rows"""
    c = Case(dims=(12, 8, 3), fanouts=(4, 4), n_seeds=8, mode="fp32", isolated=40)
    big = np.arange(0, 8, dtype=np.int64)
    c.plan.sample(c.g, torch.as_tensor(big).cuda())
    c.plan.forward(c.f)                                   # dirties the workspaces with a connected batch
    iso = np.arange(c.V - 8, c.V, dtype=np.int64)
    c.seeds = iso
    c.plan.sample(c.g, torch.as_tensor(iso).cuda())
    assert c.plan.level_nodes(2).cpu().tolist() == iso.tolist()
    logits = c.plan.forward(c.f)
    _, _, logits_ref, _, inter = c.run_oracle()
    assert float(inter[0]["neigh"].abs().max()) == 0.0
    close(logits, logits_ref, 1e-5, "isolated logits")


def test_adam_and_fused_train_steps_track_the_oracle():
    c = Case(dims=(40, 16, 4), fanouts=(5, 5), n_seeds=64, mode="fp32")
    params = {k: v.clone().double() for k, v in c.params.items()}
    state = {}
    seeds_dev = torch.as_tensor(c.seeds).cuda()
    per = torch.empty(len(c.seeds), device="cuda")
    tot = torch.empty(1, device="cuda")
    for step in range(4):
        c.plan.train_step(c.g, c.f, seeds_dev, loss_scale=1.0 / len(c.seeds), do_step=True, per_vertex_out=per, loss_sum_out=tot)
        # oracle: same minibatch (the plan's Philox step advanced by one per train_step)
        x_in, blocks = c.oracle_blocks()
        labels = c.labels[torch.as_tensor(c.seeds)]
        loss, per_ref, _, grads, _ = osage.loss_and_grads(params, x_in, blocks, labels, dtype=torch.float64)
        close(per, per_ref, 1e-4, f"step {step} loss")
        osage.adam_step(params, grads, state)
        close(c.flat, flat_from_dict({k: v.float() for k, v in params.items()}, c.L), 2e-4, f"step {step} params")
    assert float(tot.item()) < float(per_ref.sum()) * 1.5
    # consecutive steps draw different neighbourhoods (step counter advances)
    c.plan.sample(c.g, seeds_dev)
    a = c.plan.block_edges(0)[1].clone()
    c.plan.train_step(c.g, c.f, seeds_dev, do_step=False)
    c.plan.sample(c.g, seeds_dev)
    assert not torch.equal(a, c.plan.block_edges(0)[1])


def test_host_seed_path_and_eval_step():
    c = Case(dims=(30, 16, 4), fanouts=(5, 5), n_seeds=50, mode="fp32")
    pinned = torch.as_tensor(c.seeds).pin_memory()
    logits = torch.empty(len(c.seeds), 4, device="cuda")
    per = torch.empty(len(c.seeds), device="cuda")
    c.plan.eval_step(c.g, c.f, pinned, logits_out=logits, per_vertex_out=per)
    _, per_ref, logits_ref, _, _ = c.run_oracle()
    close(logits, logits_ref, 1e-5, "eval logits")
    close(per, per_ref, 1e-5, "eval loss")


def test_autograd_bridge_matches_fused_path():
    """GraphSAGE.forward(blocks, x) + loss.backward() (the reference's train_step shape, pytorch/model.py:96-107)"""
    import ogl_b200
    from ogl_b200.sampling import MultiLayerNeighborSampler, NodeDataLoader
    ogl_b200.config.set_precision("fp32")
    V, F, H, C = 600, 20, 12, 3
    rng = np.random.default_rng(5)
    src, dst = rng.integers(0, V, 5000), rng.integers(0, V, 5000)
    dg = ogl_b200.DeviceGraph(V, 10000, F)
    feats = rng.standard_normal((V, F)).astype(np.float32)
    labels = rng.integers(0, C, (V, 1))
    dg.add_nodes(V, {"feat": feats, "target": labels})
    dg.add_edges(src, dst, symmetric=True)
    torch.manual_seed(0)
    model = ogl_b200.GraphSAGE(F, H, C, 1, torch.nn.functional.relu, 0, "pool").cuda()
    plan = model.plan_for(dg, [6, 6], 32)
    loader = NodeDataLoader(dg, np.arange(64), MultiLayerNeighborSampler([6, 6]), batch_size=32, plan=plan)
    loss_fn = torch.nn.CrossEntropyLoss()
    for input_nodes, seeds, blocks in loader:
        x = dg.ndata["feat"][input_nodes]
        y = dg.ndata["target"][seeds].flatten()
        logits = model(blocks, x)
        loss = loss_fn(logits, y)
        loss.backward()
        g_auto = [p.grad.clone() for p in model.parameters()]
        for p in model.parameters():
            p.grad = None
        # oracle on the same blocks
        params = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        ob = [dict(n_dst=b.number_of_dst_nodes(), edge_src=b._lid.long().cpu(), fanout=b.fanout) for b in blocks]
        _, _, lref, gref, _ = osage.loss_and_grads(params, x.cpu(), ob, y.cpu(), dtype=torch.float64)
        close(logits, lref, 1e-5, "autograd logits")
        for (k, _), ga in zip(model.named_parameters(), g_auto):
            close(ga, gref[k], 1e-5, "autograd grad " + k)
    ogl_b200.config.set_precision("tf32")


def test_cuda_graph_replay_equals_direct_launches():
    """the captured-graph train step and the direct launch sequence produce the same parameters; pool rebuilds of the
    streaming graph re-capture"""
    runs = []
    for use_graph in (1, 0):
        c = Case(dims=(64, 32, 5), fanouts=(6, 4), n_seeds=64, mode="bf16", gemm_impl=0)
        c.plan.set_option("cuda_graph", use_graph)
        seeds_dev = torch.as_tensor(c.seeds).cuda()
        per = torch.empty(len(c.seeds), device="cuda")
        tot = torch.empty(1, device="cuda")
        outs = []
        for step in range(5):
            if step == 3:      # grow the graph: forces a pool rebuild (new adjacency pointers)
                extra = torch.randint(0, c.V - 40, (30000,), generator=torch.Generator().manual_seed(5)).cuda()
                c.g.insert_edges(extra, extra.flip(0), symmetric=True)
            c.plan.train_step(c.g, c.f, seeds_dev, loss_scale=1.0 / len(c.seeds), do_step=True, per_vertex_out=per, loss_sum_out=tot)
            outs.append((per.clone(), tot.clone()))
        torch.cuda.synchronize()
        st = c.plan.graph_stats()
        if use_graph:
            assert st["replays"] == 5 and st["captures"] >= 1
        else:
            assert st["replays"] == 0
        runs.append((c.flat.clone(), outs))
    # the forward pass is deterministic; in the backward pass the reverse edge lists are filled in atomic order, so a
    # source row's few bf16 contributions may be summed in a different order (almost always exact in fp32 anyway)
    close(runs[0][0], runs[1][0], 1e-4, "params graph vs direct")
    for (p0, t0), (p1, t1) in zip(runs[0][1], runs[1][1]):
        close(p0, p1, 1e-4, "per-vertex loss graph vs direct")
        close(t0, t1, 1e-4, "loss sum graph vs direct")


def test_step_begin_finish_equals_fused_step():
    """the two-call form used by the data-parallel pipeline (sample + gather | forward .. Adam) is the same step"""
    runs = []
    for split in (0, 1, 2):
        c = Case(dims=(64, 32, 5), fanouts=(6, 4), n_seeds=64, mode="bf16", gemm_impl=0)
        seeds_dev = torch.as_tensor(c.seeds).cuda()
        pinned = torch.as_tensor(c.seeds).pin_memory()
        per = torch.empty(len(c.seeds), device="cuda")
        tot = torch.empty(1, device="cuda")
        outs = []
        for step in range(4):
            sd = pinned if step % 2 else seeds_dev          # host and device seed paths
            if split == 1:
                c.plan.step_begin(c.g, c.f, sd)
                c.plan.step_finish(c.f, 1.0 / len(c.seeds), do_step=True, per_vertex_out=per, loss_sum_out=tot)
            elif split == 2:                                 # bucketed form: head | tail (last weight-gradient GEMM) | Adam
                c.plan.step_begin(c.g, c.f, sd)
                c.plan.step_finish_head(c.f, 1.0 / len(c.seeds), per_vertex_out=per, loss_sum_out=tot)
                assert c.plan.tail_params == 64 * 64
                c.plan.step_finish_tail(c.f)
                c.plan.adam_step()
            else:
                c.plan.train_step(c.g, c.f, sd, loss_scale=1.0 / len(c.seeds), do_step=True, per_vertex_out=per, loss_sum_out=tot)
            outs.append(per.clone())
        torch.cuda.synchronize()
        runs.append((c.flat.clone(), outs))
    for other in (1, 2):
        close(runs[0][0], runs[other][0], 1e-4, "params fused vs split form %d" % other)
        for a, b in zip(runs[0][1], runs[other][1]):
            close(a, b, 1e-4, "per-vertex loss fused vs split form %d" % other)


def test_prefetch_pipeline_equals_fused_steps():
    """software pipeline (ogl_plan_prefetch: sample + gather of minibatch i+1 on the plan's own stream / second buffer set while
    minibatch i trains) == the same minibatches through the fused step: same sampled frontiers (bit-exact), same losses / weights"""
    runs = []
    n_steps, B = 7, 48
    for mode in ("fused", "prefetch", "pipeline-class"):
        c = Case(dims=(64, 32, 5), fanouts=(6, 4), n_seeds=B, mode="bf16", gemm_impl=0)
        rng = np.random.default_rng(3)
        allseeds = rng.permutation(c.V - 40)[:n_steps * B].astype(np.int64)
        batches = [torch.as_tensor(allseeds[i * B:(i + 1) * B]) for i in range(n_steps)]
        batches = [b.cuda() if i % 3 == 0 else (b.pin_memory() if i % 3 == 1 else b.clone()) for i, b in enumerate(batches)]
        per = torch.empty(B, device="cuda")
        tot = torch.empty(1, device="cuda")
        outs, fronts = [], []
        if mode == "fused":
            for sd in batches:
                c.plan.train_step(c.g, c.f, sd, loss_scale=1.0 / B, do_step=True, per_vertex_out=per, loss_sum_out=tot)
                outs.append((per.clone(), tot.clone()))
                fronts.append(c.plan.level_nodes(2).clone())
        elif mode == "prefetch":
            c.plan.prefetch(c.g, c.f, batches[0])
            for i, sd in enumerate(batches):
                if i + 1 < n_steps:
                    c.plan.prefetch(c.g, c.f, batches[i + 1])
                    assert c.plan.prefetch_pending == 2
                c.plan.train_step(c.g, c.f, sd, loss_scale=1.0 / B, do_step=True, per_vertex_out=per, loss_sum_out=tot)
                outs.append((per.clone(), tot.clone()))
            assert c.plan.prefetch_pending == 0
        else:
            import ogl_b200
            pipe = ogl_b200.parallel.Pipeline(c.plan, c.g, c.f, c.grad, B)
            pipe.begin(batches[0])
            for i in range(n_steps):
                pipe.finish(batches[i + 1] if i + 1 < n_steps else None, per_vertex_out=per, loss_sum_out=tot)
                outs.append((per.clone(), tot.clone()))
            pipe.flush()
        torch.cuda.synchronize()
        runs.append((c.flat.clone(), outs, fronts))
    for other in (1, 2):
        close(runs[0][0], runs[other][0], 1e-4, "params fused vs pipelined (%d)" % other)
        for (p0, t0), (p1, t1) in zip(runs[0][1], runs[other][1]):
            close(p0, p1, 1e-4, "per-vertex loss fused vs pipelined (%d)" % other)
            close(t0, t1, 1e-4, "loss sum fused vs pipelined (%d)" % other)


def test_prefetched_frontier_is_bit_exact_and_guarded():
    """a prefetched minibatch has the frontier the fused step samples at the same Philox step; sampling while one is pending is refused"""
    B = 40
    c0 = Case(dims=(64, 32, 5), fanouts=(6, 4), n_seeds=B, mode="bf16", gemm_impl=0)
    c1 = Case(dims=(64, 32, 5), fanouts=(6, 4), n_seeds=B, mode="bf16", gemm_impl=0)
    rng = np.random.default_rng(5)
    seeds = [torch.as_tensor(rng.permutation(c0.V - 40)[:B].astype(np.int64)).cuda() for _ in range(3)]
    want = []
    for sd in seeds:
        c0.plan.train_step(c0.g, c0.f, sd, loss_scale=1.0 / B, do_step=True)
        want.append([c0.plan.level_nodes(lv).clone() for lv in range(3)])
    c1.plan.prefetch(c1.g, c1.f, seeds[0])
    with pytest.raises(Exception):
        c1.plan.eval_step(c1.g, c1.f, seeds[0])
    for i, sd in enumerate(seeds):
        if i + 1 < len(seeds):
            c1.plan.prefetch(c1.g, c1.f, seeds[i + 1])
        c1.plan.step_finish(c1.f, 1.0 / B, do_step=True)
        torch.cuda.synchronize()
        # after the finish the current buffer set is the NEXT minibatch's (if one is pending): check it against the fused run
        if i + 1 < len(seeds):
            for lv in range(3):
                assert torch.equal(c1.plan.level_nodes(lv), want[i + 1][lv]), "prefetched frontier level %d of step %d" % (lv, i + 1)
    close(c0.flat, c1.flat, 1e-4, "params fused vs prefetched")


def test_multi_step_call_equals_single_steps():
    """ogl_plan_train_steps (all minibatches of a timestep in one C call) == the same steps one call at a time"""
    runs = []
    for multi in (False, True):
        c = Case(dims=(64, 32, 5), fanouts=(6, 4), n_seeds=32, mode="bf16", gemm_impl=0)
        rng = np.random.default_rng(0)
        seeds = torch.as_tensor(rng.permutation(c.V - 40)[:5 * 32].astype(np.int64)).pin_memory()
        per = torch.empty(5 * 32, device="cuda")
        sums = torch.empty(5, device="cuda")
        if multi:
            c.plan.train_steps(c.g, c.f, seeds, 32, per_vertex_out=per, loss_sums_out=sums)
        else:
            for i in range(5):
                c.plan.train_step(c.g, c.f, seeds[i * 32:(i + 1) * 32], loss_scale=1.0 / 32, do_step=True,
                                  per_vertex_out=per[i * 32:(i + 1) * 32], loss_sum_out=sums[i:i + 1])
        torch.cuda.synchronize()
        runs.append((c.flat.clone(), per.clone(), sums.clone()))
    close(runs[0][0], runs[1][0], 1e-4, "params")
    close(runs[0][1], runs[1][1], 1e-4, "per-vertex losses")
    close(runs[0][2], runs[1][2], 1e-4, "loss sums")
    close(runs[0][1].view(5, 32).sum(1), runs[0][2], 1e-5, "loss sum == sum of per-vertex losses")


@pytest.mark.parametrize("mode,gemm_impl,rtol", [("fp32", 1, 1e-5), ("tf32", 0, 2e-3), ("fp16", 0, 2e-3), ("bf16", 0, 2e-2)])
def test_feat_drop_matches_the_oracle_mask(mode, gemm_impl, rtol):
    """SAGEConv(feat_drop=p) (graphsage_dgl.py:41-46): every layer's input is dropped once in training mode with the Philox-keyed
    mask of oracle/sage.py:dropout_keep, scaled by 1 / (1 - p); evaluation is untouched"""
    p_drop = 0.3
    c = Case(dims=(48, 24, 5), fanouts=(6, 4), n_seeds=96, mode=mode, gemm_impl=gemm_impl)
    plan = c.ogl.native.Plan(c.dims, c.fanouts, 96, c.V, mode=c.mode, seed=11, gemm_impl=gemm_impl, feat_drop=p_drop)
    grad = torch.zeros_like(c.flat)
    plan.bind_params(c.flat, grad)
    c.plan = plan
    seeds_dev = torch.as_tensor(c.seeds).cuda()
    # evaluation mode: identical to a plan without dropout
    plan.sample(c.g, seeds_dev)
    logits_eval = plan.forward(c.f)
    _, _, logits_ref, _, _ = c.run_oracle()
    close(logits_eval, logits_ref, rtol, "eval-mode logits")
    # training mode (optimiser step 0)
    plan.set_option("train_mode", 1)
    plan.sample(c.g, seeds_dev)
    logits = plan.forward(c.f)
    per, _ = plan.loss_backward(c.f, 1.0 / len(c.seeds))
    x_in, blocks = c.oracle_blocks()
    for l, b in enumerate(blocks):
        n_src = c.plan.level_nodes(c.L - l).numel()
        keep = osage.dropout_keep(n_src, c.dims[l], p_drop, 11, 0, l)
        assert 0.6 < keep.double().mean().item() < 0.8
        b["drop"] = (keep, 1.0 / (1.0 - float(np.float32(p_drop))))
    labels = c.labels[torch.as_tensor(c.seeds)]
    _, per_ref, logits_ref2, grads_ref, _ = osage.loss_and_grads(c.params, x_in, blocks, labels, quant=c.quant, dtype=torch.float64)
    assert (logits_ref2 - logits_ref).abs().max().item() > 0.05           # dropout did something
    close(logits, logits_ref2, rtol, "train-mode logits")
    close(per, per_ref, rtol, "train-mode losses")
    got = dict_from_flat(grad, c.dims)
    for k, v in grads_ref.items():
        if mode == "fp32":
            close(got[k], v, rtol, "grad " + k)
        else:
            close_bf16_grad(got[k], v, "grad " + k)
    # the fused train step applies it too (same optimiser step -> same mask)
    plan.set_option("train_mode", 0)
    plan.set_step(0)
    per2 = torch.empty(len(c.seeds), device="cuda")
    plan.train_step(c.g, c.f, seeds_dev, loss_scale=1.0 / len(c.seeds), do_step=False, per_vertex_out=per2)
    close(per2, per, 1e-5 if mode == "fp32" else 1e-4, "fused step losses")


@pytest.mark.parametrize("mode", ["bf16", "tf32", "fp16"])
def test_train_step_is_bit_reproducible(mode):
    """reverse edge lists are put into canonical order after the atomic fill, so the max-pool backward sums every source row's
    contributions in the same order on every run: two runs from the same state give bit-identical gradients and weights -- on a
    graph with hub sources that are picked > 1024 times in one block (CTA-wide ordering), tens of times (warp) and a few times"""
    import ogl_b200
    V, E, B = 4000, 60000, 500
    rng = np.random.default_rng(2)
    src = np.where(rng.random(E) < 0.5, rng.integers(0, 4, E), rng.integers(0, V, E)).astype(np.int64)
    dst = rng.integers(0, V, E).astype(np.int64)
    runs = []
    for _ in range(2):
        g = ogl_b200.native.Graph(V, 2 * E)
        g.insert_vertices(V)
        g.insert_edges(torch.as_tensor(src).cuda(), torch.as_tensor(dst).cuda(), symmetric=False)
        m = {"bf16": ogl_b200.OGL_BF16, "tf32": ogl_b200.OGL_TF32, "fp16": ogl_b200.OGL_FP16}[mode]
        f = ogl_b200.native.Features(V, 40, m)
        gen = torch.Generator().manual_seed(0)
        f.write(0, torch.randn(V, 40, generator=gen).cuda(), torch.randint(0, 5, (V,), generator=gen).cuda())
        params = osage.xavier_params(40, 24, 5, 1, seed=1)
        flat = flat_from_dict(params, 2).cuda()
        grad = torch.zeros_like(flat)
        plan = ogl_b200.native.Plan([40, 24, 5], [10, 10], B, V, mode=m, seed=3)
        plan.bind_params(flat, grad)
        seeds = torch.arange(100, 100 + B, dtype=torch.int64).cuda()
        for _step in range(3):
            plan.train_step(g, f, seeds, loss_scale=1.0 / B, do_step=True)
        torch.cuda.synchronize()
        rp = plan.block_edges(1)
        runs.append((flat.clone(), grad.clone()))
    assert torch.equal(runs[0][1], runs[1][1]), "gradients differ between two identical runs"
    assert torch.equal(runs[0][0], runs[1][0]), "weights differ between two identical runs"
