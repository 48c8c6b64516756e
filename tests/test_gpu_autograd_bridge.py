"""The DGL-style loop of INTEGRATION.md section B, run as written in every arithmetic mode:

    plan = model.plan_for(graph, fanouts, batch); loader = NodeDataLoader(..., plan=plan); optimizer = torch.optim.Adam(...)
    for input_nodes, seeds, blocks in loader:
        logits = model(blocks, x); loss = loss_fn(logits, y); optimizer.zero_grad(); loss.backward(); optimizer.step()

Every iteration is checked against a fresh plan bound to a copy of the current parameters (bit for bit: the bridge's weight
shadows must follow torch's optimiser) and against the oracle in the mode's arithmetic; in fp32 the whole trajectory is replayed
on the CPU with torch.optim.Adam in float64.  Further tests cover mode OGL_FP16's gradient scale for losses of any magnitude,
the dropout mask of successive training-mode forwards, and the refusal of a backward over activations that are no longer there.
"""
import numpy as np
import pytest
import torch

from oracle import sage as osage
from test_gpu_sage import close, close_bf16_grad, pin_device_argmax

pytestmark = pytest.mark.gpu

MODES = ("fp32", "tf32", "fp16", "bf16")
ULP = {"fp32": 2.0 ** -20, "tf32": 2.0 ** -11, "fp16": 2.0 ** -11, "bf16": 2.0 ** -8}


def device_graph(V, E, F, C, seed, hub_frac=0.0, symmetric=True):
    """random graph (hub_frac of the edges leave one of four hub sources), standard-normal features, labels in [0, C)"""
    import ogl_b200
    rng = np.random.default_rng(seed)
    src = rng.integers(0, V, E)
    if hub_frac:
        src = np.where(rng.random(E) < hub_frac, rng.integers(0, 4, E), src)
    dst = rng.integers(0, V, E)
    dg = ogl_b200.DeviceGraph(V, 2 * E, F)
    dg.add_nodes(V, {"feat": rng.standard_normal((V, F)).astype(np.float32), "target": rng.integers(0, C, (V, 1))})
    dg.add_edges(src, dst, symmetric=symmetric)
    return dg


def oracle_blocks(blocks):
    return [dict(n_dst=b.number_of_dst_nodes(), edge_src=b._lid.long().cpu(), fanout=b.fanout) for b in blocks]


def flat_grad(model):
    return torch.cat([p.grad.reshape(-1) for p in model.parameters()])


class precision:
    """set_precision(mode) for the body of a with-statement, restored afterwards whatever happens"""

    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        import ogl_b200
        self.keep = ogl_b200.config.precision()
        ogl_b200.config.set_precision(self.mode)

    def __exit__(self, *exc):
        import ogl_b200
        ogl_b200.config.set_precision(self.keep)


def fresh_plan_like(model, plan, dg):
    """a new plan with the bridge plan's configuration, bound to a COPY of the model's current parameters"""
    import ogl_b200
    fresh = ogl_b200.native.Plan(model.dims, plan.fanouts, plan.max_seeds, dg.v_cap, mode=dg.mode, seed=ogl_b200.config.seed(),
                                 feat_drop=model.dropout)
    fresh.bind_params(model._flat.detach().clone(), torch.zeros_like(model._flat))
    return fresh


@pytest.mark.parametrize("n_hidden_layers", [1, 2])
@pytest.mark.parametrize("mode", MODES)
def test_dgl_loop_follows_the_optimiser(mode, n_hidden_layers):
    import ogl_b200
    from ogl_b200.sampling import MultiLayerNeighborSampler, NodeDataLoader
    V, F, H, C, B, iters = 800, 20, 16, 4, 32, 4
    L = n_hidden_layers + 1
    fan = [4] * L
    with precision(mode):
        dg = device_graph(V, 4000, F, C, seed=5)
        torch.manual_seed(0)
        model = ogl_b200.GraphSAGE(F, H, C, n_hidden_layers, torch.nn.functional.relu, 0, "pool").cuda()
        plan = model.plan_for(dg, fan, B)
        loader = NodeDataLoader(dg, np.arange(iters * B), MultiLayerNeighborSampler(fan), batch_size=B, plan=plan)
        optimizer = torch.optim.Adam(model.parameters())
        loss_fn = torch.nn.CrossEntropyLoss()
        names = [k for k, _ in model.named_parameters()]
        replay = None
        if mode == "fp32":                     # the same loop on the CPU: oracle forward, torch.optim.Adam, float64
            replay = {k: v.detach().cpu().double().clone().requires_grad_(True) for k, v in model.named_parameters()}
            replay_opt = torch.optim.Adam([replay[k] for k in names])
        for it, (input_nodes, seeds, blocks) in enumerate(loader):
            x = dg.ndata["feat"][input_nodes]
            y = dg.ndata["target"][seeds].flatten()
            params = {k: v.detach().cpu().clone() for k, v in model.named_parameters()}
            logits = model(blocks, x)
            seen = []
            logits.register_hook(lambda g: seen.append(g.detach().clone()))
            loss = loss_fn(logits, y)
            optimizer.zero_grad()
            loss.backward()
            grads = flat_grad(model).clone()
            dlogits = seen[0]
            # a fresh plan on the same minibatch (same Philox step: sampling through the loader does not advance it)
            fresh = fresh_plan_like(model, plan, dg)
            fresh.sample(dg.native, seeds)
            assert torch.equal(fresh.level_nodes(L), plan.level_nodes(L)), "iteration %d: the fresh plan drew another minibatch" % it
            fresh.set_input(x)
            assert torch.equal(fresh.forward(None), logits.detach()), "iteration %d: logits differ from a fresh plan's" % it
            fresh.backward(dlogits)
            assert torch.equal(fresh._grads, grads), "iteration %d: gradients differ from a fresh plan's" % it
            # the oracle at the current parameters, in the mode's arithmetic, routed through the device's argmax slots
            quant = None if mode == "fp32" else mode
            ob = oracle_blocks(blocks)
            _, _, lref, _, inter = osage.loss_and_grads(params, x.cpu(), ob, y.cpu(), quant=quant, dtype=torch.float64)
            close(logits.detach(), lref, 1e-5 if mode == "fp32" else 1e-3, "iteration %d logits" % it)
            pin_device_argmax(plan, ob, inter, ULP[mode])
            gs = osage.grad_scale_for(dlogits.abs().max().item())
            _, _, _, gref, _ = osage.loss_and_grads(params, x.cpu(), ob, y.cpu(), quant=quant, dtype=torch.float64, grad_scale=gs)
            for k, p in model.named_parameters():
                if mode == "fp32":
                    close(p.grad, gref[k], 1e-5, "iteration %d grad %s" % (it, k))
                else:
                    close_bf16_grad(p.grad, gref[k], "iteration %d grad %s" % (it, k))
            optimizer.step()
            if replay is not None:
                lr_, _ = osage.forward(replay, x.cpu().double(), oracle_blocks(blocks))
                rloss = torch.nn.functional.cross_entropy(lr_, y.cpu())
                close(loss.detach(), rloss.detach().reshape(()), 1e-4, "iteration %d loss vs CPU replay" % it)
                replay_opt.zero_grad()
                rloss.backward()
                replay_opt.step()
                for k, p in model.named_parameters():
                    close(p.detach(), replay[k].detach(), 2e-4, "iteration %d %s vs CPU replay" % (it, k))
        assert it == iters - 1


@pytest.mark.parametrize("B", [1, 16, 256])
@pytest.mark.parametrize("reduction,mult", [("mean", 1.0), ("sum", 1.0), ("mean", 1000.0)])
def test_fp16_bridge_scales_gradients_by_their_magnitude(reduction, mult, B):
    """mode OGL_FP16 stores activation gradients times a power of two; the bridge picks it from max |dlogits| (the fused step's rule),
    so a summed or scaled loss keeps the fused step's headroom.  Four hub sources take half of the edges: at B = 256 one is picked
    ~1,100 times in the outer block, and the max-pool backward sums those picks into one fp16 row"""
    import ogl_b200
    from ogl_b200.sampling import MultiLayerNeighborSampler, NodeDataLoader
    V, F, H, C, fan = 4000, 40, 24, 5, [10, 10]
    with precision("fp16"):
        dg = device_graph(V, 60000, F, C, seed=2, hub_frac=0.5, symmetric=False)
        torch.manual_seed(0)
        model = ogl_b200.GraphSAGE(F, H, C, 1, torch.nn.functional.relu, 0, "pool").cuda()
        plan = model.plan_for(dg, fan, B)
        loader = NodeDataLoader(dg, np.arange(100, 100 + B), MultiLayerNeighborSampler(fan), batch_size=B, plan=plan)
        input_nodes, seeds, blocks = next(iter(loader))
        x = dg.ndata["feat"][input_nodes]
        y = dg.ndata["target"][seeds].flatten()
        params = {k: v.detach().cpu().clone() for k, v in model.named_parameters()}
        logits = model(blocks, x)
        seen = []
        logits.register_hook(lambda g: seen.append(g.detach().clone()))
        loss = torch.nn.CrossEntropyLoss(reduction=reduction)(logits, y) * mult
        loss.backward()
        assert torch.isfinite(flat_grad(model)).all(), "non-finite weight gradients (%s x %g, batch %d)" % (reduction, mult, B)
        ob = oracle_blocks(blocks)
        _, _, _, _, inter = osage.loss_and_grads(params, x.cpu(), ob, y.cpu(), quant="fp16", dtype=torch.float64)
        pin_device_argmax(plan, ob, inter, ULP["fp16"])
        gs = osage.grad_scale_for(seen[0].abs().max().item())
        _, _, _, gref, _ = osage.loss_and_grads(params, x.cpu(), ob, y.cpu(), quant="fp16", dtype=torch.float64, reduction=reduction,
                                                loss_mult=mult, grad_scale=gs)
        for k, p in model.named_parameters():
            close_bf16_grad(p.grad, gref[k], "grad %s (%s x %g, batch %d)" % (k, reduction, mult, B))
        # control: the fused step on the same minibatch keeps its gradients finite at this hub size
        fused = fresh_plan_like(model, plan, dg)
        fused.train_step(dg.native, dg.features, seeds.contiguous(), loss_scale=1.0 / B, do_step=False)
        torch.cuda.synchronize()
        assert torch.equal(fused.level_nodes(2), plan.level_nodes(2)), "the fused step drew another minibatch"
        assert torch.isfinite(fused._grads).all(), "control: the fused step overflows fp16 at this hub size"


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_bridge_dropout_draws_a_new_mask_every_training_forward(mode):
    """SAGEConv(feat_drop=p) through the bridge: the k-th training-mode forward of a plan drops with the mask of
    oracle/sage.py:dropout_keep at step k (its own counter: torch's optimiser never runs the plan's Adam); evaluation drops nothing
    and does not advance the counter"""
    import ogl_b200
    from ogl_b200.sampling import MultiLayerNeighborSampler, NodeDataLoader
    V, F, H, C, B, p_drop, fan = 600, 24, 16, 4, 32, 0.3, [5, 5]
    with precision(mode):
        dg = device_graph(V, 3000, F, C, seed=7)
        torch.manual_seed(0)
        model = ogl_b200.GraphSAGE(F, H, C, 1, torch.nn.functional.relu, p_drop, "pool").cuda()
        plan = model.plan_for(dg, fan, B)
        # the same seeds three times at one Philox step: identical blocks, so only the mask can change
        loader = NodeDataLoader(dg, np.tile(np.arange(B), 3), MultiLayerNeighborSampler(fan), batch_size=B, plan=plan)
        optimizer = torch.optim.Adam(model.parameters())
        loss_fn = torch.nn.CrossEntropyLoss()
        quant = None if mode == "fp32" else mode
        rtol = 1e-5 if mode == "fp32" else 2e-2
        seed = ogl_b200.config.seed()
        masks = []
        for it, (input_nodes, seeds, blocks) in enumerate(loader):
            x = dg.ndata["feat"][input_nodes]
            y = dg.ndata["target"][seeds].flatten()
            params = {k: v.detach().cpu().double() for k, v in model.named_parameters()}
            ob = oracle_blocks(blocks)
            n_src = blocks[0].number_of_src_nodes()
            if it == 2:                          # evaluation in between: no mask, and the counter stays at 2
                model.eval()
                logits = model(blocks, x)
                assert bool((plan.tensor("x", rows=n_src)[:, :F] != 0).all()), "evaluation dropped input elements"
                close(logits.detach(), osage.forward(params, x.cpu().double(), ob, quant=quant)[0].detach(), rtol, "eval logits")
            model.train()
            logits = model(blocks, x)
            kept = (plan.tensor("x", rows=n_src)[:, :F] != 0).cpu()            # the input features are never 0 themselves
            want = osage.dropout_keep(n_src, F, p_drop, seed, it, 0)
            assert torch.equal(kept, want), "iteration %d: layer-0 mask is not dropout_keep(step=%d)" % (it, it)
            masks.append(kept)
            scale = 1.0 / (1.0 - float(np.float32(p_drop)))
            for l, b in enumerate(ob):
                n = n_src if l == 0 else blocks[l].number_of_src_nodes()
                b["drop"] = (osage.dropout_keep(n, model.dims[l], p_drop, seed, it, l), scale)
            lref = osage.forward(params, x.cpu().double(), ob, quant=quant)[0].detach()
            close(logits.detach(), lref, rtol, "iteration %d train-mode logits" % it)
            loss = loss_fn(logits, y)
            optimizer.zero_grad()
            loss.backward()
            optimizer.step()
        assert len(masks) == 3
        assert not torch.equal(masks[0], masks[1]) and not torch.equal(masks[1], masks[2]), "two training forwards shared one mask"


def test_bridge_backward_refuses_overwritten_activations():
    """the plan keeps one set of activations: a backward after another forward, or after the loader sampled again, would
    differentiate the wrong ones and must raise instead"""
    import ogl_b200
    from ogl_b200.sampling import MultiLayerNeighborSampler, NodeDataLoader
    V, F, H, C, B, fan = 600, 20, 12, 3, 32, [4, 4]
    with precision("fp32"):
        dg = device_graph(V, 3000, F, C, seed=9)
        torch.manual_seed(0)
        model = ogl_b200.GraphSAGE(F, H, C, 1, torch.nn.functional.relu, 0, "pool").cuda()
        plan = model.plan_for(dg, fan, B)
        loader = iter(NodeDataLoader(dg, np.arange(2 * B), MultiLayerNeighborSampler(fan), batch_size=B, plan=plan))
        loss_fn = torch.nn.CrossEntropyLoss()
        input_nodes, seeds, blocks = next(loader)
        x = dg.ndata["feat"][input_nodes]
        y = dg.ndata["target"][seeds].flatten()
        first = model(blocks, x)
        second = model(blocks, x)
        with pytest.raises(RuntimeError, match="another forward"):
            loss_fn(first, y).backward()
        loss_fn(second, y).backward()                 # the latest forward is still there
        assert torch.isfinite(flat_grad(model)).all()
        third = model(blocks, x)
        next(loader)                                  # samples the next minibatch into the plan
        with pytest.raises(RuntimeError, match="another forward"):
            loss_fn(third, y).backward()
