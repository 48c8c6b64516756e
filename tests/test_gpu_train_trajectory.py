"""Several fused train steps against the fp64 oracle in every arithmetic mode, and the step forms against each other bit for bit.

A one-step test never reads a weight shadow that Adam wrote: the shadows of its only step come from k_weight_shadow at bind time.
Here every step t (P_t = the flat parameters before it, G_t = the gradient it leaves in the bound buffer) is checked three ways:
- Adam: P_{t+1} against Adam restated in fp64 from the device's own gradients G_0 .. G_t (both halves of the split update -- the
  side-stream part during the backward pass and the rest after it -- and the step counter's bias correction);
- shadows: a second plan bound to a copy of P_{t+1} builds its shadows with k_weight_shadow; on the same minibatch its logits and
  gradients must equal the trained plan's bit for bit, so every shadow element k_adam_shadow wrote is the one a rebuild gives;
- gradients: G_t against the oracle at P_t in the mode's arithmetic, routed through the device's argmax slots.
The learning rate is large enough that weights one step stale move the logits well beyond every tolerance used here.
"""
import math

import numpy as np
import pytest
import torch

from oracle import sage as osage
from test_gpu_sage import Case, close, close_bf16_grad, dict_from_flat, flat_from_dict, pin_device_argmax

pytestmark = pytest.mark.gpu

LR = 3e-3
STEPS = 5
# mode -> (gemm_impl, ulp of the stored operands for the argmax check)
MODES = {"fp32": (1, 2.0 ** -20), "tf32": (0, 2.0 ** -11), "fp16": (0, 2.0 ** -11), "bf16": (0, 2.0 ** -8)}
SHAPES = {
    # pitches that are not multiples of the vector width (50, 24, 5), isolated vertices among the seeds
    "2layer": dict(V=1500, E=9000, dims=(50, 24, 5), fanouts=(6, 4), n_seeds=96),
    "3layer": dict(V=3000, E=20000, dims=(128, 32, 32, 40), fanouts=(4, 3, 2), n_seeds=50),
    "hubs": None,
}


class HubCase(Case):
    """the graph of test_gpu_sage.py::test_train_step_is_bit_reproducible: half of the edges leave one of four hub sources, so a hub
    is picked more than 1,024 times in one block (the CTA-wide ordering of the reverse edge lists), others tens of times or a few"""

    def __init__(self, mode, gemm_impl):
        import ogl_b200
        self.ogl = ogl_b200
        V, E, B = 4000, 60000, 500
        rng = np.random.default_rng(2)
        src = np.where(rng.random(E) < 0.5, rng.integers(0, 4, E), rng.integers(0, V, E)).astype(np.int64)
        dst = rng.integers(0, V, E).astype(np.int64)
        self.V, self.dims, self.fanouts, self.L = V, [40, 24, 5], [10, 10], 2
        self.mode = {"bf16": ogl_b200.OGL_BF16, "tf32": ogl_b200.OGL_TF32, "fp16": ogl_b200.OGL_FP16}.get(mode, ogl_b200.OGL_F32)
        self.quant = mode if mode in ("bf16", "tf32", "fp16") else None
        self.g = ogl_b200.native.Graph(V, 2 * E)
        self.g.insert_vertices(V)
        self.g.insert_edges(torch.as_tensor(src).cuda(), torch.as_tensor(dst).cuda(), symmetric=False)
        gen = torch.Generator().manual_seed(0)
        self.feats = torch.randn(V, 40, generator=gen)
        self.labels = torch.randint(0, 5, (V,), generator=gen)
        self.f = ogl_b200.native.Features(V, 40, self.mode)
        self.f.write(0, self.feats.cuda(), self.labels.cuda())
        self.params = osage.xavier_params(40, 24, 5, 1, seed=1)
        self.flat = flat_from_dict(self.params, 2).cuda()
        self.grad = torch.zeros_like(self.flat)
        self.plan = ogl_b200.native.Plan(self.dims, self.fanouts, B, V, mode=self.mode, seed=11, gemm_impl=gemm_impl)
        self.plan.bind_params(self.flat, self.grad)
        self.seeds = np.arange(100, 100 + B, dtype=np.int64)


def make_case(shape, mode):
    gemm_impl = MODES[mode][0]
    c = HubCase(mode, gemm_impl) if SHAPES[shape] is None else Case(mode=mode, gemm_impl=gemm_impl, seed=3, **SHAPES[shape])
    c.gemm_impl = gemm_impl
    c.plan = plan_like(c, c.flat, c.grad)
    return c


def plan_like(c, flat, grad):
    """a plan with c's configuration, seed and learning rate, bound to (flat, grad): its weight shadows come from k_weight_shadow"""
    plan = c.ogl.native.Plan(c.dims, c.fanouts, max(len(c.seeds), 8), c.V, mode=c.mode, seed=11, gemm_impl=c.gemm_impl, lr=LR)
    plan.bind_params(flat, grad)
    return plan


class AdamF64:
    """torch.optim.Adam restated in fp64 on the flat buffer, with the plan's hyper-parameters as the device holds them (fp32)"""

    def __init__(self, p0):
        f32 = lambda x: float(np.float32(x))
        self.lr, self.b1, self.b2, self.eps = f32(LR), f32(0.9), f32(0.999), f32(1e-8)
        self.p = p0.double().cpu()
        self.m = torch.zeros_like(self.p)
        self.v = torch.zeros_like(self.p)
        self.t = 0

    def step(self, g):
        g = g.double().cpu()
        self.t += 1
        self.m = self.b1 * self.m + (1 - self.b1) * g
        self.v = self.b2 * self.v + (1 - self.b2) * g * g
        bc1, bc2 = 1 - self.b1 ** self.t, 1 - self.b2 ** self.t
        self.p = self.p - (self.lr / bc1) * self.m / (self.v.sqrt() / math.sqrt(bc2) + self.eps)
        return self.p


def adam_bound(p_ref, lr):
    """|device - fp64 Adam|: the fp32 result p - u is rounded once (1/2 ulp of p) and p itself is the device's own fp32 value of the
    previous step, restated exactly.  The update u = step * m / (sqrt(v) * rsqrt(bc2) + eps) carries the fp32 rounding of m and v
    (about three roundings each per step, relative error < 5 * 3 * 2^-24 over five steps), of powf in bc1 / bc2, of rsqrtf (2 ulps),
    sqrtf, the product and the quotient: < 40 * 2^-24 = 2.4e-6 of |u|.  Adam's |u| stays below 3 * lr in these runs (|m_hat| /
    sqrt(v_hat) <= (1 - b1) / sqrt(1 - b2) in the worst case), so 2 ulps of p + 1e-4 * lr bounds the error with margin; a wrong
    gradient, a stale half of the split update or a wrong step counter moves p by a sizeable fraction of lr."""
    ulp = torch.where(p_ref == 0, torch.full_like(p_ref, 2.0 ** -149), 2.0 ** (torch.floor(torch.log2(p_ref.abs())) - 23))
    return 2 * ulp + 1e-4 * lr


def check_gradients(c, mode, per, grad, params_t):
    """G_t against the oracle at P_t (the second pass of test_forward_backward_parity_tcgen05: the mode's arithmetic, the device's
    argmax routing)"""
    quant = c.quant
    x_in, blocks = c.oracle_blocks()
    labels = c.labels[torch.as_tensor(c.seeds)]
    _, per_free, _, _, inter = osage.loss_and_grads(params_t, x_in, blocks, labels, quant=quant, dtype=torch.float64)
    pin_device_argmax(c.plan, blocks, inter, MODES[mode][1])
    _, per_ref, _, grads_ref, _ = osage.loss_and_grads(params_t, x_in, blocks, labels, quant=quant, dtype=torch.float64)
    got = dict_from_flat(grad, c.dims)
    for k, v in grads_ref.items():
        if mode == "fp32":
            close(got[k], v, 1e-5, "grad " + k)
        else:
            close_bf16_grad(got[k], v, "grad " + k)
    close(per, per_free, 1e-5 if mode == "fp32" else 1e-3, "per-vertex loss")


def oracle_logits(c, flat):
    """the oracle's logits in c's arithmetic at the parameters `flat`, on the minibatch in c.plan's buffers"""
    x_in, blocks = c.oracle_blocks()
    params = {k: v.cpu().double() for k, v in dict_from_flat(flat, c.dims).items()}
    return osage.forward(params, x_in.double(), blocks, quant=c.quant)[0].detach()


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("mode", list(MODES))
def test_fused_step_trajectory_tracks_the_oracle(mode, shape):
    c = make_case(shape, mode)
    B = len(c.seeds)
    seeds_dev = torch.as_tensor(c.seeds).cuda()
    per = torch.empty(B, device="cuda")
    tot = torch.empty(1, device="cuda")
    adam = AdamF64(c.flat)
    for t in range(STEPS):
        p_t = c.flat.clone()
        c.plan.train_step(c.g, c.f, seeds_dev, loss_scale=1.0 / B, do_step=True, per_vertex_out=per, loss_sum_out=tot)
        torch.cuda.synchronize()
        g_t, p_next = c.grad.clone(), c.flat.clone()
        assert torch.isfinite(g_t).all() and torch.isfinite(p_next).all(), "step %d: non-finite gradients / parameters" % t
        # Adam in fp64 from the device's gradients
        p_ref = adam.step(g_t)
        err = (p_next.double().cpu() - p_ref).abs()
        bad = err > adam_bound(p_ref, LR)
        assert not bad.any(), "step %d: %d / %d parameters off fp64 Adam, max err %.3e (lr %g)" % (
            t, int(bad.sum()), err.numel(), err.max().item(), LR)
        # sensitivity: on step t's minibatch (still in the plan's buffers), one step moves the logits by more than 1e-2 of their scale -- beyond every bound used
        # here, so weights one step stale could not pass (the shadow check below is bit-exact in any case)
        l_t, l_next = oracle_logits(c, p_t), oracle_logits(c, p_next)
        rel = (l_next - l_t).abs().max().item() / l_t.abs().max().item()
        assert rel > 1e-2, "step %d: lr %g moves the logits by only %.2e of their scale" % (t, LR, rel)
        # G_t against the oracle at P_t
        check_gradients(c, mode, per, g_t, {k: v.cpu() for k, v in dict_from_flat(p_t, c.dims).items()})
        close(tot, per.sum().reshape(1), 1e-5, "loss sum")
        # shadows: a plan bound to a copy of P_{t+1} (k_weight_shadow) computes what the trained plan (k_adam_shadow) computes
        fresh = plan_like(c, p_next.clone(), torch.zeros_like(p_next))
        for plan in (c.plan, fresh):
            plan.set_step(t + 1)
            plan.sample(c.g, seeds_dev)
        la, lb = c.plan.forward(c.f), fresh.forward(c.f)
        assert torch.equal(la, lb), "step %d: logits of the Adam-written shadows differ from rebuilt ones" % t
        pa, _ = c.plan.loss_backward(c.f, 1.0 / B)
        pb, _ = fresh.loss_backward(c.f, 1.0 / B)
        torch.cuda.synchronize()
        assert torch.equal(pa, pb), "step %d: losses of the Adam-written shadows differ from rebuilt ones" % t
        assert torch.equal(c.grad, fresh._grads), "step %d: gradients of the Adam-written shadows differ from rebuilt ones" % t


def _run_form(form, mode, n_steps=5, B=48):
    import ogl_b200
    c = make_case("2layer", mode)
    rng = np.random.default_rng(3)
    allseeds = rng.permutation(c.V - 40)[:n_steps * B].astype(np.int64)
    flat_seeds = torch.as_tensor(allseeds)
    batches = [flat_seeds[i * B:(i + 1) * B] for i in range(n_steps)]
    batches = [b.cuda() if i % 3 == 0 else (b.pin_memory() if i % 3 == 1 else b.clone()) for i, b in enumerate(batches)]
    per = torch.empty(n_steps * B, device="cuda")
    sums = torch.empty(n_steps, device="cuda")
    plan = c.plan
    out = lambda i: dict(per_vertex_out=per[i * B:(i + 1) * B], loss_sum_out=sums[i:i + 1])
    if form in ("graph", "direct"):
        plan.set_option("cuda_graph", int(form == "graph"))
        for i, sd in enumerate(batches):
            plan.train_step(c.g, c.f, sd, loss_scale=1.0 / B, do_step=True, **out(i))
    elif form == "begin_finish":
        for i, sd in enumerate(batches):
            plan.step_begin(c.g, c.f, sd)
            plan.step_finish(c.f, 1.0 / B, do_step=True, **out(i))
    elif form == "head_tail":
        for i, sd in enumerate(batches):
            plan.step_begin(c.g, c.f, sd)
            plan.step_finish_head(c.f, 1.0 / B, **out(i))
            plan.step_finish_tail(c.f)
            plan.adam_step()
    elif form == "train_steps":
        plan.train_steps(c.g, c.f, flat_seeds.pin_memory(), B, per_vertex_out=per, loss_sums_out=sums)
    elif form == "prefetch":
        plan.prefetch(c.g, c.f, batches[0])
        for i, sd in enumerate(batches):
            if i + 1 < n_steps:
                plan.prefetch(c.g, c.f, batches[i + 1])
            plan.train_step(c.g, c.f, sd, loss_scale=1.0 / B, do_step=True, **out(i))
    elif form == "pipeline":
        pipe = ogl_b200.parallel.Pipeline(plan, c.g, c.f, c.grad, B)
        pipe.begin(batches[0])
        for i in range(n_steps):
            pipe.finish(batches[i + 1] if i + 1 < n_steps else None, **out(i))
        pipe.flush()
    torch.cuda.synchronize()
    return c.flat.clone(), per.clone(), sums.clone()


FORMS = ("direct", "begin_finish", "head_tail", "train_steps", "prefetch", "pipeline")


@pytest.mark.parametrize("mode", list(MODES))
def test_step_forms_are_bit_identical(mode):
    """every form of the train step runs the same kernels on the same operands in the same order -- reverse edge lists in canonical
    order, one Adam arithmetic whether it is split across the backward pass or not -- so from one initial state they end in the
    same bits: parameters, per-vertex losses and loss sums"""
    ref = _run_form("graph", mode)
    for form in FORMS:
        got = _run_form(form, mode)
        for name, a, b in zip(("parameters", "per-vertex losses", "loss sums"), ref, got):
            assert torch.equal(a, b), "%s: %s differ between the graph-replayed step and %s (max diff %.3e)" % (
                mode, name, form, (a - b).abs().max().item())
