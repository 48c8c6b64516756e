"""GraphSAGE-pool forward/backward, loss and Adam -- oracle only (torch CPU).

Layer formula = DGL SAGEConv(in, out, 'pool') as imported at
train/graphsage/pytorch/graphsage_dgl.py:3 and unrolled by the reference itself at
inference_optimized.py:135-139,258-260,273-276:

    h_self = x[:n_dst];  hp = relu(fc_pool(x));  neigh[d] = max_{e: dst(e)=d} hp[src(e)] (0 if none)
    out = fc_self(h_self) + fc_neigh(neigh);  relu unless last layer

Model = GraphSAGE(F, H, C, n_layers=depth-1, relu, dropout, 'pool')
(graphsage_dgl.py:10-59; `pool_feats`/`edge_feats` are ignored there, so fc_pool is in->in).
Loss = CrossEntropyLoss(mean | none) on labels.flatten(), Adam(lr=1e-3)
(pytorch/model.py:20-25,103-107).  PARITY UNPINNED against DGL (absent); the argmax tie
rule (lowest edge slot wins) is this repo's specification.

``quant='bf16'`` / ``quant='tf32'`` / ``quant='fp16'`` model the product's tensor-core paths: every GEMM
operand (activations, weights, activation gradients) is rounded to bf16 / TF32 / fp16 exactly where the
product stores it, accumulation stays fp32/fp64.  fp16 also models the product's static loss scaling
(csrc/plan.cu: grad_scale_for): activation gradients are rounded AS STORED, i.e. times a power of two
chosen from the loss scale, so that the rounding grid (and fp16's subnormal range) is the device's.  ``quant=None`` is the reference's own fp32
arithmetic (train/utils.py:63-64) -- the oracle every tolerance is stated against; the
quantised variants only show that a kernel implements the arithmetic it claims.
"""
import math
import torch

_QUANT = [None]          # rounding of the autograd functions below; set per call by forward()
_GSCALE = [1.0]          # quant='fp16': the power of two the stored activation gradients carry (set by loss_and_grads)


def grad_scale_for(loss_scale):
    """csrc/plan.cu: grad_scale_for -- 2^floor(log2(64 / loss_scale)): the largest |dlogits| element is stored in (32, 64]"""
    a = abs(float(loss_scale))
    if not (a > 0.0) or math.isinf(a):
        return 1.0
    m, e = math.frexp(64.0 / a)
    return math.ldexp(1.0, e - 1)


def round_tf32(x):
    """nearest TF32 (10 explicit mantissa bits), ties away from zero -- PTX cvt.rna.tf32.f32"""
    b = x.detach().to(torch.float32).contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32).to(x.dtype)


def _round(x):
    if _QUANT[0] == "tf32":
        return round_tf32(x)
    if _QUANT[0] == "fp16":
        return x.to(torch.float16).to(x.dtype)
    return x.to(torch.bfloat16).to(x.dtype)


def _round_grad(g):
    """an activation gradient as the product stores it (fp16: times the loss scale, see _GSCALE)"""
    if _QUANT[0] == "fp16" and _GSCALE[0] != 1.0:
        return _round(g * _GSCALE[0]) / _GSCALE[0]
    return _round(g)


def xavier_params(in_feats, n_hidden, n_classes, n_layers, seed, dtype=torch.float32):
    """Parameters with DGL SAGEConv.reset_parameters() semantics [recalled]: Xavier-uniform
    weights with gain=sqrt(2) (calculate_gain('relu')), nn.Linear default biases.
    Key names follow the reference state_dict (inference_optimized.py:135-139)."""
    g = torch.Generator().manual_seed(seed)
    dims = [(in_feats, n_hidden)] + [(n_hidden, n_hidden)] * (n_layers - 1) + [(n_hidden, n_classes)]
    p = {}
    for i, (fi, fo) in enumerate(dims):
        for name, (o, k) in (("fc_pool", (fi, fi)), ("fc_self", (fo, fi)), ("fc_neigh", (fo, fi))):
            a = math.sqrt(2.0) * math.sqrt(6.0 / (o + k))
            p[f"layers.{i}.{name}.weight"] = ((torch.rand(o, k, generator=g, dtype=torch.float64) * 2 - 1) * a).to(dtype)
            b = 1.0 / math.sqrt(k)
            p[f"layers.{i}.{name}.bias"] = ((torch.rand(o, generator=g, dtype=torch.float64) * 2 - 1) * b).to(dtype)
    return p


class _Q(torch.autograd.Function):
    """Round to bf16 in forward AND round the incoming gradient to bf16 in backward
    (the product stores activation gradients once, in bf16)."""
    @staticmethod
    def forward(ctx, x):
        return _round(x)

    @staticmethod
    def backward(ctx, g):
        return _round_grad(g)


class _Qf(torch.autograd.Function):
    """Round forward only (weights / leaves: their gradients stay full precision)."""
    @staticmethod
    def forward(ctx, x):
        return _round(x)

    @staticmethod
    def backward(ctx, g):
        return g


class _Qb(torch.autograd.Function):
    """Identity forward, round the gradient (models a stored bf16 activation gradient)."""
    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return _round_grad(g)


def segment_max(hp, edge_src, n_dst, fanout, arg=None):
    """neigh[d, f] = max_j hp[edge_src[d*fanout+j], f]; empty slots (-1) ignored; rows with
    no edge give 0.  Returns (neigh, argslot[int64 n_dst x F], -1 where no edge).  Gradient
    flows only to the FIRST slot attaining the max.

    ``arg`` (int64 [n_dst, F], -1 = no edge) overrides the slot choice: used by the bf16 parity
    tests to route the gradient through the slots the device picked, after checking that every
    device slot attains the oracle's max within one bf16 ulp (in bf16 two neighbours often round
    to the same value, so WHICH of them is 'the' argmax is decided by the last bit of the fp32
    accumulation order -- not something a different summation order can reproduce)."""
    F_ = hp.shape[1]
    es = edge_src.view(n_dst, fanout)
    valid = es >= 0
    vals = hp[es.clamp(min=0)]                                  # [n_dst, fanout, F]
    neg = torch.full((), -float("inf"), dtype=hp.dtype)
    vals = torch.where(valid[:, :, None], vals, neg)
    mx = vals.max(dim=1).values
    if arg is not None:
        first = arg.clamp(min=0)
    else:
        first = (vals == mx[:, None, :]).to(torch.int8).argmax(dim=1)   # first slot attaining the max
    picked = torch.gather(vals, 1, first[:, None, :]).squeeze(1)
    has = valid.any(dim=1)
    neigh = torch.where(has[:, None], picked, torch.zeros((), dtype=hp.dtype))
    arg = torch.where(has[:, None].expand(-1, F_), first, torch.full((), -1, dtype=torch.int64))
    return neigh, arg


def dropout_keep(n_rows, n_cols, p, seed, step, layer):
    """keep mask [n_rows, n_cols] (bool) of the product's feat_drop (csrc/sage_kernels.cu: k_feat_drop):
    keep(r, c) = philox4x32_10(counter = (c >> 2, r, 0xD0 + layer, optimiser step), key = seed)[c & 3] >= floor(p * 2^32)"""
    import numpy as np
    from .philox import philox4x32, split_seed
    k0, k1 = split_seed(seed)
    q = (n_cols + 3) // 4
    w = philox4x32(np.arange(q, dtype=np.uint64)[None, :], np.arange(n_rows, dtype=np.uint64)[:, None], 0xD0 + layer, step, k0, k1)
    words = np.stack(w, axis=-1).reshape(n_rows, 4 * q)[:, :n_cols]
    thresh = min(4294967295, int(math.floor(float(np.float32(p)) * 4294967296.0)))
    return torch.from_numpy(words.astype(np.int64) >= thresh)


def sage_layer(x, n_dst, edge_src, fanout, Wp, bp, Ws, bs, Wn, bn, relu_out, quant=None, arg=None, mask_hp=None, mask_out=None, drop=None):
    """``mask_hp`` / ``mask_out`` (bool, optional) replace the two ReLUs by a fixed on/off pattern: together with ``arg`` they pin
    the piecewise-linear region in which the layer is evaluated (oracle/parity.py: the device's region, to compare gradients
    without the jumps that a sign or an argmax decided inside rounding error causes)."""
    q = _Q.apply if quant else (lambda t: t)
    qf = _Qf.apply if quant else (lambda t: t)
    if drop is not None:                       # SAGEConv's feat_drop: (keep mask, 1 / (1 - p)) on the layer input, once
        keep, scale = drop
        x = q(torch.where(keep, x * scale, torch.zeros((), dtype=x.dtype)))
    hp_pre = x @ qf(Wp).t() + bp
    hp = q(torch.relu(hp_pre) if mask_hp is None else torch.where(mask_hp, hp_pre, torch.zeros((), dtype=hp_pre.dtype)))
    neigh, arg = segment_max(hp, edge_src, n_dst, fanout, arg=arg)
    if quant:
        neigh = _Qb.apply(neigh)
    out_pre = x[:n_dst] @ qf(Ws).t() + neigh @ qf(Wn).t() + (bs + bn)
    out = out_pre
    if relu_out:
        out = q(torch.relu(out_pre) if mask_out is None else torch.where(mask_out, out_pre, torch.zeros((), dtype=out_pre.dtype)))
    return out, dict(hp=hp, neigh=neigh, arg=arg, hp_pre=hp_pre.detach(), out_pre=out_pre.detach())


def forward(params, x_in, blocks, quant=None):
    """blocks: list (input layer first) of dict(n_dst, edge_src[int64], fanout[, arg]).  x_in: features
    of blocks[0]'s src nodes.  Returns (logits, per-layer intermediates)."""
    assert quant in (None, "bf16", "tf32", "fp16")
    _QUANT[0] = quant
    h = _Qf.apply(x_in) if quant else x_in
    inter = []
    L = len(blocks)
    for i, b in enumerate(blocks):
        g = lambda n: params[f"layers.{i}.{n}"]
        h, it = sage_layer(h, b["n_dst"], b["edge_src"], b["fanout"],
                           g("fc_pool.weight"), g("fc_pool.bias"), g("fc_self.weight"), g("fc_self.bias"),
                           g("fc_neigh.weight"), g("fc_neigh.bias"), relu_out=(i < L - 1), quant=quant, arg=b.get("arg"),
                           mask_hp=b.get("mask_hp"), mask_out=b.get("mask_out"), drop=b.get("drop"))
        it["out"] = h
        inter.append(it)
    return h, inter


def xent(logits, labels, reduction="mean", quant=None):
    if quant:
        logits = _Qb.apply(logits)
    return torch.nn.functional.cross_entropy(logits, labels.flatten(), reduction=reduction)


def loss_and_grads(params, x_in, blocks, labels, quant=None, dtype=torch.float32, reduction="mean", loss_mult=1.0, grad_scale=None):
    """One fwd+bwd of loss = loss_mult * cross_entropy(reduction).  Returns (loss, per_vertex_loss, logits, grads dict, intermediates).
    quant='fp16': grad_scale is the power of two the device's stored activation gradients carry; default: the fused step's for
    the mean over the labels (the autograd bridge picks it from max |dlogits|: grad_scale_for(max |dlogits|))."""
    p = {k: v.detach().to(dtype).requires_grad_(True) for k, v in params.items()}
    if grad_scale is None:
        grad_scale = grad_scale_for(1.0 / max(1, labels.numel()))
    _GSCALE[0] = grad_scale if quant == "fp16" else 1.0
    logits, inter = forward(p, x_in.to(dtype), blocks, quant=quant)
    per = xent(logits, labels, "none", quant=quant)
    loss = loss_mult * (per.mean() if reduction == "mean" else per.sum())
    loss.backward()
    return loss.detach(), per.detach(), logits.detach(), {k: v.grad for k, v in p.items()}, inter


def adam_step(params, grads, state, lr=1e-3, b1=0.9, b2=0.999, eps=1e-8):
    """torch.optim.Adam defaults (pytorch/model.py:25), single step, in place."""
    state["t"] = state.get("t", 0) + 1
    t = state["t"]
    for k, p in params.items():
        g = grads[k].to(p.dtype)
        m = state.setdefault("m." + k, torch.zeros_like(p))
        v = state.setdefault("v." + k, torch.zeros_like(p))
        m.mul_(b1).add_(g, alpha=1 - b1)
        v.mul_(b2).addcmul_(g, g, value=1 - b2)
        bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
        denom = (v.sqrt() / math.sqrt(bc2)).add_(eps)
        p.addcdiv_(m, denom, value=-(lr / bc1))
    return params
