"""Test reference of full-neighbourhood inference (DGL's model.inference(g, x)) on the CPU, for the full-inference tests.

Every layer runs over EVERY vertex with its whole in-neighbourhood, in eval mode, with the layer formula and rounding points of
oracle/sage.py:sage_layer: ``quant`` rounds the layer input, the weights, hp and the hidden outputs where the product stores them
(bf16 / TF32 / fp16), accumulation in ``dtype``.  The segment max is a scatter_reduce('amax') over the edge list -- no ELL: hubs would
make one huge -- and rows without in-edges give 0."""
import torch

from oracle.sage import round_tf32


def _rounder(quant):
    if quant is None:
        return lambda t: t
    if quant == "tf32":
        return round_tf32
    if quant == "fp16":
        return lambda t: t.to(torch.float16).to(t.dtype)
    assert quant == "bf16", quant
    return lambda t: t.to(torch.bfloat16).to(t.dtype)


def full_forward(params, indptr, indices, x, quant=None, dtype=torch.float64):
    """params: state_dict-style `layers.<i>.<fc>.<weight|bias>` of the layers to run; in-CSR indptr [V+1], indices [E] = sources;
    x [V, F].  Returns the logits [V, C] in `dtype`."""
    q = _rounder(quant)
    indptr = torch.as_tensor(indptr, dtype=torch.int64)
    src = torch.as_tensor(indices, dtype=torch.int64)
    V = indptr.numel() - 1
    deg = indptr[1:] - indptr[:-1]
    dst = torch.repeat_interleave(torch.arange(V), deg)
    has = deg > 0
    h = q(x.to(dtype))
    L = len({k.split(".")[1] for k in params})
    with torch.no_grad():
        for i in range(L):
            g = lambda n: params[f"layers.{i}.{n}"].to(dtype)
            hp = q(torch.relu(h @ q(g("fc_pool.weight")).t() + g("fc_pool.bias")))
            neigh = torch.zeros_like(hp)
            if src.numel():
                neigh = neigh.scatter_reduce(0, dst[:, None].expand(-1, hp.shape[1]), hp[src], "amax", include_self=False)
            neigh = torch.where(has[:, None], neigh, torch.zeros((), dtype=dtype))
            out = h @ q(g("fc_self.weight")).t() + neigh @ q(g("fc_neigh.weight")).t() + (g("fc_self.bias") + g("fc_neigh.bias"))
            h = q(torch.relu(out)) if i < L - 1 else out
    return h
