"""Parity of the benchmarked arithmetic at the BENCHMARKED shape against the unquantised oracle.

Reddit hyper-parameters of BASELINE.json (F / hidden / classes = 602 / 600 / 41, B = 1024, fan-outs 25 / 10) on a 120 k-vertex
graph, so that the hop-2 frontier holds ~9e4 rows and every CTA pair of the persistent tcgen05 GEMMs runs > 10 tiles (accumulator
ping-pong, ring wrap, TMA-store epilogue all in play).  The device step (through the C ABI) is compared with oracle/sage.py in
fp64 with quant=None -- the reference's own fp32 arithmetic (train/utils.py:63-64, pytorch/model.py:96-107) restated -- on the
same sampled blocks.  north_star's tolerance is rtol 1e-3 for the tensor-core modes and 1e-5 for fp32; it is applied here as
|a - b| <= rtol * |b| + atol with atol = rtol * max |b| (single elements of a 600-term dot product cancel to ~0, a pure relative
bound is meaningless for them; DESIGN.md section 5 states the same).  The achieved errors are printed (pytest -s) and returned by
oracle/parity.py for bench.py's JSON line.
"""
import json

import numpy as np
import pytest
import torch

from oracle import parity as opar
from oracle import sage as osage

pytestmark = pytest.mark.gpu

V, E, DIMS, FAN, B = 120000, 6000000, (602, 600, 41), (25, 10), 1024

# mode -> (plan mode name, gemm_impl, rounding of a stored hp value, bounds)
#   logits / loss: max |err| / scale;  grad_pinned: rel. Frobenius with the oracle evaluated in the device's linear region (its
#   max-pool slots and ReLU patterns, each checked to be a valid choice within rounding);  grad_free: rel. Frobenius against the
#   free-running oracle (includes the gradient's jumps between neighbouring regions, see oracle/parity.py)
CASES = {
    "fp32": dict(gemm_impl=1, slot_tol=2.0 ** -20, logits=1e-5, grad_pinned=1e-5, grad_free=5e-3, outside=0.0),
    # tf32: every element of the logits, the losses and (pinned) every gradient within rtol 1e-3 (`outside` = 0); the relative
    # Frobenius error of a TF32 GEMM chain is ~4e-4 per GEMM (two operands rounded at 2^-11), ~1e-3 after the five on the longest path
    "tf32": dict(gemm_impl=0, slot_tol=2.0 ** -10, logits=1e-3, grad_pinned=1.5e-3, grad_free=1e-1, outside=0.0),
    # fp16 storage has TF32's ten explicit mantissa bits; with the static loss scaling of csrc/plan.cu (grad_scale_for) the activation
    # gradients stay in fp16's normal range, so the bounds are tf32's
    "fp16": dict(gemm_impl=0, slot_tol=2.0 ** -10, logits=1e-3, grad_pinned=1.5e-3, grad_free=1e-1, outside=0.0),
    # bf16 is a labelled DEVIATION from the 1e-3 target (bench.py prints its measured error beside the tf32 line)
    "bf16": dict(gemm_impl=0, slot_tol=2.0 ** -8, logits=1e-2, grad_pinned=1e-2, grad_free=3e-1, outside=0.5),
}

_world = {}


def world():
    if not _world:
        import ogl_b200
        rng = np.random.default_rng(1)
        # degree-skewed endpoints (squared uniform) so that hubs and low-degree rows both occur
        src = (rng.random(E) ** 1.3 * V).astype(np.int64)
        dst = rng.integers(0, V, E).astype(np.int64)
        g = ogl_b200.native.Graph(V, 2 * E)
        g.insert_vertices(V)
        g.insert_edges(torch.as_tensor(src).cuda(), torch.as_tensor(dst).cuda(), symmetric=True)
        feats = torch.from_numpy(rng.standard_normal((V, DIMS[0])).astype(np.float32))
        labels = torch.from_numpy(rng.integers(0, DIMS[-1], V).astype(np.int64))
        params = osage.xavier_params(DIMS[0], DIMS[1], DIMS[2], 1, seed=0)
        seeds = rng.permutation(V)[:B].astype(np.int64)
        _world.update(g=g, feats=feats, labels=labels, params=params, seeds=seeds)
    return _world


@pytest.mark.parametrize("mode", ["tf32", "fp16", "bf16", "fp32"])
def test_step_vs_unquantised_oracle_at_bench_shape(mode):
    import ogl_b200
    w, c = world(), CASES[mode]
    m = {"fp32": ogl_b200.OGL_F32, "tf32": ogl_b200.OGL_TF32, "bf16": ogl_b200.OGL_BF16, "fp16": ogl_b200.OGL_FP16}[mode]
    fs = ogl_b200.native.Features(V, DIMS[0], m)
    fs.write(0, w["feats"].cuda(), w["labels"].cuda())
    flat = torch.cat([w["params"]["layers.%d.%s" % (i, n)].reshape(-1).float() for i in range(2) for n in opar.NAMES]).cuda()
    grad = torch.zeros_like(flat)
    plan = ogl_b200.native.Plan(list(DIMS), list(FAN), B, V, mode=m, seed=11, gemm_impl=c["gemm_impl"])
    plan.bind_params(flat, grad)
    seeds_dev = torch.as_tensor(w["seeds"]).cuda()
    plan.sample(w["g"], seeds_dev)
    logits = plan.forward(fs)
    per, tot = plan.loss_backward(fs, 1.0 / B)
    torch.cuda.synchronize()
    res = opar.compare_step(plan, w["params"], w["feats"], w["labels"], w["seeds"], logits, per, grad, c["slot_tol"])
    s = opar.summary(res)
    print("\nPARITY %s %s" % (mode, json.dumps(s)))
    n1, n0 = res["level_counts"][1], res["level_counts"][2]
    assert n0 > 80000 and n1 > 20000, "frontier too small to exercise the persistent GEMM loops: %r" % (res["level_counts"],)
    assert s["argmax_not_a_max_within_rounding"] == [0, 0], s["argmax_not_a_max_within_rounding"]
    assert s["relu_sign_not_within_rounding"] == [0, 0, 0], s["relu_sign_not_within_rounding"]
    assert s["logits_max_err_of_scale"] <= c["logits"], s
    assert s["loss_max_err_of_scale"] <= c["logits"], s
    assert s["logits_frac_outside_rtol"] <= c["outside"], s
    assert s["grad_rel_fro_pinned_max"] <= c["grad_pinned"], s
    if mode != "bf16":
        assert s["grad_frac_outside_rtol_pinned_max"] == 0.0, s          # every gradient element within rtol * |b| + rtol * scale
    if mode == "fp32":
        assert s["grad_max_err_of_scale_pinned_max"] <= c["logits"], s
    assert s["grad_rel_fro_free_max"] <= c["grad_free"], s
    if mode != "fp32":
        # the graph-replayed fused step on the same minibatch (same Philox step) reproduces the direct launches
        direct = grad.clone()
        plan.set_step(0)
        per2 = torch.empty(B, device="cuda")
        plan.train_step(w["g"], fs, seeds_dev, loss_scale=1.0 / B, do_step=False, per_vertex_out=per2)
        torch.cuda.synchronize()
        # the step launches the kernels of sample + forward + loss_backward on the same operands, and the reverse edge lists are in
        # canonical order, so the max-pool backward sums in the same order too: bit-identical
        assert torch.equal(per2, per), "fused step losses differ from the direct launches by %g" % (per2 - per).abs().max().item()
        assert torch.equal(grad, direct), "fused step gradients differ from the direct launches by %g" % (grad - direct).abs().max().item()
