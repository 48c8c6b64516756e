"""Perf experiments on the tcgen05 kernels at the shapes of the Reddit-shaped step, next to cuBLAS (torch.matmul) on the same
operands."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from ogl_b200 import native


def bench(fn, iters=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


for (m, n, k) in ((89000, 602, 602), (18432, 600, 600), (18432, 602, 600)):
    ldk = (k + 7) // 8 * 8
    a = torch.randn(m, ldk, device="cuda").bfloat16()
    b = (torch.randn(n, ldk, device="cuda") * 0.05).bfloat16()
    bias = torch.randn(n, device="cuda")
    fl = 2.0 * m * n * k
    ref = torch.relu(a[:, :k].float() @ b[:, :k].float().t() + bias)
    ac, bc = a[:, :k].contiguous(), b[:, :k].contiguous()
    ms = bench(lambda: torch.matmul(ac, bc.t()))
    print("NT m=%d n=%d k=%d cuBLAS (no epilogue)      %.4f ms  %.0f TFLOP/s" % (m, n, k, ms, fl / ms / 1e9), flush=True)
    for cg in (1, 2):
        out = native.gemm_bf16_nt_ex(a, b, k=k, out_bf16=True, bias=bias, relu=True, cg=cg)
        err = (out.float() - ref).abs().max().item()
        ms = bench(lambda: native.gemm_bf16_nt_ex(a, b, k=k, out_bf16=True, bias=bias, relu=True, cg=cg))
        print("NT m=%d n=%d k=%d cg=%d  %.4f ms  %.0f TFLOP/s  max_err %.3g" % (m, n, k, cg, ms, fl / ms / 1e9, err), flush=True)

for (m, n, k) in ((89000, 602, 602), (18432, 600, 602), (18432, 600, 600), (18432, 41, 600)):
    ldn, ldk = (n + 7) // 8 * 8, (k + 7) // 8 * 8
    a = torch.randn(m, ldn, device="cuda").bfloat16()
    b = torch.randn(m, ldk, device="cuda").bfloat16()
    fl = 2.0 * m * n * k
    ref = a[:, :n].float().t() @ b[:, :k].float()
    ac, bc = a[:, :n].contiguous(), b[:, :k].contiguous()
    ms = bench(lambda: torch.matmul(ac.t(), bc))
    print("TN m=%d n=%d k=%d cuBLAS                    %.4f ms  %.0f TFLOP/s" % (m, n, k, ms, fl / ms / 1e9), flush=True)
    ws = torch.empty(1 << 24, device="cuda")
    got = native.gemm_bf16_tn(a, b, n=n, k=k, workspace_elems=1 << 24)
    err = (got - ref).abs().max().item() / ref.abs().max().item()
    ms = bench(lambda: native.gemm_bf16_tn(a, b, n=n, k=k, workspace_elems=1 << 24))
    print("TN m=%d n=%d k=%d ours                      %.4f ms  %.0f TFLOP/s  rel_err %.3g" % (m, n, k, ms, fl / ms / 1e9, err), flush=True)

# ---- launch floor: the same kernels on one or two tiles (prologue + pipeline fill + drain + teardown, no steady state)
for (m, n, k) in ((256, 600, 600), (2048, 600, 600), (1024, 41, 600)):
    ldk = (k + 7) // 8 * 8
    a = torch.randn(m, ldk, device="cuda").bfloat16()
    b = (torch.randn(n, ldk, device="cuda") * 0.05).bfloat16()
    bias = torch.randn(n, device="cuda")
    for cg in (1, 2):
        ms = bench(lambda: native.gemm_bf16_nt_ex(a, b, k=k, out_bf16=True, bias=bias, relu=True, cg=cg), iters=50)
        print("floor NT m=%d n=%d k=%d cg=%d  %.2f us" % (m, n, k, cg, ms * 1e3), flush=True)
for (m, n, k) in ((512, 600, 600), (1024, 41, 600)):
    ldn, ldk = (n + 7) // 8 * 8, (k + 7) // 8 * 8
    a = torch.randn(m, ldn, device="cuda").bfloat16()
    b = torch.randn(m, ldk, device="cuda").bfloat16()
    ms = bench(lambda: native.gemm_bf16_tn(a, b, n=n, k=k, workspace_elems=1 << 24), iters=50)
    print("floor TN m=%d n=%d k=%d (+ split reduce)  %.2f us" % (m, n, k, ms * 1e3), flush=True)
x = torch.zeros(1 << 20, device="cuda")
ms = bench(lambda: x.add_(1.0), iters=200)
print("floor torch elementwise 4 MB  %.2f us" % (ms * 1e3), flush=True)
