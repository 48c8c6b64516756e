"""NVLink peer-memory gradient exchange fused with Adam (csrc/peer.cu), exercised on ONE GPU: two ranks live in this process, each
with its own plan / stream, wired with ogl_peer_connect_local.  The multi-process (CUDA IPC) wiring is the same kernels behind
ogl_peer_connect; bench.py --gpus N runs it."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from test_gpu_sage import Case  # noqa: E402


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_peer_adam_two_ranks_equals_summed_gradient_adam(mode, offset):
    """every rank loads every peer's gradients and sums them in rank order: the sum equals the summed gradient bit for bit, and the
    weights equal Adam on it.  offset = 0: the data-parallel pipeline's two buckets; 1: the bucket boundary moved one float off the
    16-byte grid, so that both buckets also run the kernel's scalar head / tail loops"""
    from ogl_b200 import native
    W, B = 2, 64
    kw = dict(dims=(64, 32, 5), fanouts=(6, 4), n_seeds=B, mode=mode, gemm_impl=0 if mode == "bf16" else 1)
    ranks = [Case(**kw) for _ in range(W)]
    ref = Case(**kw)
    n = ref.plan.n_params
    peers = [native.Peer(r, W, n) for r in range(W)]
    native.Peer.connect_local(peers)
    for c, p in zip(ranks, peers):
        c.plan.bind_params(c.flat, p.grads)
    rng = np.random.default_rng(9)
    streams = [torch.cuda.Stream() for _ in range(W)]
    n0 = ref.plan.tail_params + offset
    reduced = [torch.zeros(n, device="cuda") for _ in range(W)]
    for step in range(3):
        for r, c in enumerate(ranks):
            seeds = torch.as_tensor(rng.permutation(c.V - 40)[:B].astype(np.int64)).cuda()
            peers[r].wait_readers()
            c.plan.train_step(c.g, c.f, seeds, loss_scale=1.0 / (W * B), do_step=False)
        torch.cuda.synchronize()
        want = peers[0].grads.clone()
        for r in range(1, W):
            want += peers[r].grads
        ref.grad.copy_(want)
        ref.plan.adam_step()
        # two buckets; every rank on its own stream (the kernels wait for each other)
        for lo, hi, last in ((n0, n, False), (0, n0, True)):
            for r, c in enumerate(ranks):
                with torch.cuda.stream(streams[r]):
                    c.plan.peer_adam(peers[r], lo, hi, last, reduced_out=reduced[r])
        torch.cuda.synchronize()
        for r, c in enumerate(ranks):
            assert torch.equal(reduced[r], want), "rank %d: summed gradient differs" % r
            # the same Adam expression in both kernels; allow for different FMA contraction around it
            err = (c.flat - ref.flat).abs().max().item()
            assert err <= 1e-6 * ref.flat.abs().max().item(), "rank %d: weights differ from Adam on the summed gradient (step %d): %g" % (r, step, err)
    assert torch.equal(ranks[0].flat, ranks[1].flat)


def test_peer_adam_single_rank_equals_adam_step():
    from ogl_b200 import native
    B = 32
    kw = dict(dims=(50, 24, 5), fanouts=(5, 3), n_seeds=B, mode="bf16", gemm_impl=0)
    a, b = Case(**kw), Case(**kw)
    peer = native.Peer(0, 1, a.plan.n_params)
    a.plan.bind_params(a.flat, peer.grads)
    seeds = torch.as_tensor(a.seeds).cuda()
    for _ in range(2):
        peer.wait_readers()
        a.plan.train_step(a.g, a.f, seeds, loss_scale=1.0 / B, do_step=False)
        a.plan.peer_adam(peer, 0, a.plan.n_params, True)
        b.plan.train_step(b.g, b.f, seeds, loss_scale=1.0 / B, do_step=True)
    torch.cuda.synchronize()
    # same Adam arithmetic; the gradients differ only by the summation order of the reverse edge lists
    assert (a.flat - b.flat).abs().max().item() <= 1e-4 * b.flat.abs().max().item()


@pytest.mark.parametrize("mode", ["bf16", "tf32"])
def test_one_graph_data_parallel_finish_two_ranks(mode):
    """ogl_plan_step_finish_dp: forward .. backward + both gradient exchanges + Adam as ONE captured launch sequence per rank (the
    exchange kernels take their epoch from device memory, so the graph is replayed every step).  Two ranks in this process, each
    on its own stream: the weights must equal Adam on the summed gradients, and the replicas each other bit for bit."""
    from ogl_b200 import native
    W, B = 2, 64
    kw = dict(dims=(300, 32, 5), fanouts=(6, 4), n_seeds=B, mode=mode, gemm_impl=0)
    ranks = [Case(**kw) for _ in range(W)]
    ref = Case(**kw)
    n = ref.plan.n_params
    peers = [native.Peer(r, W, n) for r in range(W)]
    native.Peer.connect_local(peers)
    for c, p in zip(ranks, peers):
        c.plan.bind_params(c.flat, p.grads)
    rng = np.random.default_rng(4)
    streams = [torch.cuda.Stream() for _ in range(W)]
    for step in range(4):
        seeds = [torch.as_tensor(rng.permutation(ranks[0].V - 40)[:B].astype(np.int64)).cuda() for _ in range(W)]
        torch.cuda.synchronize()
        for r, c in enumerate(ranks):
            with torch.cuda.stream(streams[r]):
                c.plan.step_begin(c.g, c.f, seeds[r])
                c.plan.step_finish_dp(peers[r], c.f, 1.0 / (W * B))
        torch.cuda.synchronize()
        want = peers[0].grads.clone()
        for r in range(1, W):
            want += peers[r].grads
        ref.grad.copy_(want)
        ref.plan.adam_step()
        for r, c in enumerate(ranks):
            err = (c.flat - ref.flat).abs().max().item()
            assert err <= 1e-6 * ref.flat.abs().max().item(), "rank %d, step %d: weights differ from Adam on the summed gradient: %g" % (r, step, err)
        assert torch.equal(ranks[0].flat, ranks[1].flat)
    st = ranks[0].plan.graph_stats()
    assert st["captures"] <= 3 and st["replays"] >= 8, st          # begin + finish graphs captured once, replayed every step
