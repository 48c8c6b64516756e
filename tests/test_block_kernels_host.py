"""The block-kernel references of tests/block_oracle.py against independent formulations, on the CPU: the segment max against the
oracle's (oracle/sage.py:segment_max), the reverse edge lists against a per-source loop, and the sequential max-pool backward against
the oracle's autograd gradient routed through the same argmax."""
import numpy as np
import pytest
import torch

from oracle import sage as osage
from block_oracle import (naive_reverse_lists, pool_bwd_ref, reverse_lists_ref, segmax_ref, storage_ulp, to_storage,
                          xent_ref)


def _block(seed, n_dst, n_src, fanout, p_empty=0.15, hub=None):
    """random ELL block: slots -1 with probability p_empty, the first rows entirely empty (isolated), `hub` = (row, count) makes
    row `row` the pick of `count` slots"""
    g = torch.Generator().manual_seed(seed)
    lid = torch.randint(0, n_src, (n_dst * fanout,), generator=g)
    lid[torch.rand(n_dst * fanout, generator=g) < p_empty] = -1
    lid[:3 * fanout] = -1
    if hub is not None:
        row, count = hub
        lid[torch.randperm(n_dst * fanout, generator=g)[:count]] = row
    return lid


@pytest.mark.parametrize("n_dst,n_src,fanout", [(50, 80, 1), (200, 300, 5), (64, 64, 25)])
def test_segmax_ref_matches_the_oracle(n_dst, n_src, fanout):
    """continuous fp64 values (no ties): same maxima, same slots, 255 / 0 on empty rows"""
    lid = _block(n_dst + fanout, n_dst, n_src, fanout)
    hp = torch.randn(n_src, 24, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    neigh, arg = segmax_ref(hp, lid, n_dst, fanout)
    ref_n, ref_a = osage.segment_max(hp, lid, n_dst, fanout)
    ref_a = torch.where(ref_a < 0, torch.full_like(ref_a, 255), ref_a)
    assert torch.equal(arg.long(), ref_a)
    assert torch.equal(neigh.double(), ref_n.float().double())
    assert bool((arg[:3] == 255).all()) and bool((neigh[:3] == 0).all())


def test_segmax_ref_ties_keep_the_first_slot():
    """repeat picks, equal rows of distinct sources, ReLU zeros of both signs: the first slot attaining the maximum wins"""
    hp = torch.tensor([[0.0, 1.0, -0.0], [0.0, 1.0, 0.0], [-0.0, 0.5, 0.0]])
    lid = torch.tensor([2, 0, 1, 0, -1, 1, -1, -1, -1])
    neigh, arg = segmax_ref(hp, lid, 3, 3)
    assert arg.tolist() == [[0, 1, 0], [0, 0, 0], [255, 255, 255]]
    assert neigh.tolist() == [[0.0, 1.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 0.0]]


@pytest.mark.parametrize("n_dst,n_src,fanout,hub", [(40, 60, 1, None), (300, 500, 4, (7, 900)), (60, 90, 25, (0, 1100))])
def test_reverse_lists_ref_matches_a_per_source_loop(n_dst, n_src, fanout, hub):
    lid = _block(fanout, n_dst, n_src, fanout, hub=hub)
    n_src_max = n_src + 13                                        # rows past the live count stay empty
    ptr, edge = reverse_lists_ref(lid, n_dst, fanout, n_src_max)
    ptr_n, edge_n = naive_reverse_lists(lid, n_dst, fanout, n_src_max)
    assert np.array_equal(ptr.numpy(), ptr_n) and np.array_equal(edge.numpy(), edge_n)
    if hub is not None:
        assert int(ptr[hub[0] + 1] - ptr[hub[0]]) >= hub[1]


@pytest.mark.parametrize("n_dst,n_src,fanout,hub", [(80, 120, 1, (3, 60)), (200, 150, 6, (10, 1030)), (40, 30, 10, None)])
def test_pool_bwd_ref_matches_the_oracle_gradient(n_dst, n_src, fanout, hub):
    """summed in fp64, the list-order gather equals the gradient the oracle's segment max routes through the same argmax"""
    lid = _block(7 * fanout, n_dst, n_src, fanout, hub=hub)
    g = torch.Generator().manual_seed(2)
    hp = torch.relu(torch.randn(n_src, 16, dtype=torch.float64, generator=g)).requires_grad_(True)
    neigh, arg = osage.segment_max(hp, lid, n_dst, fanout)
    dng = torch.randn(n_dst, 16, dtype=torch.float64, generator=g)
    (neigh * dng).sum().backward()
    ptr, edge = reverse_lists_ref(lid, n_dst, fanout, n_src)
    arg8 = torch.where(arg < 0, torch.full_like(arg, 255), arg).to(torch.uint8)
    got = pool_bwd_ref(dng, arg8, ptr, edge, n_src, acc=torch.float64)
    assert torch.allclose(got, hp.grad, rtol=1e-12, atol=1e-12)
    # fp32: the order of the sum is the list order (a different order gives other roundings somewhere)
    dng32 = dng.float() * 1e3
    a = pool_bwd_ref(dng32, arg8, ptr, edge, n_src)
    ref = torch.zeros(n_src, 16, dtype=torch.float32)
    for s in range(n_src):
        for e in edge[ptr[s]:ptr[s + 1]].tolist():
            d, j = e >> 8, e & 255
            ref[s] = ref[s] + torch.where(arg8[d].long() == j, dng32[d], torch.zeros(()))
    assert torch.equal(a.view(torch.int32), ref.view(torch.int32))


def test_storage_rounding_and_ulp():
    x = torch.tensor([1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 65520.0, 2.0 ** -20, -3.0])
    assert to_storage(x, "fp16").float().tolist() == [1.0, 1.0 + 2.0 ** -9, float("inf"), 2.0 ** -20, -3.0]
    assert to_storage(x, "tf32").tolist()[:2] == [1.0 + 2.0 ** -10, 1.0 + 2.0 ** -9]      # ties away from zero
    assert storage_ulp(torch.tensor([1.0, 2.0 ** -30]), "fp16").tolist() == [2.0 ** -10, 2.0 ** -24]
    assert storage_ulp(torch.tensor([3.0]), "bf16").tolist() == [2.0 ** -6]


def test_xent_ref_is_stable_at_large_logits():
    logits = torch.tensor([[100.0, -100.0, 99.0], [0.0, 0.0, 0.0]])
    lse, loss, p = xent_ref(logits, torch.tensor([2, 1]))
    assert torch.isfinite(lse).all() and abs(float(loss[0]) - (1.0 + np.log1p(np.exp(-1.0) + np.exp(-200.0)))) < 1e-12
    assert abs(float(loss[1]) - np.log(3.0)) < 1e-12 and torch.allclose(p.sum(1), torch.ones(2, dtype=torch.float64))
