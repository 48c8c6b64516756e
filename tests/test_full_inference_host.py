"""Full-neighbourhood inference, host side (no GPU): the edge-list reference full_forward (tests/full_oracle.py) against the
block oracle, and the driver's --eval_neighbourhood flag."""
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import sage as osage
from oracle.graph import in_csr
from full_oracle import full_forward

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("quant", [None, "bf16", "tf32", "fp16"])
def test_full_forward_equals_the_block_oracle_on_the_whole_graph(quant):
    """with every vertex as a destination and every in-edge as a slot, the ELL block oracle (sage_layer) and the edge-list full_forward
    compute the same layers at the same rounding points: identical results, isolated vertices included"""
    rng = np.random.default_rng(0)
    V, E, dims = 80, 300, (12, 9, 9, 4)
    src, dst = rng.integers(0, V, E), rng.integers(0, V - 6, E)
    ip, ix, _ = (np.asarray(a) for a in in_csr(src, dst, V))
    fan = int(np.diff(ip).max())
    ell = -np.ones((V, fan), dtype=np.int64)
    for v in range(V):
        ell[v, :ip[v + 1] - ip[v]] = ix[ip[v]:ip[v + 1]]
    params = osage.xavier_params(dims[0], dims[1], dims[-1], len(dims) - 2, seed=1)
    x = torch.randn(V, dims[0], dtype=torch.float64)
    blocks = [dict(n_dst=V, edge_src=torch.from_numpy(ell.reshape(-1)), fanout=fan)] * (len(dims) - 1)
    ref, _ = osage.forward({k: v.double() for k, v in params.items()}, x, blocks, quant=quant)
    got = full_forward(params, ip, ix, x, quant=quant)
    assert torch.equal(got, ref.detach())
    assert bool((np.diff(ip)[-6:] == 0).all())


def _driver():
    spec = importlib.util.spec_from_file_location("ogl_train_main", os.path.join(ROOT, "train", "__main__.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_driver_eval_neighbourhood_flag():
    m = _driver()
    assert m.parse(["pubmed", "pytorch", "o.csv", "t", "--cuda"])[1]["eval_neighbourhood"] == "sampled"
    assert m.parse(["pubmed", "pytorch", "o.csv", "t", "--cuda", "--eval_neighbourhood", "full"])[1]["eval_neighbourhood"] == "full"
    with pytest.raises(SystemExit):
        m.parse(["pubmed", "pytorch", "o.csv", "t", "--cuda", "--eval_neighbourhood", "exact"])
