"""The train step's sampled-block memory kernels one by one, in all four arithmetic modes, each against a reference computed from the
inputs the kernel actually read (read back from the plan, tests/block_oracle.py):

- k_segmax_fwd: neigh value-equal and the argmax slot exactly equal (first slot attaining the maximum) over the full pitch, pad rows 0;
- the reverse edge lists (k_rev_count / k_rev_fill / k_rev_sort / k_rev_sort_long): offsets and ascending entries exactly equal;
- k_pool_bwd: bit-exact against the sequential fp32 sum in list order, rounded once to the storage type, pad rows 0;
- k_colsum_partial / k_colsum_final: the three bias gradients (with fp16's 1 / loss scale) within n * 2^-24 * sum |x| of fp64 sums;
- k_xent: per-vertex loss and dlogits against an fp64 log-softmax, pad columns and rows of the dlogits exactly 0.

The minibatches aim at the edges: star-shaped hubs picked 1 ... 1025 times in one block (each size class of the list sort) and one
picked 25,600 times at the benchmarked width, ties between repeat picks, between equal feature rows of distinct sources and at ReLU
zeros, fp16-large and tiny values, isolated seeds, partial 16-byte column strips, a level of more than 8,192 rows (more than 32
column-sum chunks), 255 / 256 / 257 seeds, 2 ... 41 classes with logits past exp's fp32 range, a short minibatch after a long one on
the same plan, and the fused train step replayed as a CUDA graph."""
import numpy as np
import pytest
import torch

from oracle import sage as osage
from block_oracle import BITS, colsum_ref, pool_bwd_ref, reverse_lists_ref, segmax_ref, storage_ulp, to_storage, xent_ref

pytestmark = pytest.mark.gpu

MODES = ("fp32", "tf32", "bf16", "fp16")
NAMES = ("fc_pool.weight", "fc_pool.bias", "fc_self.weight", "fc_self.bias", "fc_neigh.weight", "fc_neigh.bias")
STAR_SIZES = (1, 2, 8, 9, 31, 32, 33, 1024, 1025)     # picks of one source in one block: the thread / warp / CTA sort classes


def _pad128(n):
    return (n + 127) // 128 * 128


def param_views(flat, dims):
    """name -> view into a flat fp32 parameter (or gradient) buffer laid out like the plan's"""
    out, off = {}, 0
    for i in range(len(dims) - 1):
        fi, fo = dims[i], dims[i + 1]
        for n, shape in zip(NAMES, ((fi, fi), (fi,), (fo, fi), (fo,), (fo, fi), (fo,))):
            k = int(np.prod(shape))
            out[f"layers.{i}.{n}"] = flat[off:off + k].view(shape)
            off += k
    assert off == flat.numel()
    return out


class Setup:
    """graph (in-edges src -> dst), feature store, plan and bound parameters in one arithmetic mode"""

    def __init__(self, mode, dims, fanouts, V, src, dst, feats, labels, max_seeds, params):
        import ogl_b200
        self.mode, self.dims, self.fanouts, self.L = mode, list(dims), list(fanouts), len(fanouts)
        m = {"fp32": ogl_b200.OGL_F32, "tf32": ogl_b200.OGL_TF32, "bf16": ogl_b200.OGL_BF16, "fp16": ogl_b200.OGL_FP16}[mode]
        self.g = ogl_b200.native.Graph(V, len(src))
        self.g.insert_vertices(V)
        self.g.insert_edges(torch.as_tensor(src).cuda(), torch.as_tensor(dst).cuda(), symmetric=False)
        self.labels = torch.as_tensor(labels).cuda()
        self.f = ogl_b200.native.Features(V, dims[0], m)
        self.f.write(0, torch.as_tensor(feats).cuda(), self.labels)
        self.flat = torch.cat([params[f"layers.{i}.{n}"].reshape(-1).float() for i in range(self.L) for n in NAMES]).cuda()
        self.grad = torch.zeros_like(self.flat)
        self.plan = ogl_b200.native.Plan(self.dims, self.fanouts, max_seeds, V, mode=m, seed=7)
        self.plan.bind_params(self.flat, self.grad)

    def gs(self, loss_scale):
        """the power of two fp16's stored activation gradients carry (1 in the other modes)"""
        return osage.grad_scale_for(loss_scale) if self.mode == "fp16" else 1.0


def _bits(t, mode):
    return t.contiguous().view(BITS[mode])


def check_block_kernels(s, gs):
    """every layer's segment max, reverse lists, max-pool backward and bias sums; returns {hop: row lengths of its reverse lists}"""
    plan, L, mode = s.plan, s.L, s.mode
    grads = param_views(s.grad, s.dims)
    lens = {}
    for l in range(L):
        h = L - 1 - l
        fan, what = s.fanouts[h], f"{mode} layer {l}"
        n_dst, n_src = plan.level_nodes(h).numel(), plan.level_nodes(h + 1).numel()
        lid = plan.block_edges(h)[0]
        hp, neigh, arg = plan.tensor(f"hp{l}"), plan.tensor(f"neigh{l}"), plan.tensor(f"arg{l}")
        nmax_dst, nmax_src = neigh.shape[0], hp.shape[0]

        # k_segmax_fwd over the full pitch
        ref_n, ref_a = segmax_ref(hp[:n_src], lid, n_dst, fan)
        assert torch.equal(neigh[:n_dst].float(), ref_n), "%s: neigh differs in %d elements" % (
            what, int((neigh[:n_dst].float() != ref_n).sum()))
        bad = arg[:n_dst] != ref_a
        assert not bad.any(), "%s: %d argmax slots differ, first at %s (device %d, first maximum %d)" % (
            what, int(bad.sum()), bad.nonzero()[0].tolist(), int(arg[:n_dst][bad][0]), int(ref_a[bad][0]))
        assert not neigh[n_dst:min(_pad128(n_dst), nmax_dst)].float().any(), what + ": neigh pad rows not zero"

        # reverse edge lists: all nmax_src + 1 offsets, the live entries
        rp, re = plan.tensor(f"rev_ptr{h}").view(-1), plan.tensor(f"rev_edge{h}").view(-1)
        ptr, edge = reverse_lists_ref(lid, n_dst, fan, nmax_src)
        assert rp.numel() == nmax_src + 1 and torch.equal(rp.long(), ptr), what + ": reverse list offsets differ"
        n_e = int(ptr[n_src])
        bad = re[:n_e].long() != edge
        assert not bad.any(), "%s: %d reverse list entries differ (of %d)" % (what, int(bad.sum()), n_e)
        lens[h] = (ptr[1:n_src + 1] - ptr[:n_src]).cpu()

        # k_pool_bwd: bit-exact, rows [0, pad128(n_src)), every column
        dng, dhp = plan.tensor(f"dng{l}"), plan.tensor(f"dhp{l}")
        ref = to_storage(pool_bwd_ref(dng[:n_dst], arg[:n_dst], rp, re, n_src), mode)
        bad = _bits(dhp[:n_src], mode) != _bits(ref, mode)
        assert not bad.any(), "%s: dhp differs in %d elements, first at %s (device %r, reference %r)" % (
            what, int(bad.sum()), bad.nonzero()[0].tolist(), float(dhp[:n_src][bad][0]), float(ref[bad][0]))
        assert not _bits(dhp[n_src:min(_pad128(n_src), nmax_src)], mode).any(), what + ": dhp pad rows not zero"

        # bias gradients: fc_pool.bias = colsum(dng), fc_self.bias = fc_neigh.bias = colsum(dpre), times 1 / gs
        dpre = plan.tensor(f"dpre{l}")
        for name, x, cols in (("fc_pool.bias", dng, s.dims[l]), ("fc_self.bias", dpre, s.dims[l + 1])):
            ref, mag = colsum_ref(x, n_dst, cols)
            got = grads[f"layers.{l}.{name}"].double()
            err, bound = (got - ref / gs).abs(), n_dst * 2.0 ** -24 * mag / gs
            assert bool((err <= bound).all()), "%s: %s off by %.3e (bound %.3e, sum %.3e)" % (
                what, name, float((err - bound).max()), float(bound[(err - bound).argmax()]), float(ref[(err - bound).argmax()]))
        assert torch.equal(grads[f"layers.{l}.fc_self.bias"], grads[f"layers.{l}.fc_neigh.bias"]), what
    return lens


def check_xent(s, per_loss, loss_scale):
    """k_xent against the fp64 log-softmax of the logits it read"""
    plan, mode, C = s.plan, s.mode, s.dims[-1]
    n = plan.level_nodes(0).numel()
    logits = plan.tensor(f"out{s.L - 1}")[:n, :C]
    y = s.labels[plan.level_nodes(0).long()]
    lse, loss, p = xent_ref(logits, y)
    ly = logits.double().gather(1, y[:, None]).squeeze(1)
    tol_l = 8 * 2.0 ** -23 * torch.maximum(torch.maximum(lse.abs(), ly.abs()), torch.ones_like(lse)) + C * 2.0 ** -24
    err = (per_loss.double() - loss).abs()
    assert bool((err <= tol_l).all()), "%s: loss off by %.3e (lse %.3f)" % (mode, float(err.max()), float(lse[err.argmax()]))
    scale = loss_scale * s.gs(loss_scale)
    g_ref = (p - torch.nn.functional.one_hot(y, C).double()) * scale
    d = plan.tensor(f"dpre{s.L - 1}", rows=_pad128(n))
    tol = storage_ulp(g_ref, mode) + (p * tol_l[:, None] + 2.0 ** -22) * abs(scale)
    err = (d[:n, :C].double() - g_ref).abs()
    assert bool((err <= tol).all()), "%s: dlogits off by %.3e (tolerance %.3e)" % (mode, float(err.max()), float(tol.flatten()[err.argmax()]))
    assert not d[:n, C:].float().any() and not d[n:].float().any(), mode + ": dlogits pad columns / rows not zero"


# ---------------------------------------------------------------------------------------------------------------------------------
def star_graph(rng, sizes, NR=3000, n_iso=8):
    """a random region [0, NR) (in-degree 8, a fifth of the picks from 16 popular sources), then one hub per size m with m leaves whose
    only in-neighbour is the hub (the last hub has no in-edges itself), then isolated vertices.  -> (V, src, dst, hubs, leaves, iso)"""
    E = NR * 8
    src = [np.where(rng.random(E) < 0.2, rng.integers(0, 16, E), rng.integers(0, NR, E))]
    dst = [rng.integers(0, NR, E)]
    hubs = NR + np.arange(len(sizes))
    off, leaves = NR + len(sizes), []
    for i, (hub, m) in enumerate(zip(hubs, sizes)):
        if i + 1 < len(sizes):
            src.append(rng.integers(0, NR, 6))
            dst.append(np.full(6, hub))
        leaves.append(np.arange(off, off + m))
        src.append(np.full(m, hub))
        dst.append(leaves[-1])
        off += m
    iso = np.arange(off, off + n_iso)
    return off + n_iso, np.concatenate(src).astype(np.int64), np.concatenate(dst).astype(np.int64), hubs, leaves, iso


def star_features(rng, V, NR, F):
    """ties and range: 30 % of the random region copies one of 12 rows, column 1 is negative everywhere (hp = 0: rows whose maximum
    is 0), column 2 holds 6e4 in a tenth of the rows, column 3 multiples of 2^-20 in a fifth; ReLU zeros elsewhere"""
    x = rng.standard_normal((V, F)).astype(np.float32)
    dup = np.nonzero(rng.random(NR) < 0.3)[0]
    x[dup] = x[rng.integers(0, NR, 12)[rng.integers(0, 12, dup.size)]]
    x[:, 1] = -np.abs(x[:, 1]) - 0.5
    x[rng.random(V) < 0.1, 2] = 6.0e4
    tiny = rng.random(V) < 0.2
    x[tiny, 3] = 2.0 ** -20 * rng.integers(1, 4, int(tiny.sum()))
    return x


def star_params(dims):
    """layer 0: fc_pool = identity without bias, so hp is relu(x) exactly in every mode, and the 6e4 column enters fc_self / fc_neigh
    times 2^-16.  Layer 1: fc_pool.bias opens columns c % 5 == 0 (+4) and closes c % 5 == 1 (-1e3: exact ReLU zeros), fc_neigh
    selects dneigh[:, c] = dpre[:, c % C]"""
    p = osage.xavier_params(dims[0], dims[1], dims[-1], len(dims) - 2, seed=1)
    p["layers.0.fc_pool.weight"] = torch.eye(dims[0])
    p["layers.0.fc_pool.bias"] = torch.zeros(dims[0])
    for n in ("fc_self.weight", "fc_neigh.weight"):
        p["layers.0." + n][:, 2] *= 2.0 ** -16
    c = torch.arange(dims[1])
    b = p["layers.1.fc_pool.bias"]
    b[c % 5 == 0], b[c % 5 == 1] = 4.0, -1.0e3
    C = dims[2]
    p["layers.1.fc_neigh.weight"] = (torch.arange(C)[:, None] == (c % C)[None, :]).float()
    return p


def star_dlogits(rng, n, C, hub_rows, M=0.125):
    """dlogits for backward(): |x| <= M / 64 at random, and in column 0 of every hub's first four leaves M, 0, M * 2^-26, -M (zeros
    after them), so that the hub's fp32 sum depends on the order of its list entries: (M + t) - M = 0 but (M - M) + t = t"""
    d = rng.uniform(-1.0, 1.0, (n, C)) * (M / 64)
    for rows in hub_rows:
        if len(rows) >= 4:
            d[rows, 0] = 0.0
            d[rows[:4], 0] = (M, 0.0, M * 2.0 ** -26, -M)
    return torch.as_tensor(d, dtype=torch.float32).cuda(), M


def _local_rows(plan, level, ids):
    nodes = plan.level_nodes(level).long().cpu().numpy()
    pos = {int(v): i for i, v in enumerate(nodes)}
    return np.array([pos[int(v)] for v in ids])


@pytest.mark.parametrize("mode", MODES)
def test_star_hubs_ties_and_a_short_batch_after_a_long_one(mode):
    """sample -> forward -> backward(dlogits) on stars of 1 ... 1025 leaves (hop 0, fanout 1: a hub's list has exactly m entries; hop 1,
    fanout 4: every leaf picks its hub four times, equal rows), then a short minibatch through the same plan"""
    rng = np.random.default_rng(0)
    NR, dims, fanouts = 3000, (12, 33, 5), (1, 4)
    V, src, dst, hubs, leaves, iso = star_graph(rng, STAR_SIZES, NR)
    rand = rng.choice(NR, 200, replace=False)
    seeds = np.concatenate(leaves[:4] + [iso[:4]] + leaves[4:] + [rand, iso[4:]]).astype(np.int64)
    s = Setup(mode, dims, fanouts, V, src, dst, star_features(rng, V, NR, dims[0]), rng.integers(0, dims[-1], V), len(seeds),
              star_params(dims))
    pos = {int(v): i for i, v in enumerate(seeds)}
    s.plan.sample(s.g, torch.as_tensor(seeds).cuda())
    s.plan.forward(s.f, want_logits=False)
    d, amax = star_dlogits(rng, len(seeds), dims[-1], [np.array([pos[int(v)] for v in lv]) for lv in leaves])
    s.plan.backward(d, amax)
    torch.cuda.synchronize()
    lens = check_block_kernels(s, s.gs(amax))
    # every hub's hop-0 list holds exactly its leaves: each size class of the list sort is reached
    assert lens[0][_local_rows(s.plan, 1, hubs)].tolist() == list(STAR_SIZES)
    assert int(lens[0].max()) > 1024 and bool(((lens[0] > 8) & (lens[0] <= 1024)).any()) and bool(((lens[0] > 1) & (lens[0] <= 8)).any())
    assert int(lens[1].max()) >= 4 * 1025                           # hop 1: four picks per leaf
    # a short minibatch after the long one: every buffer is reused with fewer live rows
    short = np.concatenate([leaves[1], leaves[3], rand[:30], iso[:2]]).astype(np.int64)
    s.plan.sample(s.g, torch.as_tensor(short).cuda())
    s.plan.forward(s.f, want_logits=False)
    d, amax = star_dlogits(rng, len(short), dims[-1], [np.arange(2, 11)])
    s.plan.backward(d, amax)
    torch.cuda.synchronize()
    lens = check_block_kernels(s, s.gs(amax))
    assert lens[0][_local_rows(s.plan, 1, hubs[[1, 3]])].tolist() == [2, 9]


@pytest.mark.parametrize("mode", MODES)
def test_bench_width_hub_through_the_replayed_train_step(mode):
    """the fused train step (captured once, replayed as a CUDA graph) at the benchmarked widths 602 / 600 / 41 and fan-outs 25 / 10:
    1,024 seeds whose only in-neighbour is one hub (25,600 entries in its hop-0 list, 10,240 at hop 1), 1,024 seeds of a random region
    (a level-1 frontier of more than 8,192 rows) and isolated seeds"""
    gen = np.random.default_rng(1)
    NR, deg, dims, fanouts = 60000, 30, (602, 600, 41), (25, 10)
    hub = NR
    leaves = NR + 1 + np.arange(1024)
    iso = NR + 1025 + np.arange(16)
    V = NR + 1041
    src = np.concatenate([gen.integers(0, NR, NR * deg), gen.integers(0, NR, 50), np.full(1024, hub)]).astype(np.int64)
    dst = np.concatenate([gen.integers(0, NR, NR * deg), np.full(50, hub), leaves]).astype(np.int64)
    seeds = np.concatenate([leaves[:512], iso[:8], gen.choice(NR, 1024, replace=False), leaves[512:], iso[8:]]).astype(np.int64)
    feats = torch.randn(V, dims[0], generator=torch.Generator().manual_seed(2))
    s = Setup(mode, dims, fanouts, V, src, dst, feats, gen.integers(0, dims[-1], V), len(seeds),
              osage.xavier_params(dims[0], dims[1], dims[-1], 1, seed=3))
    n = len(seeds)
    per = torch.empty(n, device="cuda")
    s.plan.train_step(s.g, s.f, torch.as_tensor(seeds).cuda(), loss_scale=1.0 / n, do_step=True, per_vertex_out=per)
    torch.cuda.synchronize()
    assert s.plan.graph_stats()["replays"] == 1
    assert s.plan.level_nodes(1).numel() > 32 * 256                # k_colsum_final sums more than 32 chunks
    lens = check_block_kernels(s, s.gs(1.0 / n))
    check_xent(s, per, 1.0 / n)
    assert int(lens[0][_local_rows(s.plan, 1, [hub])][0]) == 25600
    assert int(lens[1][_local_rows(s.plan, 2, [hub])][0]) == 10240


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("n,C", [(255, 2), (256, 31), (257, 32), (255, 33), (256, 41)])
def test_xent_and_bias_sums_at_row_and_class_edges(mode, n, C):
    """255 / 256 / 257 seeds (the column sums' 256-row chunks, the dlogits' 128-row padding), C at 32-lane boundaries, and head biases
    spreading the logits over +-100: exp overflows fp32 beyond 88.7 unless the maximum is subtracted first"""
    rng = np.random.default_rng(n + C)
    V, E, dims = 1500, 9000, (33, 16, C)
    src, dst = rng.integers(0, V - 20, E), rng.integers(0, V - 20, E)
    s = Setup(mode, dims, (3, 2), V, src, dst, rng.standard_normal((V, dims[0])).astype(np.float32), rng.integers(0, C, V), n,
              osage.xavier_params(dims[0], dims[1], C, 1, seed=4))
    p = param_views(s.flat, dims)
    p["layers.1.fc_self.bias"].copy_(torch.linspace(-100.0, 100.0, C)[torch.randperm(C, generator=torch.Generator().manual_seed(C))])
    p["layers.1.fc_neigh.bias"].zero_()
    s.plan.refresh_params()
    seeds = np.concatenate([rng.choice(V - 20, n - 4, replace=False), V - 4 + np.arange(4)]).astype(np.int64)
    s.plan.sample(s.g, torch.as_tensor(seeds).cuda())
    logits = s.plan.forward(s.f)
    per, _ = s.plan.loss_backward(s.f, 1.0 / n)
    torch.cuda.synchronize()
    assert float(logits.max()) > 89.0 and bool(torch.isfinite(per).all())
    check_xent(s, per, 1.0 / n)
    check_block_kernels(s, s.gs(1.0 / n))
