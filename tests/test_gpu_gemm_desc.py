"""The train step's GEMM descriptors (csrc/gemm.cuh: GemmNT, GemmTN) against a plain fp64 reference of their contract, in the forms
the plan builds them (csrc/plan.cu: pool_gemm, out_gemm, plan_backward_layers), on every path of the dispatcher: tcgen05 with one
CTA per tile, with CTA pairs and the automatic choice, and the SIMT kernels.

Operands are drawn in the mode's storage type, so their products are exact in fp32 and a result differs from the fp64 reference
only by the fp32 accumulation, |err| <= 1e-6 * (sqrt(K) + 8) * scale, and by the rounding of a stored output to its type (one unit
of 2^-8 for bf16, 2^-11 for tf32 and fp16).  Everything the contract says is never read is filled with NaN: A rows at or past
round_up(rows_valid, 128), pad columns >= k, B rows >= n.  Such a run must equal, bit for bit, a run on the same path whose
unread elements are zero.  Rows [rows_valid, round_up(rows_valid, 128)) hold zeros, the precondition the producers keep.

The plan-level tests at the end run a step after a longer one on the same plan and compare it with a fresh plan's step: a step's
results must not depend on what earlier steps left in the plan's buffers.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

NAN = float("nan")


def _ru(x, m):
    return (x + m - 1) // m * m


def _modes():
    import ogl_b200
    # name -> (mode, storage dtype, one rounding unit of a stored output)
    return {"bf16": (ogl_b200.OGL_BF16, torch.bfloat16, 2.0 ** -8), "tf32": (ogl_b200.OGL_TF32, torch.float32, 2.0 ** -11),
            "fp16": (ogl_b200.OGL_FP16, torch.float16, 2.0 ** -11), "fp32": (ogl_b200.OGL_F32, torch.float32, 2.0 ** -23)}


def _paths(mode_name):
    """(label, force_simt, cg) of every path a mode can take"""
    simt = [("simt", True, 0)]
    if mode_name == "fp32":
        return simt
    return [("cg1", False, 1), ("cg2", False, 2), ("auto", False, 0)] + simt


def _operand(shape, mode_name, gen, scale=1.0):
    from ogl_b200 import native
    mode, dtype, _ = _modes()[mode_name]
    x = torch.randn(shape, generator=gen, device="cuda") * scale
    if mode_name == "tf32":
        x = native.round_tf32(x)
    return x.to(dtype)


def _bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def _row_count(sel, m_max):
    """a dynamic row count of the grids below: an int, or "max", "max-1", "max+5", ... relative to the static bound"""
    return sel if isinstance(sel, int) else m_max + int(sel[3:] or 0)


def _i32(v):
    return torch.tensor([int(v)], dtype=torch.int32, device="cuda")


# ---------------------------------------------------------------------------------------------------------------- NT descriptors
# (layer dims d0, d1, d2; static row bound of the layer's source level; row bound of its destination level)
SIZES = {"small": dict(dims=(64, 64, 8), m_max=1200, nmax_dst=600),
         # the bench model at the Reddit shape: max_seeds 1024, fanouts (25, 10) -> 26,624 source rows, 3 column tiles of 600: every
         # CTA pair runs 4 - 5 tiles
         "bench": dict(dims=(602, 600, 41), m_max=26624, nmax_dst=1024)}
BUILDERS = ["pool", "hidden_out", "logits_out", "dneigh", "dx"]
M_DYN = [1, 127, 128, 129, 255, 256, 257, "max-1", "max", "max+5"]     # (m_max + 5 is clamped to m_max)
N_DST = [0, 1, 100, 128, 129, 300, 384, 385, None]     # (None: the dynamic row count)
DX_ALPHA = [1.0, 2.0, 1.0 / 0.7]


def _nt_problem(builder, size, mode_name, gen):
    """full-size random buffers of one descriptor form, laid out as the plan lays them out (row pitch round_up(d, 8))"""
    d0, d1, d2 = SIZES[size]["dims"]
    m_max, nmax_dst = SIZES[size]["m_max"], SIZES[size]["nmax_dst"]
    p8 = lambda d: _ru(d, 8)                       # noqa: E731  (plan.cu pitch_of)
    op = lambda r, c, s=1.0: _operand((r, c), mode_name, gen, s)   # noqa: E731
    bias = lambda n: 0.1 * torch.randn(n, generator=gen, device="cuda")   # noqa: E731
    pr = dict(relu=False, bias=None, bias2=None, mask=None, out_f32=False, zero_tail=True, bounded=False)
    if builder == "pool":                          # hp = relu(x Wp^T + bp)
        k, n = d0, d0
        pr.update(segs=[(op(m_max, p8(k)), op(n + 40, p8(k), k ** -0.5), k, m_max)], n=n, ldc=p8(n), bias=bias(n), relu=True)
    elif builder in ("hidden_out", "logits_out"):  # [h_self | neigh] [Ws | Wn]^T + bs + bn
        k, n = (d0, d1) if builder == "hidden_out" else (d1, d2)
        pr.update(segs=[(op(m_max, p8(k)), op(n + 40, p8(k), k ** -0.5), k, m_max) for _ in range(2)], n=n, ldc=p8(n),
                  bias=bias(n), bias2=bias(n), relu=builder == "hidden_out", out_f32=builder == "logits_out")
    elif builder == "dneigh":                      # dneigh = mask(neigh) * (dpre Wn), no zero tail
        k, n = d2, d1
        pr.update(segs=[(op(m_max, p8(k)), op(n + 40, p8(k), k ** -0.5), k, m_max)], n=n, ldc=p8(n), zero_tail=False)
        pr["mask"] = op(m_max, p8(n))
    else:                                          # dx: mask(act) * alpha * (dhp Wp + [dpre Ws on the first n_dst rows])
        n = d1
        pr.update(segs=[(op(m_max, p8(d1)), op(n + 40, p8(d1), d1 ** -0.5), d1, m_max),
                        (op(_ru(nmax_dst, 128), p8(d2)), op(n + 40, p8(d2), d2 ** -0.5), d2, _ru(nmax_dst, 128))],
                  n=n, ldc=p8(n), bounded=True)
        pr["mask"] = op(m_max, p8(n))
    if pr["mask"] is not None:                     # positive, +0, -0 and negative entries
        pr["mask"][::3] = 0.0
        pr["mask"][1::7] = -0.0
    pr["m_max"], pr["nmax_dst"] = m_max, nmax_dst
    return pr


def _nt_inputs(pr, m_dyn, rvs, poison):
    """operands of one launch: rows [rv, round_up(rv, 128)) zero, everything never read = poison"""
    segs = []
    for (a, b, k, rows), rv in zip(pr["segs"], rvs):
        a = a.clone()
        pad = min(_ru(rv, 128), rows)
        a[rv:pad] = 0
        a[pad:] = poison
        a[:, k:] = poison
        b = b.clone()
        b[pr["n"]:] = poison
        b[:, k:] = poison
        segs.append((a, b, k))
    mask = None
    if pr["mask"] is not None:
        mask = pr["mask"].clone()
        mask[m_dyn:] = poison
        mask[:, pr["n"]:] = poison
    return segs, mask


def _nt_reference(pr, segs, mask, m_dyn, rvs, alpha):
    """fp64 result of rows [0, m_dyn) and the scale of its accumulation error"""
    n = pr["n"]
    acc = torch.zeros(m_dyn, n, dtype=torch.float64, device="cuda")
    for (a, b, k), rv in zip(segs, rvs):
        if rv:
            acc[:rv] += a[:rv, :k].double() @ b[:n, :k].double().t()
    acc *= alpha
    scale = acc.abs().max().item() if m_dyn else 0.0
    ref = acc
    for bb in (pr["bias"], pr["bias2"]):
        if bb is not None:
            ref = ref + bb.double()
    if pr["relu"]:
        ref = torch.relu(ref)
    if mask is not None:
        ref = torch.where(mask[:m_dyn, :n].double() > 0, ref, torch.zeros_like(ref))
    return ref, scale


def _nt_launch(pr, mode_name, path, segs, mask, m_dyn_dev, rows_dev, alpha):
    from ogl_b200 import native
    mode, dtype, _ = _modes()[mode_name]
    _, simt, cg = path
    c = torch.full((pr["m_max"], pr["ldc"]), NAN, dtype=torch.float32 if pr["out_f32"] else dtype, device="cuda")
    args = [(a, b, k, rows_dev if (pr["bounded"] and i == 1) else None, rows)
            for i, ((a, b, k), (_, _, _, rows)) in enumerate(zip(segs, pr["segs"]))]
    native.gemm_nt(c, args, pr["m_max"], pr["n"], mode, m_dev=m_dyn_dev, bias=pr["bias"], bias2=pr["bias2"], relu=pr["relu"],
                   alpha=alpha, mask=mask, out_f32=pr["out_f32"], zero_tail=pr["zero_tail"], cg=cg, force_simt=simt)
    return c


def _nt_check(pr, c, ref, bound, m_dyn, path, what):
    """the rows and columns of the output: results, zero tail, what the kernels write past them and what they leave alone"""
    n, ldc, m_max = pr["n"], pr["ldc"], pr["m_max"]
    m_pad = min(_ru(m_dyn, 128), m_max) if pr["zero_tail"] else m_dyn
    cf = c.double()
    err = (cf[:m_dyn, :n] - ref).abs()
    assert bool((err <= bound).all()), "%s: max err %.3e over bound (%.3e at the worst element)" % (
        what, err.max().item(), bound.flatten()[err.flatten().argmax()].item() if err.numel() else 0.0)
    assert bool((cf[m_dyn:m_pad, :n] == 0).all()), what + ": zero tail"
    tc = path[0] != "simt"
    # columns [n, ldc): the tcgen05 epilogues store zeros there (whole store boxes), the SIMT kernel does not touch them
    if ldc > n:
        pad_cols = cf[:m_pad, n:]
        assert bool((pad_cols == 0).all() if tc else pad_cols.isnan().all()), what + ": pad columns"
    # rows past the zero tail: the TMA-store epilogues write whole 128-row tiles (256-row tiles of a CTA pair) with zeros; the
    # rest is never written
    hi = min(_ru(m_pad, 256), m_max) if tc else m_pad
    between = cf[m_pad:hi]
    assert bool(((between == 0) | between.isnan()).all()), what + ": rows past the zero tail"
    assert bool(cf[hi:].isnan().all()), what + ": rows past the last tile were written"


@pytest.mark.parametrize("size", list(SIZES))
@pytest.mark.parametrize("mode_name", ["bf16", "tf32", "fp16", "fp32"])
@pytest.mark.parametrize("builder", BUILDERS)
def test_gemm_nt_descriptor(builder, mode_name, size):
    ulp = _modes()[mode_name][2]
    gen = torch.Generator(device="cuda").manual_seed(BUILDERS.index(builder) * 10 + len(mode_name) + len(size))
    pr = _nt_problem(builder, size, mode_name, gen)
    m_max, nmax_dst = pr["m_max"], pr["nmax_dst"]
    K = sum(k for _, _, k, _ in pr["segs"])
    it = 0
    for m_sel in M_DYN:
        m_dev = _row_count(m_sel, m_max)
        m_dyn = min(m_dev, m_max)
        n_dsts = sorted({min(m_dyn if v is None else v, m_dyn, nmax_dst) for v in N_DST}) if pr["bounded"] else [None]
        for n_dst in n_dsts:
            alpha = DX_ALPHA[it % 3] if builder == "dx" else 1.0
            it += 1
            rvs = [m_dyn] + ([n_dst] if pr["bounded"] else [m_dyn] * (len(pr["segs"]) - 1))
            segs, mask = _nt_inputs(pr, m_dyn, rvs, NAN)
            clean_segs, clean_mask = _nt_inputs(pr, m_dyn, rvs, 0.0)
            ref, scale = _nt_reference(pr, segs, mask, m_dyn, rvs, alpha)
            out_ulp = 2.0 ** -23 if pr["out_f32"] else ulp
            bound = 1e-6 * (K ** 0.5 + 8) * scale + out_ulp * ref.abs() + 2.0 ** -25
            m_dyn_dev, rows_dev = _i32(m_dev), _i32(n_dst if n_dst is not None else 0)
            got = {}
            for path in _paths(mode_name):
                what = "%s %s %s m_dyn %d n_dst %s alpha %.4g %s" % (builder, mode_name, size, m_dev, n_dst, alpha, path[0])
                c = _nt_launch(pr, mode_name, path, segs, mask, m_dyn_dev, rows_dev, alpha)
                _nt_check(pr, c, ref, bound, m_dyn, path, what)
                again = _nt_launch(pr, mode_name, path, segs, mask, m_dyn_dev, rows_dev, alpha)
                assert torch.equal(_bits(c), _bits(again)), what + ": two identical launches differ"
                clean = _nt_launch(pr, mode_name, path, clean_segs, clean_mask, m_dyn_dev, rows_dev, alpha)
                assert torch.equal(_bits(c), _bits(clean)), what + ": the result depends on elements that are never read"
                got[path[0]] = c[:m_dyn, :pr["n"]].double()
            for x, y in (("simt", "auto"), ("cg1", "cg2")):
                if x in got and y in got:
                    assert bool(((got[x] - got[y]).abs() <= 2 * bound).all()), "%s %s %s m_dyn %d n_dst %s: %s and %s disagree" % (
                        builder, mode_name, size, m_dev, n_dst, x, y)


# ---------------------------------------------------------------------------------------------------------------- TN descriptors
# a layer's weight-gradient group: dW_pool of the layer above (in' x in'), dW_self and dW_neigh (out x in); a fourth (in x out)
# fills the group
TN_SIZES = {"small": dict(dims=(64, 8), m_max=1200), "bench": dict(dims=(600, 41), m_max=26624)}
TN_ALPHA = [2.0 ** -7, 1.0, 0.5, 3.0]
TN_M_DYN = [1, 100, 1001, "max-3", "max+5"]


def _tn_expect_error(path, shapes, ws):
    """the dispatcher's workspace rule: the tcgen05 path stores a single problem directly when the split partials do not fit and
    needs them for a group; the SIMT path always stages its splits"""
    if path[1]:
        return ws is None or ws < max(n * k for n, k in shapes)
    return len(shapes) > 1 and (ws is None or ws < sum(n * _ru(k, 4) for n, k in shapes))


@pytest.mark.parametrize("count", [1, 2, 3, 4])
@pytest.mark.parametrize("size", list(TN_SIZES))
@pytest.mark.parametrize("mode_name", ["bf16", "tf32", "fp16", "fp32"])
def test_gemm_tn_group_descriptor(mode_name, size, count):
    import ogl_b200
    from ogl_b200 import native
    mode = _modes()[mode_name][0]
    d_in, d_out = TN_SIZES[size]["dims"]
    m_max = TN_SIZES[size]["m_max"]
    shapes = [(d_in, d_in), (d_out, d_in), (d_out, d_in), (d_in, d_out)][:count]
    gen = torch.Generator(device="cuda").manual_seed(count * 7 + len(mode_name) + len(size))
    full = [(_operand((m_max, _ru(n, 8)), mode_name, gen), _operand((m_max, _ru(k, 8)), mode_name, gen)) for n, k in shapes]
    one_split = sum(n * _ru(k, 4) for n, k in shapes)
    wss = {"none": None, "short": one_split - 1, "one_split": one_split, "plan": max(n * k for n, k in shapes) * 32, "large": 1 << 25}
    for m_sel in TN_M_DYN:
        m_dev = _row_count(m_sel, m_max)
        m_dyn = min(m_dev, m_max)
        pad = min(_ru(m_dyn, 128), m_max)

        def inputs(poison):
            ops = []
            for a, b in full:
                a, b = a.clone(), b.clone()
                a[m_dyn:pad] = 0                      # the activation gradients' zero tail; the other operand's rows are real there
                a[pad:] = poison
                b[pad:] = poison
                ops.append((a, b))
            return ops

        ops, clean_ops = inputs(NAN), inputs(0.0)
        for i, (n, k) in enumerate(shapes):         # pad columns are never read either
            ops[i][0][:, n:] = NAN
            ops[i][1][:, k:] = NAN
        refs = [TN_ALPHA[i] * (a[:m_dyn, :n].double().t() @ b[:m_dyn, :k].double()) for i, ((n, k), (a, b)) in enumerate(zip(shapes, ops))]
        m_dyn_dev = _i32(m_dev)
        for path in _paths(mode_name):
            got = {}
            for ws_name, ws in wss.items():
                what = "TN %s %s count %d m_dyn %d ws %s %s" % (mode_name, size, count, m_dev, ws_name, path[0])

                def launch(operands):
                    outs = [torch.full((n, k), NAN, device="cuda") for n, k in shapes]
                    probs = [(a, b, c, n, k, TN_ALPHA[i]) for i, ((n, k), (a, b), c) in enumerate(zip(shapes, operands, outs))]
                    w = torch.zeros(ws, device="cuda") if ws is not None else None
                    native.gemm_tn_group(probs, m_max, mode, m_dev=m_dyn_dev, workspace=w, force_simt=path[1])
                    return outs

                if _tn_expect_error(path, shapes, ws):
                    with pytest.raises(ogl_b200.OglError, match="error -2"):
                        launch(ops)
                    continue
                outs = launch(ops)
                for i, (c, ref) in enumerate(zip(outs, refs)):
                    err = (c.double() - ref).abs()
                    scale = ref.abs().max().item()
                    assert bool((err <= 1e-6 * (m_dyn ** 0.5 + 8) * scale + 1e-30).all()), "%s problem %d: max err %.3e (scale %.3e)" % (
                        what, i, err.max().item(), scale)
                again, clean = launch(ops), launch(clean_ops)
                for c, c2, c3 in zip(outs, again, clean):
                    assert torch.equal(_bits(c), _bits(c2)), what + ": two identical launches differ"
                    assert torch.equal(_bits(c), _bits(c3)), what + ": the result depends on rows that are never read"
                got[ws_name] = outs
            if path[0] != "simt":
                # the split count follows the workspace; every split count gives the reference's result within the bound, and
                # one split (the direct store and the single-split reduce) must agree exactly
                if "none" in got:
                    for x, y in zip(got["none"], got["one_split"]):
                        assert torch.equal(_bits(x), _bits(y)), "TN %s %s m_dyn %d: direct store and single-split reduce differ" % (
                            mode_name, size, m_dev)


# ---------------------------------------------------------------------------------------------------------------- plan steps
PLAN_V = 40000
PLAN_MODES = {"bf16": 0, "tf32": 0, "fp16": 0, "fp32": 1}        # -> gemm_impl (fp32: the SIMT kernels, the control)


@pytest.fixture(scope="module")
def graph40k():
    """40,000 vertices, mean in-degree 15: with max_seeds 1,024 and fanouts (25, 10) the level below the seeds holds up to 26,624
    rows, enough source-row tiles for the layer-1 dx GEMM to run on CTA pairs"""
    from ogl_b200 import native
    rng = np.random.default_rng(4)
    E = 300000
    g = native.Graph(PLAN_V, 2 * E)
    g.insert_vertices(PLAN_V)
    g.insert_edges(torch.as_tensor(rng.integers(0, PLAN_V, E)).cuda(), torch.as_tensor(rng.integers(0, PLAN_V, E)).cuda(), symmetric=True)
    return g, rng.permutation(PLAN_V)


_FEATS = {}


def _features(F, C, mode_name):
    from ogl_b200 import native
    key = (F, C, mode_name)
    if key not in _FEATS:
        gen = torch.Generator().manual_seed(F + C)
        f = native.Features(PLAN_V, F, _modes()[mode_name][0])
        f.write(0, torch.randn(PLAN_V, F, generator=gen).cuda(), torch.randint(0, C, (PLAN_V,), generator=gen).cuda())
        _FEATS[key] = f
    return _FEATS[key]


def _fresh_plan(dims, fanouts, mode_name):
    from ogl_b200 import native
    from oracle import sage as osage
    from test_gpu_sage import flat_from_dict
    L = len(fanouts)
    flat = flat_from_dict(osage.xavier_params(dims[0], dims[1], dims[-1], L - 1, seed=1), L).cuda()
    grad = torch.zeros_like(flat)
    plan = native.Plan(list(dims), list(fanouts), 1024, PLAN_V, mode=_modes()[mode_name][0], seed=11, gemm_impl=PLAN_MODES[mode_name])
    plan.bind_params(flat, grad)
    return plan, grad


def _poison(plan):
    for l in range(plan.L):
        for name in ("dpre", "hp", "neigh", "out"):
            plan.tensor("%s%d" % (name, l)).fill_(NAN)


def _fused_tail(plan, grad, g, f, tail, step):
    plan.set_step(step)
    per = torch.empty(len(tail), device="cuda")
    plan.train_step(g, f, tail, loss_scale=1.0 / len(tail), do_step=False, per_vertex_out=per)
    torch.cuda.synchronize()
    return grad.clone(), per


def _tail_after_full_batch(graph40k, dims, fanouts, mode_name, n_tail, poison):
    g, perm = graph40k
    f = _features(dims[0], dims[-1], mode_name)
    seeds = torch.as_tensor(perm[:1024]).cuda()
    tail = torch.as_tensor(perm[1024:1024 + n_tail]).cuda()
    plan, grad = _fresh_plan(dims, fanouts, mode_name)
    plan.train_step(g, f, seeds, do_step=False)
    if poison:
        _poison(plan)
    ga, pa = _fused_tail(plan, grad, g, f, tail, 5)
    fresh, fgrad = _fresh_plan(dims, fanouts, mode_name)
    gb, pb = _fused_tail(fresh, fgrad, g, f, tail, 5)
    what = "%s %s fanouts %s tail %d" % (mode_name, dims, fanouts, n_tail)
    assert bool(torch.isfinite(ga).all()), what + ": non-finite gradients"
    assert torch.equal(pa, pb), what + ": per-vertex losses depend on the earlier step"
    assert torch.equal(ga, gb), what + ": gradients depend on the earlier step (%d of %d differ)" % (int((ga != gb).sum()), ga.numel())


@pytest.mark.parametrize("n_tail", [100, 129, 300, 1000])
@pytest.mark.parametrize("mode_name", list(PLAN_MODES))
def test_tail_step_does_not_read_an_earlier_step(graph40k, mode_name, n_tail):
    """the trainers' ragged tail after full batches on the same plan: dpre of the last layer is zero only up to
    round_up(n_tail, 128), rows past that hold the full batch's gradients"""
    _tail_after_full_batch(graph40k, (64, 64, 8), (25, 10), mode_name, n_tail, poison=False)


@pytest.mark.parametrize("n_tail", [100, 129, 300, 1000])
@pytest.mark.parametrize("mode_name", list(PLAN_MODES))
def test_tail_step_over_poisoned_buffers(graph40k, mode_name, n_tail):
    """every activation and gradient buffer NaN before the step: nothing past the rows a step writes is read"""
    _tail_after_full_batch(graph40k, (64, 64, 8), (25, 10), mode_name, n_tail, poison=True)


@pytest.mark.parametrize("mode_name", list(PLAN_MODES))
def test_tail_step_three_layers(graph40k, mode_name):
    """three layers: the level counts below the seeds change from step to step, so every step meets rows an earlier one wrote"""
    for n_tail in (100, 300):
        _tail_after_full_batch(graph40k, (64, 64, 64, 8), (25, 10, 5), mode_name, n_tail, poison=False)


@pytest.mark.parametrize("mode_name", list(PLAN_MODES))
def test_tail_step_bench_shape(graph40k, mode_name):
    _tail_after_full_batch(graph40k, (602, 600, 41), (25, 10), mode_name, 100, poison=True)


@pytest.mark.parametrize("mode_name", list(PLAN_MODES))
def test_autograd_bridge_step_after_a_larger_one(graph40k, mode_name):
    """the autograd bridge's order (sample, forward, backward of caller-made dlogits) with a batch that shrinks"""
    g, perm = graph40k
    dims, fanouts = (64, 64, 8), (25, 10)
    f = _features(dims[0], dims[-1], mode_name)
    gen = torch.Generator(device="cuda").manual_seed(3)

    def bridge_step(plan, seeds, step, dlogits):
        plan.set_step(step)
        plan.sample(g, seeds)
        logits = plan.forward(f)
        plan.backward(dlogits)
        torch.cuda.synchronize()
        return logits

    big, small = torch.as_tensor(perm[:1024]).cuda(), torch.as_tensor(perm[1024:1124]).cuda()
    d_big = torch.randn(1024, dims[-1], generator=gen, device="cuda") / 1024
    d_small = torch.randn(100, dims[-1], generator=gen, device="cuda") / 100
    plan, grad = _fresh_plan(dims, fanouts, mode_name)
    bridge_step(plan, big, 0, d_big)
    la = bridge_step(plan, small, 5, d_small)
    fresh, fgrad = _fresh_plan(dims, fanouts, mode_name)
    lb = bridge_step(fresh, small, 5, d_small)
    assert torch.equal(la, lb), mode_name + ": logits depend on the earlier step"
    assert bool(torch.isfinite(grad).all())
    assert torch.equal(grad, fgrad), mode_name + ": gradients depend on the earlier step (%d differ)" % int((grad != fgrad).sum())
