"""Thin object layer over the C ABI: device memory stays in torch tensors, every call is
ordered on torch's current CUDA stream.  Nothing here computes: it only marshals pointers."""
import ctypes as C
import numpy as np
import torch

from ._lib import lib, check, PlanConfig, OGL_F32, OGL_BF16, OGL_TF32, OGL_FP16, kernel_launches  # noqa: F401


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    if t is None:
        return None
    assert t.is_contiguous(), "ogl_b200: tensors crossing the C ABI must be contiguous"
    return C.c_void_p(t.data_ptr())


def _dev(t, dtype):
    """torch CUDA tensor of `dtype` from a tensor / ndarray / list (H2D copy if needed)."""
    if isinstance(t, torch.Tensor):
        return t.to(device="cuda", dtype=dtype).contiguous()
    return torch.as_tensor(np.ascontiguousarray(t), dtype=dtype).cuda()


class _CAI:
    def __init__(self, ptr, shape, typestr, strides):
        self.__cuda_array_interface__ = dict(shape=tuple(shape), typestr=typestr, data=(int(ptr), False), version=2,
                                             strides=strides)


_TYPESTR = {torch.float32: ("<f4", 4), torch.int32: ("<i4", 4), torch.int64: ("<i8", 8), torch.uint8: ("|u1", 1),
            torch.float64: ("<f8", 8), torch.bfloat16: ("<i2", 2), torch.float16: ("<f2", 2)}


def wrap_device(ptr, shape, dtype, pitch=None):
    """Zero-copy torch view of library-owned device memory ([rows, cols] with row pitch in elements)."""
    ts, es = _TYPESTR[dtype]
    if len(shape) == 2 and pitch is not None and pitch != shape[1]:
        strides = (pitch * es, es)
    else:
        strides = None
    if any(int(s) == 0 for s in shape):
        return torch.empty(tuple(shape), dtype=dtype, device="cuda")
    t = torch.as_tensor(_CAI(ptr, shape, ts, strides), device="cuda")
    return t.view(torch.bfloat16) if dtype == torch.bfloat16 else t


class Graph:
    """ogl_graph handle: streaming in-edge CSR."""

    def __init__(self, v_cap, e_cap_directed):
        self._h = C.c_void_p()
        check(lib.ogl_graph_create(C.byref(self._h), int(v_cap), int(e_cap_directed)))
        self.v_cap = int(v_cap)

    def __del__(self):
        # (at interpreter shutdown the module globals may already be gone: nothing left to free then)
        if getattr(self, "_h", None) and self._h.value and lib is not None and C is not None:
            lib.ogl_graph_destroy(self._h)
            self._h = C.c_void_p()

    def insert_vertices(self, n):
        check(lib.ogl_graph_insert_vertices(self._h, int(n), _stream()))

    def insert_edges(self, src, dst, symmetric=True):
        """src/dst: CUDA int64 tensors (device path) or host arrays / CPU tensors (host path: the
        H2D copy happens inside the call)."""
        if isinstance(src, torch.Tensor) and src.is_cuda:
            s, d = src.to(torch.int64).contiguous(), dst.to(torch.int64).contiguous()
            check(lib.ogl_graph_insert_edges(self._h, _ptr(s), _ptr(d), s.numel(), int(symmetric), _stream()))
            return
        if isinstance(src, torch.Tensor):
            s, d = src.to(torch.int64).contiguous(), dst.to(torch.int64).contiguous()
            ps, pd, n = C.c_void_p(s.data_ptr()), C.c_void_p(d.data_ptr()), s.numel()
        else:
            s = np.ascontiguousarray(src, dtype=np.int64)
            d = np.ascontiguousarray(dst, dtype=np.int64)
            ps, pd, n = C.c_void_p(s.ctypes.data), C.c_void_p(d.ctypes.data), s.size
        check(lib.ogl_graph_insert_edges_host(self._h, ps, pd, int(n), int(symmetric), _stream()))
        torch.cuda.current_stream().synchronize()   # host buffers may be released by the caller

    def set_source_bound(self, n_sources):
        """accept source ids in [0, n_sources): a destination-range shard stores global source ids in its local rows"""
        check(lib.ogl_graph_set_source_bound(self._h, int(n_sources)))

    def load_parent(self, indptr, indices, eids):
        ip, ix, ei = _dev(indptr, torch.int64), _dev(indices, torch.int64), _dev(eids, torch.int64)
        check(lib.ogl_graph_load_parent(self._h, _ptr(ip), _ptr(ix), _ptr(ei), ip.numel() - 1, _stream()))
        torch.cuda.current_stream().synchronize()

    def set_active_prefix(self, n_active):
        check(lib.ogl_graph_set_active_prefix(self._h, int(n_active), _stream()))

    @property
    def num_vertices(self):
        v = C.c_int64()
        check(lib.ogl_graph_num_vertices(self._h, C.byref(v)))
        return v.value

    @property
    def num_edges(self):
        v = C.c_int64()
        check(lib.ogl_graph_num_edges(self._h, C.byref(v)))
        return v.value

    def degrees(self):
        out = torch.empty(self.num_vertices, dtype=torch.int64, device="cuda")
        check(lib.ogl_graph_degrees(self._h, _ptr(out), _stream()))
        return out

    def export_csr(self, with_eids=True):
        V, E = self.num_vertices, self.num_edges
        indptr = torch.empty(V + 1, dtype=torch.int64, device="cuda")
        indices = torch.empty(E, dtype=torch.int64, device="cuda")
        eids = torch.empty(E, dtype=torch.int64, device="cuda") if with_eids else None
        check(lib.ogl_graph_export_csr(self._h, _ptr(indptr), _ptr(indices), _ptr(eids), _stream()))
        return indptr, indices, eids

    def compact(self):
        check(lib.ogl_graph_compact(self._h, _stream()))

    def row_degrees(self, v):
        """in-degrees of the listed vertices (int64 CUDA tensor)"""
        v = _dev(v, torch.int64)
        out = torch.empty_like(v)
        check(lib.ogl_graph_row_degrees(self._h, _ptr(v), v.numel(), _ptr(out), _stream()))
        return out

    def gather_rows(self, v):
        """(offsets [n + 1], sources) of the in-edge rows of the listed vertices, each row in ascending edge id"""
        v = _dev(v, torch.int64)
        deg = self.row_degrees(v)
        offsets = torch.zeros(v.numel() + 1, dtype=torch.int64, device="cuda")
        torch.cumsum(deg, 0, out=offsets[1:])
        total = int(offsets[-1].item()) if v.numel() else 0
        src = torch.empty(total, dtype=torch.int64, device="cuda")
        if total:
            check(lib.ogl_graph_gather_rows(self._h, _ptr(v), v.numel(), _ptr(offsets), _ptr(src), _stream()))
        return offsets, src

    def segment_max(self, x, rows=None, cols=None):
        """out[r] = max over the in-edges (u -> v_r) of x[u, :cols] (0 for a vertex without in-edges), v_r = rows[r] or r for every
        vertex; x: CUDA fp32 / bf16 / fp16 [*, ld] with a row per vertex and unit column stride.  -> [n_rows, cols] of x's dtype"""
        mode = {torch.float32: OGL_F32, torch.bfloat16: OGL_BF16, torch.float16: OGL_FP16}[x.dtype]
        assert x.is_cuda and x.dim() == 2 and x.stride(1) == 1
        cols = x.shape[1] if cols is None else int(cols)
        nv = 4 if x.dtype == torch.float32 else 8
        r = None if rows is None else _dev(rows, torch.int64)
        n = self.num_vertices if r is None else r.numel()
        out = torch.empty(n, (cols + nv - 1) // nv * nv, dtype=x.dtype, device="cuda")
        check(lib.ogl_graph_segment_max(self._h, mode, C.c_void_p(x.data_ptr()), x.stride(0), cols, _ptr(r), n, _ptr(out), out.shape[1],
                                        _stream()))
        return out[:, :cols]

    def in_frontier(self, rows):
        """the in-neighbourhood frontier of the vertex ids `rows`: (ids, cost), ids = the distinct vertices of rows and of the sources
        of their in-edges, ascending (CUDA int64), cost = sum over them of (in-degree + 1).  Ids outside the graph are ignored."""
        r = _dev(rows, torch.int64)
        out = torch.empty(max(self.num_vertices, 1), dtype=torch.int32, device="cuda")
        n, cost = C.c_int64(), C.c_int64()
        check(lib.ogl_graph_in_frontier(self._h, _ptr(r), r.numel(), _ptr(out), C.byref(n), C.byref(cost), _stream()))
        return out[:n.value].to(torch.int64), cost.value

    def stats(self):
        a = (C.c_int64 * 4)()
        check(lib.ogl_graph_stats(self._h, C.byref(a)))
        return dict(pool_used=a[0], pool_cap=a[1], relocations=a[2], compactions=a[3])


class Features:
    """ogl_features handle: padded feature rows in the arithmetic mode + int32 labels."""

    def __init__(self, v_cap, n_feats, mode):
        self._h = C.c_void_p()
        check(lib.ogl_features_create(C.byref(self._h), int(v_cap), int(n_feats), int(mode)))
        self.v_cap, self.n_feats, self.mode = int(v_cap), int(n_feats), int(mode)

    def __del__(self):
        # (at interpreter shutdown the module globals may already be gone: nothing left to free then)
        if getattr(self, "_h", None) and self._h.value and lib is not None and C is not None:
            lib.ogl_features_destroy(self._h)
            self._h = C.c_void_p()

    def write(self, row0, feats, labels):
        """feats fp32 [n, F], labels int64 [n] (or [n,1]); CUDA tensors or host tensors/arrays."""
        on_host = not (isinstance(feats if feats is not None else labels, torch.Tensor) and
                       (feats if feats is not None else labels).is_cuda)
        if on_host:
            f = None if feats is None else torch.as_tensor(feats, dtype=torch.float32).contiguous()
            l = None if labels is None else torch.as_tensor(labels, dtype=torch.int64).reshape(-1).contiguous()
        else:
            f = None if feats is None else feats.to(torch.float32).contiguous()
            l = None if labels is None else labels.to(torch.int64).reshape(-1).contiguous()
        n = f.shape[0] if f is not None else l.numel()
        check(lib.ogl_features_write(self._h, int(row0), int(n), _ptr(f), _ptr(l), int(on_host), _stream()))
        if on_host:
            torch.cuda.current_stream().synchronize()

    def write_permuted(self, feats_dev, labels_dev, src_rows_dev):
        f = feats_dev.to(torch.float32).contiguous()
        l = labels_dev.to(torch.int64).reshape(-1).contiguous()
        r = src_rows_dev.to(torch.int64).contiguous()
        check(lib.ogl_features_write_permuted(self._h, r.numel(), _ptr(f), _ptr(l), _ptr(r), _stream()))


class Plan:
    """ogl_plan handle: sampler + L-layer GraphSAGE-pool + Adam over one workspace."""

    def __init__(self, dims, fanouts, max_seeds, v_cap, mode=OGL_BF16, seed=0, lr=1e-3, betas=(0.9, 0.999), eps=1e-8,
                 gemm_impl=0, feat_drop=0.0):
        L = len(fanouts)
        assert len(dims) == L + 1
        cfg = PlanConfig()
        cfg.n_layers = L
        for i, d in enumerate(dims):
            cfg.dims[i] = int(d)
        for i, f in enumerate(fanouts):
            cfg.fanouts[i] = int(f)
        cfg.max_seeds, cfg.v_cap, cfg.mode, cfg.gemm_impl, cfg.seed = int(max_seeds), int(v_cap), int(mode), int(gemm_impl), int(seed)
        cfg.lr, cfg.beta1, cfg.beta2, cfg.eps = lr, betas[0], betas[1], eps
        cfg.feat_drop = float(feat_drop or 0.0)
        self._h = C.c_void_p()
        check(lib.ogl_plan_create(C.byref(self._h), C.byref(cfg)))
        self.dims, self.fanouts, self.L = list(dims), list(fanouts), L
        self.max_seeds, self.v_cap, self.mode = int(max_seeds), int(v_cap), int(mode)
        self.dtype = {OGL_BF16: torch.bfloat16, OGL_FP16: torch.float16}.get(mode, torch.float32)
        self.n_params = int(lib.ogl_plan_param_count(self._h))
        self._params = self._grads = None
        self.n_seeds = 0
        self._stamp = 0
        self._forwards = 0
        self._version = 0

    def __del__(self):
        # (at interpreter shutdown the module globals may already be gone: nothing left to free then)
        if getattr(self, "_h", None) and self._h.value and lib is not None and C is not None:
            lib.ogl_plan_destroy(self._h)
            self._h = C.c_void_p()

    # -- parameters ---------------------------------------------------------------------------
    def bind_params(self, flat_params, flat_grads):
        assert flat_params.is_cuda and flat_params.dtype == torch.float32 and flat_params.numel() == self.n_params
        assert flat_grads.is_cuda and flat_grads.dtype == torch.float32 and flat_grads.numel() == self.n_params
        self._params, self._grads = flat_params, flat_grads      # keep alive
        check(lib.ogl_plan_bind_params(self._h, _ptr(flat_params), _ptr(flat_grads), _stream()))

    def refresh_params(self):
        check(lib.ogl_plan_refresh_params(self._h, _stream()))

    def set_step(self, step):
        check(lib.ogl_plan_set_step(self._h, int(step) & 0xFFFFFFFF, _stream()))

    # -- minibatch ----------------------------------------------------------------------------
    def sample(self, graph, seeds_dev):
        s = seeds_dev.to(device="cuda", dtype=torch.int64).contiguous()
        check(lib.ogl_plan_sample(self._h, graph._h, _ptr(s), s.numel(), _stream()))
        self.n_seeds = s.numel()
        self._stamp += 1

    def forward(self, features, want_logits=True):
        out = torch.empty(self.n_seeds, self.dims[-1], dtype=torch.float32, device="cuda") if want_logits else None
        check(lib.ogl_plan_forward(self._h, features._h if features is not None else None, _ptr(out), _stream()))
        self._forwards += 1              # the activations a backward pass differentiates are this forward's now
        return out

    def set_input(self, x):
        x = x.to(device="cuda", dtype=torch.float32).contiguous()
        check(lib.ogl_plan_set_input(self._h, _ptr(x), x.shape[0], _stream()))

    def loss_backward(self, features, loss_scale, want_per_vertex=True):
        per = torch.empty(self.n_seeds, dtype=torch.float32, device="cuda") if want_per_vertex else None
        tot = torch.empty(1, dtype=torch.float32, device="cuda")
        check(lib.ogl_plan_loss_backward(self._h, features._h, float(loss_scale), _ptr(per), _ptr(tot), _stream()))
        return per, tot

    def backward(self, dlogits, amax=None):
        """back-propagate caller-computed fp32 dlogits [n_seeds, C] through the last forward.  amax = max |dlogits|, which mode
        OGL_FP16 needs for its gradient scale: read from the device (one synchronisation) when not given; other modes ignore it"""
        d = dlogits.to(device="cuda", dtype=torch.float32).contiguous()
        if amax is None:
            amax = float(d.abs().amax()) if self.mode == OGL_FP16 and d.numel() else 0.0
        check(lib.ogl_plan_backward(self._h, _ptr(d), float(amax), _stream()))

    def adam_step(self):
        check(lib.ogl_plan_adam_step(self._h, _stream()))

    def peer_adam(self, peer, lo, hi, last, reduced_out=None):
        """data-parallel Adam: gradients [lo, hi) summed over the ranks through peer memory inside the Adam kernel"""
        check(lib.ogl_plan_peer_adam(self._h, peer._h, int(lo), int(hi), int(last), _ptr(reduced_out), _stream()))

    def train_step(self, graph, features, seeds, loss_scale=None, do_step=True, per_vertex_out=None, loss_sum_out=None):
        """seeds: CUDA int64 tensor (device path) or pinned/pageable CPU int64 tensor (host path)."""
        n = seeds.numel()
        on_host = not seeds.is_cuda
        assert seeds.dtype == torch.int64 and seeds.is_contiguous()
        if loss_scale is None:
            loss_scale = 1.0 / n
        check(lib.ogl_plan_train_step(self._h, graph._h, features._h, C.c_void_p(seeds.data_ptr()), n, int(on_host),
                                      float(loss_scale), int(do_step), _ptr(per_vertex_out), _ptr(loss_sum_out), _stream()))
        self.n_seeds = n
        self._stamp += 1

    def train_steps(self, graph, features, seeds, batch, loss_scale=None, do_step=True, per_vertex_out=None, loss_sums_out=None):
        """seeds: flat int64 tensor of n_batches * batch ids (CUDA or pinned/pageable CPU); all steps in one C call"""
        n = seeds.numel()
        assert seeds.dtype == torch.int64 and seeds.is_contiguous() and n % batch == 0
        if loss_scale is None:
            loss_scale = 1.0 / batch
        check(lib.ogl_plan_train_steps(self._h, graph._h, features._h, C.c_void_p(seeds.data_ptr()), n // batch, int(batch),
                                       int(not seeds.is_cuda), float(loss_scale), int(do_step), _ptr(per_vertex_out), _ptr(loss_sums_out),
                                       _stream()))
        self.n_seeds = batch
        self._stamp += 1

    def step_begin(self, graph, features, seeds):
        """sample + gather of the next minibatch (no weights involved)"""
        n = seeds.numel()
        assert seeds.dtype == torch.int64 and seeds.is_contiguous()
        check(lib.ogl_plan_step_begin(self._h, graph._h, features._h, C.c_void_p(seeds.data_ptr()), n, int(not seeds.is_cuda), _stream()))
        self.n_seeds = n
        self._stamp += 1

    def prefetch(self, graph, features, seeds):
        """sample + gather of a FUTURE minibatch on the plan's own stream / second buffer set (the role of NodeDataLoader's
        workers): it overlaps whatever train step is running.  The next train_step / step_finish consumes the oldest pending
        minibatch.  Order for full overlap: prefetch(0); for i: prefetch(i+1); train_step(i)"""
        n = seeds.numel()
        assert seeds.dtype == torch.int64 and seeds.is_contiguous()
        check(lib.ogl_plan_prefetch(self._h, graph._h, features._h, C.c_void_p(seeds.data_ptr()), n, int(not seeds.is_cuda), _stream()))
        self._prefetch_refs = (getattr(self, "_prefetch_refs", ()) + (seeds,))[-3:]      # seeds stay alive until consumed
        self._stamp += 1

    @property
    def prefetch_pending(self):
        return int(lib.ogl_plan_prefetch_pending(self._h))

    def step_finish(self, features, loss_scale, do_step=True, per_vertex_out=None, loss_sum_out=None):
        """forward + loss + backward (+ Adam) over the minibatch begun with step_begin"""
        check(lib.ogl_plan_step_finish(self._h, features._h, float(loss_scale), int(do_step), _ptr(per_vertex_out), _ptr(loss_sum_out),
                                       _stream()))

    def step_finish_dp(self, peer, features, loss_scale, per_vertex_out=None, loss_sum_out=None):
        """data-parallel finish in one launch sequence: forward .. backward + the peer-memory gradient exchange + Adam"""
        check(lib.ogl_plan_step_finish_dp(self._h, peer._h, features._h, float(loss_scale), _ptr(per_vertex_out), _ptr(loss_sum_out), _stream()))

    def step_finish_head(self, features, loss_scale, per_vertex_out=None, loss_sum_out=None):
        """forward + loss + backward except the last weight-gradient GEMM (layer 0 fc_pool.weight)"""
        check(lib.ogl_plan_step_finish_head(self._h, features._h, float(loss_scale), _ptr(per_vertex_out), _ptr(loss_sum_out), _stream()))

    def step_finish_tail(self, features):
        """the last weight-gradient GEMM (layer 0 fc_pool.weight)"""
        check(lib.ogl_plan_step_finish_tail(self._h, features._h, _stream()))

    @property
    def tail_params(self):
        """number of leading floats of the flat gradient buffer that step_finish_tail produces (layer 0 fc_pool.weight)"""
        return self.dims[0] * self.dims[0]

    def eval_step(self, graph, features, seeds, logits_out=None, per_vertex_out=None):
        n = seeds.numel()
        on_host = not seeds.is_cuda
        assert seeds.dtype == torch.int64 and seeds.is_contiguous()
        check(lib.ogl_plan_eval_step(self._h, graph._h, features._h, C.c_void_p(seeds.data_ptr()), n, int(on_host),
                                     _ptr(logits_out), _ptr(per_vertex_out), _stream()))
        self.n_seeds = n
        self._stamp += 1

    def infer_full(self, graph, features, seeds=None, logits_out=None):
        """logits [n, C] fp32 of every listed vertex (seeds: int64 ids; None: every vertex of `graph`, in id order) from its WHOLE
        in-neighbourhood, layer by layer over all vertices, no sampling; changes no plan state.  Out-of-range ids raise bit 0 of
        error_flags()."""
        s = None if seeds is None else _dev(seeds, torch.int64)
        n = graph.num_vertices if s is None else s.numel()
        out = logits_out
        if out is None:
            out = torch.empty(n, self.dims[-1], dtype=torch.float32, device="cuda")
        assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and tuple(out.shape) == (n, self.dims[-1])
        check(lib.ogl_plan_infer_full(self._h, graph._h, features._h, _ptr(s), n, _ptr(out), _stream()))
        return out

    def infer_full_loss(self, graph, features, seeds=None, logits_out=None, loss_out=None):
        """infer_full followed by the per-vertex cross entropy on its logits: fp32 losses [n] (logsumexp(logits) - logits[label]), the
        training loss's arithmetic, so equal logits give bit-equal losses.  logits_out [n, C] (optional) receives the logits, bit-equal
        to infer_full's.  Changes no plan state; an out-of-range id raises bit 0 of error_flags() (vertex 0 is scored instead), a
        label outside [0, C) gives NaN and raises bit 1."""
        s = None if seeds is None else _dev(seeds, torch.int64)
        n = graph.num_vertices if s is None else s.numel()
        if logits_out is not None:
            assert logits_out.is_cuda and logits_out.dtype == torch.float32 and logits_out.is_contiguous() and \
                tuple(logits_out.shape) == (n, self.dims[-1])
        out = loss_out if loss_out is not None else torch.empty(n, dtype=torch.float32, device="cuda")
        assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and tuple(out.shape) == (n,)
        if n:                                  # (an empty id list has no device pointer: NULL would mean "every vertex")
            check(lib.ogl_plan_infer_full_loss(self._h, graph._h, features._h, _ptr(s), n, _ptr(logits_out), _ptr(out), _stream()))
        return out

    def full_xent(self, features, logits, rows=None, row0=0, out=None):
        """the loss of infer_full_loss on its own: fp32 losses [n] of the fp32 logits [n, >= C] (unit column stride, any row pitch)
        whose row r belongs to vertex rows[r] (int64 ids) or row0 + r.  Ordered on the stream, no synchronisation."""
        assert logits.is_cuda and logits.dtype == torch.float32 and logits.dim() == 2 and logits.stride(1) == 1 and \
            logits.shape[1] >= self.dims[-1], "full_xent: logits must be fp32 [n, >= %d] with unit column stride" % self.dims[-1]
        n = logits.shape[0]
        r = None if rows is None else _dev(rows, torch.int64)
        assert r is None or tuple(r.shape) == (n,), "full_xent: one vertex id per logits row"
        if out is None:
            out = torch.empty(n, dtype=torch.float32, device="cuda")
        assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and tuple(out.shape) == (n,)
        check(lib.ogl_plan_full_xent(self._h, features._h, C.c_void_p(logits.data_ptr()) if n else None, logits.stride(0),
                                     _ptr(r), int(row0), n, _ptr(out), _stream()))
        return out

    def hidden_table(self, layer, rows):
        """a [round_up(rows, 128), pitch] table in the plan's storage dtype for the output of hidden `layer` (the input `h` of layer
        + 1 of infer_full_layer); pitch = round_up(width, 8)"""
        assert 0 <= layer < self.L - 1, "layer %d has no hidden output (the model has %d layers)" % (layer, self.L)
        return torch.empty((int(rows) + 127) // 128 * 128, (self.dims[layer + 1] + 7) // 8 * 8, dtype=self.dtype, device="cuda")

    def infer_full_layer(self, graph, features, layer, h, rows=None, row0=0, n=None, out=None):
        """layer `layer` of infer_full for the destination rows `rows` (int64 ids) or [row0, row0 + n) (n None: to the last vertex):
        the pool GEMM over every vertex of h (a hidden_table(layer - 1, V) holding the previous layer's output for every vertex;
        unused for layer 0, which reads `features`), the segment max and the output GEMM over the listed rows.  -> out[:n]: the
        hidden rows (a hidden_table(layer, n) or a row slice of one) or, for the last layer, fp32 logits [n, C].  Every row is
        computed on its own, so a split of the rows gives the bits of the one call over all of them."""
        r = None if rows is None else _dev(rows, torch.int64)
        if r is not None:
            n = r.numel()
        elif n is None:
            n = graph.num_vertices - int(row0)
        last = layer == self.L - 1
        if out is None:
            out = (torch.empty(n, self.dims[-1], dtype=torch.float32, device="cuda") if last
                   else self.hidden_table(layer, n))
        assert out.is_cuda and out.dim() == 2 and out.stride(1) == 1 and out.shape[0] >= n
        assert out.dtype == (torch.float32 if last else self.dtype)
        hp, ldh = None, 0
        if h is not None:
            assert h.is_cuda and h.dim() == 2 and h.stride(1) == 1 and h.dtype == self.dtype
            hp, ldh = C.c_void_p(h.data_ptr()), h.stride(0)
        check(lib.ogl_plan_infer_full_layer(self._h, graph._h, features._h, int(layer), hp, ldh, _ptr(r), int(row0), int(n),
                                            C.c_void_p(out.data_ptr()), out.stride(0), _stream()))
        return out[:n]

    def reset_optimizer(self, philox_step=0):
        """zero Adam's moments / step counter and set the Philox step (a fresh optimiser; replays of a run from its start)"""
        check(lib.ogl_plan_reset_optimizer(self._h, int(philox_step) & 0xFFFFFFFF, _stream()))

    def error_flags(self):
        """sticky device error bits since the last call (bit 0: out-of-range seed id; bit 1: a full-inference loss met a label outside
        [0, C)); synchronises"""
        v = C.c_uint32()
        check(lib.ogl_plan_error_flags(self._h, C.byref(v)))
        return int(v.value)

    def set_option(self, name, value):
        check(lib.ogl_plan_set_option(self._h, name.encode(), int(value)))

    def graph_stats(self):
        a = (C.c_int64 * 2)()
        check(lib.ogl_plan_graph_stats(self._h, C.byref(a)))
        return dict(captures=a[0], replays=a[1])

    # -- stage profiling (bench.py) ---------------------------------------------------------------
    def profile(self, enable=True):
        check(lib.ogl_plan_profile(self._h, int(bool(enable))))

    def profile_read(self):
        """-> (dict stage -> (ms_total, launches_total), level_count_sums[L+1], n_steps)"""
        names = C.create_string_buffer(8192)
        ms = (C.c_float * 256)()
        ln = (C.c_int64 * 256)()
        n, steps = C.c_int(), C.c_int()
        sums = (C.c_int64 * 8)()
        check(lib.ogl_plan_profile_read(self._h, names, 8192, C.cast(ms, C.c_void_p), C.cast(ln, C.c_void_p), 256, C.byref(n),
                                        C.cast(sums, C.c_void_p), C.byref(steps)))
        keys = names.value.decode().split("\n")[:n.value]
        return {k: (float(ms[i]), int(ln[i])) for i, k in enumerate(keys)}, [int(sums[i]) for i in range(self.L + 1)], steps.value

    # -- introspection (parity tests, DGL-style block objects) ---------------------------------
    def level_nodes(self, level):
        p, c, m = C.c_void_p(), C.c_void_p(), C.c_int()
        check(lib.ogl_plan_level_nodes(self._h, level, C.byref(p), C.byref(c), C.byref(m)))
        n = int(wrap_device(c.value, (1,), torch.int32).item())
        return wrap_device(p.value, (n,), torch.int32)

    def block_edges(self, hop):
        a, b, e, f = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_int()
        check(lib.ogl_plan_block_edges(self._h, hop, C.byref(a), C.byref(b), C.byref(e), C.byref(f)))
        n_dst = self.level_nodes(hop).numel()
        ne = n_dst * f.value
        return (wrap_device(a.value, (ne,), torch.int32), wrap_device(b.value, (ne,), torch.int32),
                wrap_device(e.value, (ne,), torch.int64), f.value)

    def tensor(self, name, rows=None):
        p, r, pt, eb = C.c_void_p(), C.c_int(), C.c_int(), C.c_int()
        check(lib.ogl_plan_tensor(self._h, name.encode(), C.byref(p), C.byref(r), C.byref(pt), C.byref(eb)))
        dt = {1: torch.uint8, 2: self.dtype, 4: torch.float32}[eb.value]
        return wrap_device(p.value, (rows if rows is not None else r.value, pt.value), dt)


class Peer:
    """ogl_peer handle: one rank's end of the NVLink peer-memory gradient exchange (csrc/peer.cu).  `grads` is the rank's gradient
    buffer (library-owned, mapped by the peers): bind it as the plan's gradient buffer."""

    def __init__(self, rank, world, n_floats):
        self._h = C.c_void_p()
        check(lib.ogl_peer_create(C.byref(self._h), int(rank), int(world), int(n_floats)))
        self.rank, self.world, self.n_floats = int(rank), int(world), int(n_floats)
        p = C.c_void_p()
        check(lib.ogl_peer_buffer(self._h, C.byref(p)))
        self.grads = wrap_device(p.value, (self.n_floats,), torch.float32)

    def __del__(self):
        # (at interpreter shutdown the module globals may already be gone: nothing left to free then)
        if getattr(self, "_h", None) and self._h.value and lib is not None and C is not None:
            lib.ogl_peer_destroy(self._h)
            self._h = C.c_void_p()

    def handle(self):
        buf = C.create_string_buffer(64)
        check(lib.ogl_peer_handle(self._h, buf))
        return buf.raw

    def connect(self, handles):
        """handles: the 64-byte handles of all ranks, rank order (bytes of length 64 * world)"""
        assert len(handles) == 64 * self.world
        check(lib.ogl_peer_connect(self._h, C.c_char_p(handles)))

    @staticmethod
    def connect_local(peers):
        """wire up peers that live in one process (tests: several ranks on one GPU)"""
        arr = (C.c_void_p * len(peers))(*[p._h.value for p in peers])
        for p in peers:
            check(lib.ogl_peer_connect_local(p._h, arr))

    def wait_readers(self):
        """enqueue: wait until every peer has finished reading this rank's gradients of the previous exchange"""
        check(lib.ogl_peer_wait_readers(self._h, _stream()))


class SumTree:
    """ogl_sumtree handle: fp64 sum tree."""

    def __init__(self, capacity):
        self._h = C.c_void_p()
        check(lib.ogl_sumtree_create(C.byref(self._h), int(capacity)))
        self.capacity = int(capacity)

    def __del__(self):
        # (at interpreter shutdown the module globals may already be gone: nothing left to free then)
        if getattr(self, "_h", None) and self._h.value and lib is not None and C is not None:
            lib.ogl_sumtree_destroy(self._h)
            self._h = C.c_void_p()

    def set(self, idx, val):
        i, v = _dev(idx, torch.int64), _dev(val, torch.float64)
        check(lib.ogl_sumtree_set(self._h, _ptr(i), _ptr(v), i.numel(), _stream()))

    def set_from_loss(self, idx, loss, clip_lo, clip_hi, eps, alpha, minmax_state):
        i, l = _dev(idx, torch.int64), _dev(loss, torch.float32)
        check(lib.ogl_sumtree_set_from_loss(self._h, _ptr(i), _ptr(l), i.numel(), clip_lo, clip_hi, eps, alpha,
                                            _ptr(minmax_state), _stream()))

    def sum(self, lo=0, hi=None):
        out = torch.empty(1, dtype=torch.float64, device="cuda")
        check(lib.ogl_sumtree_sum(self._h, int(lo), int(self.capacity if hi is None else hi), _ptr(out), _stream()))
        return out

    def find(self, mass):
        m = _dev(mass, torch.float64)
        out = torch.empty(m.numel(), dtype=torch.int64, device="cuda")
        check(lib.ogl_sumtree_find(self._h, _ptr(m), m.numel(), _ptr(out), _stream()))
        return out

    def sample_stratified(self, uniforms, n_items):
        u = _dev(uniforms, torch.float64)
        out = torch.empty(u.numel(), dtype=torch.int64, device="cuda")
        check(lib.ogl_sumtree_sample_stratified(self._h, _ptr(u), u.numel(), int(n_items), _ptr(out), _stream()))
        return out

    def values(self):
        p, c = C.c_void_p(), C.c_int64()
        check(lib.ogl_sumtree_values(self._h, C.byref(p), C.byref(c)))
        return wrap_device(p.value, (2 * c.value,), torch.float64)


def draw_uniform(n_pop, n, seed, counter):
    out = torch.empty(int(n), dtype=torch.int64, device="cuda")
    check(lib.ogl_draw_uniform(int(n_pop), int(n), int(seed) & 0xFFFFFFFFFFFFFFFF, int(counter) & 0xFFFFFFFF, _ptr(out), _stream()))
    return out


def sample_neighbors(graph, dst, fanout, seed, step, hop, want_eids=True):
    d = _dev(dst, torch.int64)
    src = torch.empty(d.numel() * fanout, dtype=torch.int32, device="cuda")
    eid = torch.empty(d.numel() * fanout, dtype=torch.int64, device="cuda") if want_eids else None
    check(lib.ogl_sample_neighbors(graph._h, _ptr(d), d.numel(), int(fanout), int(seed) & 0xFFFFFFFFFFFFFFFF, int(step), int(hop),
                                   _ptr(src), _ptr(eid), _stream()))
    return src, eid


def rows_linear(x1, ids1, w1, b1, out, out_ids, relu=False, x2=None, ids2=None, w2=None, b2=None):
    """out[out_ids[i]] = act(x1[ids1[i]] @ w1.T + b1 (+ x2[ids2[i]] @ w2.T + b2)); fp32, torch.nn.Linear weight layout [n_out, k]"""
    for t in (x1, w1, out) + ((x2, w2) if x2 is not None else ()):
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
    n = ids1.numel()
    check(lib.ogl_infer_rows_linear(_ptr(x1), x1.shape[1], _ptr(ids1), _ptr(w1), w1.shape[1], _ptr(b1),
                                    _ptr(x2), x2.shape[1] if x2 is not None else 0, _ptr(ids2), _ptr(w2), w2.shape[1] if w2 is not None else 0,
                                    _ptr(b2), int(relu), _ptr(out), out.shape[1], _ptr(out_ids), n, w1.shape[0], _stream()))


def infer_query(graph, v, v_off, th, cap_in, cap_out, out):
    """one-launch neighbourhood query (csrc/infer.cu: k_infer_query); `out`: int64 CUDA scratch of 5 + 3 n + cap_in + 2 cap_out"""
    check(lib.ogl_infer_query(graph._h, _ptr(v), v.numel(), int(v_off), int(th), int(cap_in), int(cap_out), _ptr(out), _stream()))


def induced_mean(graph, member, nodes, proj, out):
    """out[v] = mean of proj[u] over the in-edges u -> v of `graph` with member[u] != 0 (0 without one), for v in nodes"""
    assert member.dtype == torch.uint8 and proj.dtype == torch.float32 and out.dtype == torch.float32
    check(lib.ogl_infer_induced_mean(graph._h, _ptr(member), _ptr(nodes), nodes.numel(), _ptr(proj), proj.shape[1], proj.shape[1],
                                     _ptr(out), out.shape[1], _stream()))


def gemm_bf16_nt(a, b, k=None):
    """C[M,N] fp32 = A[M,:k] bf16 @ B[N,:k]^T bf16 on the tcgen05 path (tests / bench); row pitches = shape[1]."""
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.is_cuda and b.is_cuda
    a, b = a.contiguous(), b.contiguous()
    k = a.shape[1] if k is None else int(k)
    ldc = (b.shape[0] + 7) // 8 * 8
    c = torch.empty(a.shape[0], ldc, dtype=torch.float32, device="cuda")
    check(lib.ogl_gemm_bf16_nt(_ptr(a), a.shape[1], _ptr(b), b.shape[1], _ptr(c), ldc, a.shape[0], b.shape[0], k, _stream()))
    return c[:, :b.shape[0]]


def gemm_bf16_tn(a, b, n=None, k=None, workspace_elems=1 << 24):
    """C[N,K] fp32 = A[M,:n]^T bf16 @ B[M,:k] bf16 on the tcgen05 path (tests / bench); row pitches = shape[1]."""
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.is_cuda and b.is_cuda and a.shape[0] == b.shape[0]
    a, b = a.contiguous(), b.contiguous()
    n = a.shape[1] if n is None else int(n)
    k = b.shape[1] if k is None else int(k)
    c = torch.empty(n, k, dtype=torch.float32, device="cuda")
    ws = torch.empty(workspace_elems, dtype=torch.float32, device="cuda") if workspace_elems else None
    check(lib.ogl_gemm_bf16_tn(_ptr(a), a.shape[1], _ptr(b), b.shape[1], _ptr(c), k, a.shape[0], n, k,
                               _ptr(ws), int(workspace_elems), _stream()))
    return c


def gemm_bf16_nt_ex(a, b, k=None, out_bf16=True, bias=None, relu=False, cg=0):
    """C[M,N] = act(A[M,:k] @ B[N,:k]^T + bias) with the plan's fused epilogue (bf16 out -> TMA-store path)."""
    a, b = a.contiguous(), b.contiguous()
    k = a.shape[1] if k is None else int(k)
    ldc = (b.shape[0] + 7) // 8 * 8
    c = torch.empty(a.shape[0], ldc, dtype=torch.bfloat16 if out_bf16 else torch.float32, device="cuda")
    check(lib.ogl_gemm_bf16_nt_ex(_ptr(a), a.shape[1], _ptr(b), b.shape[1], _ptr(c), ldc, a.shape[0], b.shape[0], k, int(out_bf16),
                                  _ptr(bias), int(relu), int(cg), _stream()))
    return c[:, :b.shape[0]]


def round_tf32(x):
    """fp32 tensor rounded to TF32 (10 explicit mantissa bits, round to nearest, ties away from zero = cvt.rna.tf32.f32)"""
    b = x.contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


def gemm_tf32_nt_ex(a, b, k=None, tma_out=True, bias=None, relu=False, mask=None, cg=0):
    """C[M,N] fp32 = act(A[M,:k] @ B[N,:k]^T + bias) on the tcgen05 kind::tf32 path; tma_out: TF32-rounded activation epilogue"""
    assert a.dtype == torch.float32 and b.dtype == torch.float32 and a.is_cuda and b.is_cuda
    a, b = a.contiguous(), b.contiguous()
    k = a.shape[1] if k is None else int(k)
    ldc = (b.shape[0] + 7) // 8 * 8
    c = torch.empty(a.shape[0], ldc, dtype=torch.float32, device="cuda")
    if mask is not None:
        mask = mask.contiguous()
    check(lib.ogl_gemm_tf32_nt_ex(_ptr(a), a.shape[1], _ptr(b), b.shape[1], _ptr(c), ldc, a.shape[0], b.shape[0], k, int(tma_out),
                                  _ptr(bias), int(relu), _ptr(mask), mask.shape[1] if mask is not None else 0, int(cg), _stream()))
    return c[:, :b.shape[0]]


def gemm_tf32_tn(a, b, n=None, k=None, workspace_elems=1 << 24):
    """C[N,K] fp32 = A[M,:n]^T @ B[M,:k] on the tcgen05 kind::tf32 path (MN-major operands)"""
    assert a.dtype == torch.float32 and b.dtype == torch.float32 and a.is_cuda and b.is_cuda and a.shape[0] == b.shape[0]
    a, b = a.contiguous(), b.contiguous()
    n = a.shape[1] if n is None else int(n)
    k = b.shape[1] if k is None else int(k)
    c = torch.empty(n, k, dtype=torch.float32, device="cuda")
    ws = torch.empty(workspace_elems, dtype=torch.float32, device="cuda") if workspace_elems else None
    check(lib.ogl_gemm_tf32_tn(_ptr(a), a.shape[1], _ptr(b), b.shape[1], _ptr(c), k, a.shape[0], n, k,
                               _ptr(ws), int(workspace_elems), _stream()))
    return c


def gemm_f16_nt_ex(a, b, k=None, out_f16=True, bias=None, relu=False, mask=None, cg=0):
    """C[M,N] = act(A[M,:k] @ B[N,:k]^T + bias) on the tcgen05 kind::f16 path with fp16 operands (mode OGL_FP16)"""
    assert a.dtype == torch.float16 and b.dtype == torch.float16 and a.is_cuda and b.is_cuda
    a, b = a.contiguous(), b.contiguous()
    k = a.shape[1] if k is None else int(k)
    ldc = (b.shape[0] + 7) // 8 * 8
    c = torch.empty(a.shape[0], ldc, dtype=torch.float16 if out_f16 else torch.float32, device="cuda")
    if mask is not None:
        mask = mask.contiguous()
        assert mask.dtype == torch.float16
    check(lib.ogl_gemm_f16_nt_ex(_ptr(a), a.shape[1], _ptr(b), b.shape[1], _ptr(c), ldc, a.shape[0], b.shape[0], k, int(out_f16),
                                 _ptr(bias), int(relu), _ptr(mask), mask.shape[1] if mask is not None else 0, int(cg), _stream()))
    return c[:, :b.shape[0]]


def gemm_f16_tn(a, b, n=None, k=None, alpha=1.0, workspace_elems=1 << 24):
    """C[N,K] fp32 = alpha * A[M,:n]^T @ B[M,:k] on the tcgen05 kind::f16 path with fp16 MN-major operands"""
    assert a.dtype == torch.float16 and b.dtype == torch.float16 and a.is_cuda and b.is_cuda and a.shape[0] == b.shape[0]
    a, b = a.contiguous(), b.contiguous()
    n = a.shape[1] if n is None else int(n)
    k = b.shape[1] if k is None else int(k)
    c = torch.empty(n, k, dtype=torch.float32, device="cuda")
    ws = torch.empty(workspace_elems, dtype=torch.float32, device="cuda") if workspace_elems else None
    check(lib.ogl_gemm_f16_tn(_ptr(a), a.shape[1], _ptr(b), b.shape[1], _ptr(c), k, a.shape[0], n, k, float(alpha),
                              _ptr(ws), int(workspace_elems), _stream()))
    return c


def eval_confusion(logits, labels, n_classes=None):
    """int64 [C, C] confusion matrix (rows = label, columns = argmax of the logits, first maximum wins) of CUDA logits [n, C] and
    int64 labels [n], computed on the device; labels outside [0, C) are skipped.  -> (cm CUDA tensor, n_skipped)"""
    assert logits.is_cuda and logits.dtype == torch.float32 and logits.dim() == 2 and logits.stride(1) == 1
    C_ = logits.shape[1] if n_classes is None else int(n_classes)
    lab = labels.to(device="cuda", dtype=torch.int64).reshape(-1).contiguous()
    assert lab.numel() == logits.shape[0]
    cm = torch.zeros(C_ * C_ + 1, dtype=torch.int64, device="cuda")
    check(lib.ogl_eval_confusion(C.c_void_p(logits.data_ptr()), logits.stride(0), logits.shape[0], C_, _ptr(lab), _ptr(cm), _stream()))
    return cm[:C_ * C_].view(C_, C_), cm[C_ * C_]


def macro_f1_from_confusion(cm):
    """(f1_macro, cm restricted to the classes present) exactly as sklearn computes them from (y_true, y_pred): the class set is
    the union of the labels that occur in either; f1_c = 2 tp / (2 tp + fp + fn)"""
    cm = np.asarray(cm, dtype=np.int64)
    present = (cm.sum(0) + cm.sum(1)) > 0
    sub = cm[present][:, present]
    tp = np.diag(sub).astype(np.float64)
    den = sub.sum(0) + sub.sum(1)
    f1 = np.where(den > 0, 2 * tp / np.maximum(den, 1), 0.0)
    return (float(f1.mean()) if len(f1) else 0.0), sub
