"""Test references of the train step's sampled-block memory kernels (csrc/sample.cu, csrc/sage_kernels.cu), one per kernel, for
tests/test_gpu_block_kernels.py.  Each takes the tensors the kernel read (read back from the device, so an arithmetic mode's rounding
in earlier stages cannot hide anything) and computes what the kernel's specification says it writes.  Plain torch: they run on the
device the inputs live on, and on the CPU in tests/test_block_kernels_host.py.

- segmax_ref: k_segmax_fwd.  neigh[d, c] = max over the valid ELL slots j of hp[edge_lid[d, j], c]; the slot kept is the first one
  attaining the maximum (strictly-greater update, +0 == -0); rows without a valid slot give neigh 0 and slot 255.
- reverse_lists_ref: k_rev_count / k_rev_fill / k_rev_sort[_long].  Offsets = exclusive scan of the per-source pick counts; every
  row holds the entries (destination row << 8) | slot of the picks of that source, ascending.
- pool_bwd_ref: k_pool_bwd.  dhp[s, c] = fp32 sum, starting at 0 and sequential in list order, of dng[d, c] over the list entries
  (d, j) of row s with arg[d, c] == j; to_storage then rounds it once to the storage type.
- colsum_ref: k_colsum_partial / k_colsum_final (the bias gradients), in fp64 with the sum of |x| for an error bound.
- xent_ref: k_xent.  fp64 log-softmax of the fp32 logits."""
import numpy as np
import torch

from oracle.sage import round_tf32

MANT = {"fp32": 23, "tf32": 10, "bf16": 7, "fp16": 10}      # explicit mantissa bits of the values each mode stores
BITS = {"fp32": torch.int32, "tf32": torch.int32, "bf16": torch.int16, "fp16": torch.int16}


def to_storage(x, mode):
    """fp32 -> the mode's storage values: RNE to bf16 / fp16 (overflow to inf), TF32 with ties away from zero (cvt.rna)"""
    x = x.to(torch.float32)
    if mode == "bf16":
        return x.to(torch.bfloat16)
    if mode == "fp16":
        return x.to(torch.float16)
    if mode == "tf32":
        return round_tf32(x)
    return x


def storage_ulp(x, mode):
    """one unit in the last place of the stored value nearest |x| (fp16: its subnormal step 2^-24 at the bottom)"""
    a = x.abs().double().clamp(min=2.0 ** -126)
    ulp = torch.exp2(torch.floor(torch.log2(a)) - MANT[mode])
    return ulp.clamp(min=2.0 ** -24) if mode == "fp16" else ulp


def segmax_ref(hp, edge_lid, n_dst, fanout, chunk=4096):
    """-> (neigh fp32 [n_dst, pitch], arg uint8 [n_dst, pitch]) over every column of hp (pad columns included).  hp values are compared
    in fp32, which holds every storage type exactly"""
    pitch, dev = hp.shape[1], hp.device
    lid = edge_lid[:n_dst * fanout].view(n_dst, fanout).long()
    neigh = torch.empty(n_dst, pitch, dtype=torch.float32, device=dev)
    arg = torch.empty(n_dst, pitch, dtype=torch.uint8, device=dev)
    for r0 in range(0, n_dst, chunk):
        ll = lid[r0:r0 + chunk]
        best = torch.full((ll.shape[0], pitch), -float("inf"), dtype=torch.float32, device=dev)
        slot = torch.full((ll.shape[0], pitch), 255, dtype=torch.uint8, device=dev)
        for j in range(fanout):
            x = hp[ll[:, j].clamp(min=0)].float()
            upd = (ll[:, j] >= 0)[:, None] & (x > best)
            best = torch.where(upd, x, best)
            slot = torch.where(upd, torch.full_like(slot, j), slot)
        has = (ll >= 0).any(dim=1)[:, None]
        neigh[r0:r0 + chunk] = torch.where(has, best, torch.zeros_like(best))
        arg[r0:r0 + chunk] = torch.where(has, slot, torch.full_like(slot, 255))
    return neigh, arg


def reverse_lists_ref(edge_lid, n_dst, fanout, n_src_max):
    """-> (rev_ptr int64 [n_src_max + 1], rev_edge int64 [number of valid slots])"""
    lid = edge_lid[:n_dst * fanout].long()
    p = torch.nonzero(lid >= 0).flatten()
    src = lid[p]
    ptr = torch.zeros(n_src_max + 1, dtype=torch.int64, device=lid.device)
    ptr[1:] = torch.cumsum(torch.bincount(src, minlength=n_src_max), 0)
    p = p[torch.sort(src, stable=True).indices]                 # per source, ascending slot position = ascending entry
    return ptr, ((p // fanout) << 8) | (p % fanout)


def naive_reverse_lists(edge_lid, n_dst, fanout, n_src_max):
    """reverse_lists_ref written as the per-source loop it stands for (the host test's check of it)"""
    lid = [int(v) for v in edge_lid[:n_dst * fanout]]
    rows = [[] for _ in range(n_src_max)]
    for d in range(n_dst):
        for j in range(fanout):
            s = lid[d * fanout + j]
            if s >= 0:
                rows[s].append((d << 8) | j)
    ptr = np.zeros(n_src_max + 1, dtype=np.int64)
    ptr[1:] = np.cumsum([len(r) for r in rows])
    return ptr, np.array([e for r in rows for e in sorted(r)], dtype=np.int64)


def pool_bwd_ref(dng, arg, rev_ptr, rev_edge, n_src, acc=torch.float32):
    """-> [n_src, pitch] sums in `acc`.  dng: [n_dst, pitch] (any float type), arg: uint8 [n_dst, pitch].  Vectorised over the rows,
    looping over the list position; once only one row's list goes on, that row is finished sequentially on the host"""
    dev, pitch = dng.device, dng.shape[1]
    ptr = rev_ptr[:n_src + 1].long()
    edge = rev_edge.long()
    lens = ptr[1:] - ptr[:-1]
    out = torch.zeros(n_src, pitch, dtype=acc, device=dev)
    if n_src == 0:
        return out
    order = torch.argsort(lens, descending=True, stable=True)
    lens_sorted = lens[order].cpu()
    ks = torch.arange(int(lens_sorted[0]) if n_src else 0)
    active = (n_src - torch.searchsorted(lens_sorted.flip(0).contiguous(), ks, right=True)).tolist()   # rows with len > k

    def contrib(e):
        d, j = e >> 8, e & 255
        return torch.where(arg[d].long() == j[:, None], dng[d].to(acc), torch.zeros((), dtype=acc, device=dev))

    for k, n_act in enumerate(active):
        if n_act == 1:
            r = int(order[0])
            terms = contrib(edge[int(ptr[r]) + k:int(ptr[r + 1])]).cpu().numpy()
            seq = np.add.accumulate(np.concatenate([out[r:r + 1].cpu().numpy(), terms]), axis=0)     # strictly sequential
            out[r] = torch.from_numpy(seq[-1]).to(dev)
            break
        rows = order[:n_act]
        out[rows] += contrib(edge[ptr[rows] + k])
    return out


def colsum_ref(x, n, cols):
    """-> (fp64 column sums, fp64 column sums of |x|) of x[:n, :cols]"""
    xs = x[:n, :cols].double()
    return xs.sum(0), xs.abs().sum(0)


def xent_ref(logits, labels):
    """-> (lse, per-vertex loss, softmax) in fp64 of fp32 logits [n, C] with int labels [n]"""
    l64 = logits.double()
    lse = torch.logsumexp(l64, dim=1)
    return lse, lse - l64.gather(1, labels.long()[:, None]).squeeze(1), torch.exp(l64 - lse[:, None])
