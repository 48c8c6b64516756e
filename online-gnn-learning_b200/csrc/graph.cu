// Streaming in-edge CSR on the GPU.
//
// Layout in HBM (all arrays device-resident):
//   row_start[v] int64, deg[v] int32, cap[v] int32      -- one slack row per vertex
//   adj[pool] uint64 = (edge id << 32) | source          -- adjacency pool, rows = [row_start, row_start+cap); one 8-byte
//                                                           entry per edge: a sampled pick costs ONE 32-byte sector, an
//                                                           insert ONE scattered store, and ordering a tail by edge id is
//                                                           ordering the entries as integers
// A snapshot's edges are appended into each touched row's tail (the per-snapshot delta
// region [deg_old, deg_new)); rows that run out of slack are relocated to the pool top with
// doubled capacity (bump allocation), so an insert costs O(batch) amortised instead of the
// reference's O(E_total) COO concat + CSC rebuild (dynamic_graph_edge.py:214-215, DGL
// add_edges).  Slots inside a batch are claimed with atomics and every tail is then put
// into ascending-edge-id order, so the row contents are canonical (bit-exact with the
// oracle's stable COO->CSC conversion).
#include "graph.cuh"

namespace ogl {

constexpr int kBlock = 256;

__device__ __forceinline__ int32_t grow_cap(int32_t need) {
  if (need <= 0) return 0;
  int64_t c = (int64_t)need * 2;
  if (c < 4) c = 4;
  c = (c + 3) & ~3LL;
  return (int32_t)(c > 0x7fffffffLL ? 0x7fffffff : c);
}

// -- batch edge accessor: i in [0, n) forward (src->dst), [n, 2n) reverse (dst->src) ------
struct BatchEdges {
  const int64_t* src;
  const int64_t* dst;
  int64_t n;
  int symmetric;
  __device__ __forceinline__ int64_t total() const { return symmetric ? 2 * n : n; }
  __device__ __forceinline__ void get(int64_t i, int64_t& s, int64_t& d) const {
    if (i < n) { s = src[i]; d = dst[i]; } else { s = dst[i - n]; d = src[i - n]; }
  }
};

__global__ void __launch_bounds__(kBlock) k_count(BatchEdges b, int32_t* __restrict__ add, int32_t* __restrict__ touched,
                                                  GraphCtl* ctl, int64_t n_vertices, int64_t n_sources) {
  const int64_t tot = b.total();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t s, d;
    b.get(i, s, d);
    if (s < 0 || d < 0 || s >= n_sources || d >= n_vertices) { ctl->bad_id = 1; continue; }
    int old = atomicAdd(&add[d], 1);
    if (old == 0) touched[atomicAdd(&ctl->n_touched, 1)] = (int32_t)d;
  }
}

// slots this batch must take from the pool top
__global__ void __launch_bounds__(kBlock) k_need(const int32_t* __restrict__ touched, const int32_t* __restrict__ add,
                                                 const int32_t* __restrict__ deg, const int32_t* __restrict__ cap, GraphCtl* ctl) {
  const int nt = ctl->n_touched;
  unsigned long long local = 0;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += gridDim.x * blockDim.x) {
    int v = touched[t];
    int need = deg[v] + add[v];
    if (need > cap[v]) local += (unsigned long long)grow_cap(need);
  }
  // warp reduce then one atomic per warp
  for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(&ctl->need, local);
}

// relocate rows without enough slack.  One THREAD per touched row claims the new space; rows of <= kThreadCopyMax
// entries (the overwhelming majority in a sparse batch) are copied by that thread, longer rows are queued: one warp
// per job up to kWarpCopyMax entries, all CTAs together beyond (a hub row of 10^5 entries must not hang on one warp).
// The global relocation counter and the job queue are updated once per warp / per job, not once per row.
constexpr int kThreadCopyMax = 16;
constexpr int kWarpCopyMax = 2048;
struct MoveJob { long long from, to; int len; int pad; };

__global__ void __launch_bounds__(kBlock) k_reserve(const int32_t* __restrict__ touched, const int32_t* __restrict__ add,
                                                    int64_t* __restrict__ row_start, const int32_t* __restrict__ deg,
                                                    int32_t* __restrict__ cap, int32_t* __restrict__ tail_len,
                                                    unsigned long long* __restrict__ adj, MoveJob* __restrict__ jobs,
                                                    int* __restrict__ n_jobs, int jobs_cap, GraphCtl* ctl) {
  const int nt = ctl->n_touched;
  for (int t0 = blockIdx.x * blockDim.x; t0 < nt; t0 += gridDim.x * blockDim.x) {
    const int t = t0 + threadIdx.x;
    bool moved = false;
    if (t < nt) {
      const int v = touched[t];
      const int a = add[v], d = deg[v];
      tail_len[t] = a;
      const int need = d + a;
      if (need > cap[v]) {
        moved = true;
        const int nc = grow_cap(need);
        const unsigned long long off = atomicAdd(&ctl->pool_top, (unsigned long long)nc);
        const int64_t old = row_start[v];
        if (d <= kThreadCopyMax) {
          for (int i = 0; i < d; ++i) adj[off + i] = adj[old + i];
        } else if (d <= kWarpCopyMax) {
          jobs[atomicAdd(n_jobs, 1)] = MoveJob{(long long)old, (long long)off, d, 0};                 // warp jobs: from the front
        } else {
          jobs[jobs_cap - 1 - atomicAdd(n_jobs + 1, 1)] = MoveJob{(long long)old, (long long)off, d, 0};   // big jobs: from the back
        }
        row_start[v] = (int64_t)off;
        cap[v] = nc;
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, moved);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&ctl->relocations, (unsigned long long)__popc(m));
  }
}

// queued row copies: warp jobs (front of the queue) go one per warp, big jobs (back of the queue) are swept by every CTA
__global__ void __launch_bounds__(kBlock) k_move_jobs(const MoveJob* __restrict__ jobs, const int* __restrict__ n_jobs, int jobs_cap,
                                                      unsigned long long* __restrict__ adj) {
  const int nw = n_jobs[0], nb = n_jobs[1];
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; q < nw; q += warps) {
    const MoveJob j = jobs[q];
    for (int i = lane; i < j.len; i += 32) adj[j.to + i] = adj[j.from + i];
  }
  for (int q = 0; q < nb; ++q) {
    const MoveJob j = jobs[jobs_cap - 1 - q];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < j.len; i += (int64_t)gridDim.x * blockDim.x)
      adj[j.to + i] = adj[j.from + i];
  }
}

// claim a slot in the row tail (arbitrary order inside the batch; fixed up by k_fix)
__global__ void __launch_bounds__(kBlock) k_place(BatchEdges b, int32_t* __restrict__ add, const int64_t* __restrict__ row_start,
                                                  const int32_t* __restrict__ deg, unsigned long long* __restrict__ adj,
                                                  uint32_t eid_base, int64_t n_vertices, int64_t n_sources) {
  const int64_t tot = b.total();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t s, d;
    b.get(i, s, d);
    if (s < 0 || d < 0 || s >= n_sources || d >= n_vertices) continue;
    const int p = atomicSub(&add[d], 1) - 1;      // add[] returns to zero by the end of the kernel
    const int64_t at = row_start[d] + deg[d] + p;
    adj[at] = ((unsigned long long)(eid_base + (uint32_t)i) << 32) | (uint32_t)s;
  }
}

// ---- tail ordering -------------------------------------------------------------------------------
// Slots inside a batch were claimed in arbitrary (atomic) order; every tail is put into ascending edge-id order so
// that the row contents are canonical.  Three size classes:
//   L <= 32        one warp, rank by shuffles, in registers                       (k_fix, inline)
//   L <= kMedTail  one warp, bitonic sort of (eid << 32 | src) keys in shared     (k_fix_med)
//   L <= kBigTail  one CTA, bitonic sort in dynamic shared memory                 (k_fix_big)
//   larger         one CTA, rank-by-counting through a global scratch (rare: a hub taking > 8192 edges of one batch)
constexpr int kMedTail = 512;
constexpr int kBigTail = 8192;

__device__ __forceinline__ void bitonic_step(unsigned long long* s, int i, int j, int k) {
  const int ixj = i ^ j;
  if (ixj > i) {
    const unsigned long long a = s[i], b = s[ixj];
    const bool up = (i & k) == 0;
    if ((a > b) == up) { s[i] = b; s[ixj] = a; }
  }
}

// classification, one THREAD per touched row: tails of 0 / 1 edges need no ordering (the common case in a sparse
// batch) and are finalised here; longer tails are queued by size class
__global__ void __launch_bounds__(kBlock) k_fix(const int32_t* __restrict__ touched, const int32_t* __restrict__ tail_len,
                                                int32_t* __restrict__ deg, int32_t* __restrict__ small, int32_t* __restrict__ med,
                                                int32_t* __restrict__ large, GraphCtl* ctl) {
  const int nt = ctl->n_touched;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += gridDim.x * blockDim.x) {
    const int L = tail_len[t];
    if (L <= 1) {
      if (L == 1) deg[touched[t]] += 1;
    } else if (L <= 32) {
      small[atomicAdd(&ctl->n_small, 1)] = t;
    } else if (L <= kMedTail) {
      med[atomicAdd(&ctl->n_med, 1)] = t;
    } else {
      large[atomicAdd(&ctl->n_large, 1)] = t;
    }
  }
}

// tails of 2..32 edges: one warp, rank by shuffles, in registers
__global__ void __launch_bounds__(kBlock) k_fix_small(const int32_t* __restrict__ touched, const int32_t* __restrict__ tail_len,
                                                      const int64_t* __restrict__ row_start, int32_t* __restrict__ deg,
                                                      unsigned long long* __restrict__ adj, const int32_t* __restrict__ small,
                                                      GraphCtl* ctl) {
  const int ns = ctl->n_small;
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; q < ns; q += warps) {
    const int t = small[q];
    const int v = touched[t];
    const int L = tail_len[t];
    const int64_t base = row_start[v] + deg[v];
    const unsigned long long ent = lane < L ? adj[base + lane] : ~0ull;
    const uint32_t e = (uint32_t)(ent >> 32);
    int rank = 0;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      uint32_t ej = __shfl_sync(0xffffffffu, e, j);
      rank += (j < L && ej < e) ? 1 : 0;
    }
    __syncwarp();
    if (lane < L) adj[base + rank] = ent;
    __syncwarp();
    if (lane == 0) deg[v] += L;
  }
}

__global__ void __launch_bounds__(kBlock) k_fix_med(const int32_t* __restrict__ touched, const int32_t* __restrict__ tail_len,
                                                    const int64_t* __restrict__ row_start, int32_t* __restrict__ deg,
                                                    unsigned long long* __restrict__ adj,
                                                    const int32_t* __restrict__ med, GraphCtl* ctl) {
  __shared__ unsigned long long keys[kBlock / 32][kMedTail];
  const int nm = ctl->n_med;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  unsigned long long* s = keys[w];
  for (int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; m < nm; m += warps) {
    const int t = med[m];
    const int v = touched[t];
    const int L = tail_len[t];
    const int64_t base = row_start[v] + deg[v];
    int P = 64;
    while (P < L) P <<= 1;
    for (int i = lane; i < P; i += 32) s[i] = i < L ? adj[base + i] : ~0ull;
    __syncwarp();
    for (int k = 2; k <= P; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = lane; i < P; i += 32) bitonic_step(s, i, j, k);
        __syncwarp();
      }
    for (int i = lane; i < L; i += 32) adj[base + i] = s[i];
    __syncwarp();
    if (lane == 0) deg[v] += L;
  }
}

// long tails (hub rows in a big batch): a whole CTA orders the tail
__global__ void __launch_bounds__(1024) k_fix_big(const int32_t* __restrict__ touched, const int32_t* __restrict__ tail_len,
                                                  const int64_t* __restrict__ row_start, int32_t* __restrict__ deg,
                                                  unsigned long long* __restrict__ adj, unsigned long long* __restrict__ scr,
                                                  const int32_t* __restrict__ large, GraphCtl* ctl) {
  extern __shared__ unsigned long long bk[];      // kBigTail keys
  __shared__ unsigned long long s_off;
  const int nl = ctl->n_large;
  for (int q = blockIdx.x; q < nl; q += gridDim.x) {
    const int t = large[q];
    const int v = touched[t];
    const int L = tail_len[t];
    const int64_t base = row_start[v] + deg[v];
    if (L <= kBigTail) {
      int P = 1024;
      while (P < L) P <<= 1;
      for (int i = threadIdx.x; i < P; i += blockDim.x) bk[i] = i < L ? adj[base + i] : ~0ull;
      __syncthreads();
      for (int k = 2; k <= P; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
          for (int i = threadIdx.x; i < P; i += blockDim.x) bitonic_step(bk, i, j, k);
          __syncthreads();
        }
      for (int i = threadIdx.x; i < L; i += blockDim.x) adj[base + i] = bk[i];
    } else {
      if (threadIdx.x == 0) s_off = atomicAdd(&ctl->scratch_top, (unsigned long long)L);
      __syncthreads();
      const unsigned long long off = s_off;
      for (int i = threadIdx.x; i < L; i += blockDim.x) scr[off + i] = adj[base + i];
      __syncthreads();
      for (int i = threadIdx.x; i < L; i += blockDim.x) {
        const unsigned long long e = scr[off + i];
        int rank = 0;
        for (int j = 0; j < L; ++j) rank += scr[off + j] < e ? 1 : 0;
        adj[base + rank] = e;
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) deg[v] += L;
    __syncthreads();
  }
}

// ---- the streaming regime: one snapshot = ONE kernel ------------------------------------------------------------------------
// The reference appends ~10^4 edges per evolve() (settings/reddit.json: 57.3 M stream edges over 5000 snapshots,
// dynamic_graph_edge.py:190-218).  At that size the seven-kernel sequence above is pure launch latency (nine launches and two
// memsets for < 1 MB of traffic), so batches of <= kFuseMaxEdges directed edges run through one cooperative kernel whose phases
// are separated by a grid barrier in global memory: count -> need (+ capacity / id check: on failure nothing is changed and the
// host takes the general path) -> reserve + relocate -> place -> order the tails (tails beyond kMedTail are left to k_fix_big).  Same results as the general path, bit for bit (rows end in edge-id order).
constexpr int kFuseMaxEdges = 1 << 16;
constexpr int kFuseWarpCopyMax = 1 << 14;

__device__ __forceinline__ void grid_barrier(GraphCtl* ctl, unsigned int n_blocks) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    volatile unsigned int* gen = &ctl->bar_gen;
    const unsigned int g = *gen;
    if (atomicAdd(&ctl->bar_count, 1u) == n_blocks - 1) {
      ctl->bar_count = 0;
      __threadfence();
      atomicAdd(&ctl->bar_gen, 1u);
    } else {
      while (*gen == g) __nanosleep(32);
    }
    __threadfence();
  }
  __syncthreads();
}

// what the host needs to know about a fused insert, written by the kernel straight into pinned host memory (the host spins on
// `seq` instead of paying a D2H copy + stream synchronisation per snapshot)
struct FusedStatus { volatile unsigned int seq; volatile int bad_id, overflow, n_large; };

__device__ __forceinline__ void fused_finish(GraphCtl* ctl, int* n_jobs, FusedStatus* st, unsigned int seq, int failed) {
  // every CTA is past its last read of the per-batch counters (grid barrier before this): publish, then leave them zeroed for
  // the next call (n_large stays for k_fix_big when it is not zero; the host clears it after that launch)
  st->bad_id = ctl->bad_id;
  st->overflow = failed;
  st->n_large = ctl->n_large;
  ctl->n_touched = 0; ctl->bad_id = 0; ctl->n_med = 0; ctl->n_small = 0; ctl->overflow = 0; ctl->need = 0; ctl->scratch_top = 0;
  n_jobs[0] = 0; n_jobs[1] = 0;
  __threadfence_system();
  st->seq = seq;
}

__global__ void __launch_bounds__(kBlock) k_insert_fused(BatchEdges b, int32_t* __restrict__ add, int32_t* __restrict__ touched,
                                                         int64_t* __restrict__ row_start, int32_t* __restrict__ deg, int32_t* __restrict__ cap,
                                                         int32_t* __restrict__ tail_len, unsigned long long* __restrict__ adj,
                                                         MoveJob* __restrict__ jobs, int* __restrict__ n_jobs, int jobs_cap,
                                                         int32_t* __restrict__ large, GraphCtl* ctl, int64_t n_vertices, uint32_t eid_base,
                                                         long long pool_cap, FusedStatus* status, unsigned int seq, int64_t n_sources) {
  __shared__ unsigned long long keys[kBlock / 32][kMedTail];
  const int64_t tot = b.total();
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (int64_t)gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int gwarp = (int)(tid >> 5), nwarps = (int)(nthreads >> 5);
  // ---- 1: per-row counts of the batch, list of touched rows
  for (int64_t i = tid; i < tot; i += nthreads) {
    int64_t s, d;
    b.get(i, s, d);
    if (s < 0 || d < 0 || s >= n_sources || d >= n_vertices) { ctl->bad_id = 1; continue; }
    if (atomicAdd(&add[d], 1) == 0) touched[atomicAdd(&ctl->n_touched, 1)] = (int32_t)d;
  }
  grid_barrier(ctl, gridDim.x);
  const int nt = ctl->n_touched;
  // ---- 2: pool slots the batch needs; bail out untouched if they are not there (or an id was bad)
  {
    unsigned long long local = 0;
    for (int t = (int)tid; t < nt; t += (int)nthreads) {
      const int v = touched[t];
      const int need = deg[v] + add[v];
      if (need > cap[v]) local += (unsigned long long)grow_cap(need);
    }
    for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if (lane == 0 && local) atomicAdd(&ctl->need, local);
  }
  grid_barrier(ctl, gridDim.x);
  if (ctl->bad_id || (long long)(ctl->pool_top + ctl->need) > pool_cap) {
    for (int t = (int)tid; t < nt; t += (int)nthreads) add[touched[t]] = 0;
    grid_barrier(ctl, gridDim.x);                  // (uniform: every CTA read the same values after the barrier above)
    if (tid == 0) fused_finish(ctl, n_jobs, status, seq, 1);
    return;
  }
  // ---- 3: claim tails; rows without slack move to the pool top with doubled capacity.  One THREAD per touched row (the row
  //         metadata is a chain of dependent loads: a warp per row would serialise ~60 of them); a row that must move more than
  //         kThreadCopyMax entries is then copied by its whole warp, hub rows are queued for every CTA
  for (int q0 = (int)(tid - lane); q0 < nt; q0 += (int)nthreads) {
    const int q = q0 + lane;
    int d = 0, nc = 0;
    int64_t old = 0;
    unsigned long long off = 0;
    bool warp_copy = false;
    if (q < nt) {
      const int v = touched[q];
      const int a = add[v];
      d = deg[v];
      tail_len[q] = a;
      const int need = d + a;
      if (need > cap[v]) {
        nc = grow_cap(need);
        off = atomicAdd(&ctl->pool_top, (unsigned long long)nc);
        old = row_start[v];
        if (d <= kThreadCopyMax) {
          for (int i = 0; i < d; ++i) adj[off + i] = adj[old + i];
        } else if (d <= kFuseWarpCopyMax) {
          warp_copy = true;
        } else {
          jobs[jobs_cap - 1 - atomicAdd(n_jobs + 1, 1)] = MoveJob{(long long)old, (long long)off, d, 0};   // a hub row: every CTA helps below
        }
        row_start[v] = (int64_t)off;
        cap[v] = nc;
      }
    }
    const unsigned moved = __ballot_sync(0xffffffffu, nc > 0);
    if (lane == 0 && moved) atomicAdd(&ctl->relocations, (unsigned long long)__popc(moved));
    unsigned todo = __ballot_sync(0xffffffffu, warp_copy);
    while (todo) {
      const int src_lane = __ffs(todo) - 1;
      todo &= todo - 1;
      const int dd = __shfl_sync(0xffffffffu, d, src_lane);
      const long long from = __shfl_sync(0xffffffffu, (long long)old, src_lane);
      const unsigned long long to = __shfl_sync(0xffffffffu, off, src_lane);
      // eight independent loads in flight per lane (a plain copy loop is one L2 round trip per 32 entries)
      for (int i0 = 0; i0 < dd; i0 += 256) {
        unsigned long long u[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int i = i0 + k * 32 + lane;
          u[k] = i < dd ? adj[from + i] : 0ull;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int i = i0 + k * 32 + lane;
          if (i < dd) adj[to + i] = u[k];
        }
      }
    }
  }
  grid_barrier(ctl, gridDim.x);
  // ---- 4: hub rows queued above (they write [new, new + deg), the placement below writes behind that: no conflict)
  {
    const int nb = n_jobs[1];
    for (int q = 0; q < nb; ++q) {
      const MoveJob j = jobs[jobs_cap - 1 - q];
      for (int64_t i = tid; i < j.len; i += nthreads) adj[j.to + i] = adj[j.from + i];
    }
  }
  // ---- 5: place every edge in a slot of its row's tail (arbitrary order inside the tail)
  for (int64_t i = tid; i < tot; i += nthreads) {
    int64_t s, d;
    b.get(i, s, d);
    const int p = atomicSub(&add[d], 1) - 1;        // add[] is back at zero when this phase ends
    adj[row_start[d] + deg[d] + p] = ((unsigned long long)(eid_base + (uint32_t)i) << 32) | (uint32_t)s;
  }
  grid_barrier(ctl, gridDim.x);
  // ---- 6: every tail into ascending edge-id order, then the degrees.  One thread per touched row again: tails of one edge (the
  //         common case) are finished by the thread; longer ones are ordered by the whole warp, one after the other
  unsigned long long* sk = keys[w];
  for (int q0 = (int)(tid - lane); q0 < nt; q0 += (int)nthreads) {
    const int q = q0 + lane;
    int v = 0, L = 0;
    int64_t base = 0;
    if (q < nt) {
      v = touched[q];
      L = tail_len[q];
      base = row_start[v] + deg[v];
      if (L == 1) deg[v] += 1;
      else if (L > kMedTail) large[atomicAdd(&ctl->n_large, 1)] = q;      // ordered by k_fix_big, launched by the host when the count is not zero
    }
    unsigned todo = __ballot_sync(0xffffffffu, L > 1 && L <= kMedTail);
    while (todo) {
      const int src_lane = __ffs(todo) - 1;
      todo &= todo - 1;
      const int Lw = __shfl_sync(0xffffffffu, L, src_lane);
      const int vw = __shfl_sync(0xffffffffu, v, src_lane);
      const long long bw = __shfl_sync(0xffffffffu, (long long)base, src_lane);
      if (Lw <= 32) {
        const unsigned long long ent = lane < Lw ? adj[bw + lane] : ~0ull;
        const uint32_t e = (uint32_t)(ent >> 32);
        int rank = 0;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const uint32_t ej = __shfl_sync(0xffffffffu, e, j);
          rank += (j < Lw && ej < e) ? 1 : 0;
        }
        __syncwarp();
        if (lane < Lw) adj[bw + rank] = ent;
      } else {
        int P = 64;
        while (P < Lw) P <<= 1;
        for (int i = lane; i < P; i += 32) sk[i] = i < Lw ? adj[bw + i] : ~0ull;
        __syncwarp();
        for (int k = 2; k <= P; k <<= 1)
          for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = lane; i < P; i += 32) bitonic_step(sk, i, j, k);
            __syncwarp();
          }
        for (int i = lane; i < Lw; i += 32) adj[bw + i] = sk[i];
      }
      __syncwarp();
      if (lane == 0) deg[vw] += Lw;
    }
  }
  grid_barrier(ctl, gridDim.x);
  if (tid == 0) fused_finish(ctl, n_jobs, status, seq, 0);
}

// ---- compaction / growth: rewrite all rows into a fresh pool ---------------------------------
__global__ void __launch_bounds__(kBlock) k_newcap(const int32_t* __restrict__ deg, const int32_t* __restrict__ add,
                                                   int32_t* __restrict__ newcap, int64_t n) {
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x)
    newcap[v] = grow_cap(deg[v] + add[v]);
}

__global__ void __launch_bounds__(kBlock) k_move_rows(const int64_t* __restrict__ old_start, const int64_t* __restrict__ new_start,
                                                      const int32_t* __restrict__ deg, const unsigned long long* __restrict__ old_adj,
                                                      unsigned long long* __restrict__ new_adj, int64_t n) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < n; v += warps) {
    const int d = deg[v];
    const int64_t a = old_start[v], b = new_start[v];
    for (int i = lane; i < d; i += 32) new_adj[b + i] = old_adj[a + i];
  }
}

// ---- export / degrees ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) k_deg64(const int32_t* __restrict__ deg, int64_t* __restrict__ out, int64_t n) {
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x) out[v] = deg[v];
}

__global__ void __launch_bounds__(kBlock) k_export_rows(const int64_t* __restrict__ row_start, const int32_t* __restrict__ deg,
                                                        const unsigned long long* __restrict__ adj,
                                                        const int64_t* __restrict__ indptr, int64_t* __restrict__ indices,
                                                        int64_t* __restrict__ eids, int64_t n) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < n; v += warps) {
    const int d = deg[v];
    const int64_t a = row_start[v], b = indptr[v];
    for (int i = lane; i < d; i += 32) {
      const unsigned long long ent = adj[a + i];
      indices[b + i] = (int64_t)(uint32_t)ent;
      if (eids) eids[b + i] = (int64_t)(ent >> 32);
    }
  }
}

__global__ void k_set_last(int64_t* indptr, const int64_t* total, int64_t n) { indptr[n] = *total; }

// ---- vertex streams: induced subgraph of the arrival-order prefix ------------------------------
__global__ void __launch_bounds__(kBlock) k_convert_parent(const int64_t* __restrict__ indices, const int64_t* __restrict__ eids,
                                                           int32_t* __restrict__ p_indices, uint32_t* __restrict__ p_eids, int64_t e) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < e; i += (int64_t)gridDim.x * blockDim.x) {
    p_indices[i] = (int32_t)indices[i];
    p_eids[i] = (uint32_t)eids[i];
  }
}

__global__ void __launch_bounds__(kBlock) k_prefix_count(const int64_t* __restrict__ p_indptr, const int32_t* __restrict__ p_indices,
                                                         int32_t* __restrict__ deg, int32_t* __restrict__ cap, int64_t n_active, int64_t v_all) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < v_all; v += warps) {
    int c = 0;
    if (v < n_active) {
      const int64_t a = p_indptr[v], b = p_indptr[v + 1];
      for (int64_t i = a + lane; i < b; i += 32) c += (p_indices[i] < n_active) ? 1 : 0;
      for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
    }
    if (lane == 0) { deg[v] = c; cap[v] = c; }
  }
}

__global__ void __launch_bounds__(kBlock) k_prefix_fill(const int64_t* __restrict__ p_indptr, const int32_t* __restrict__ p_indices,
                                                        const uint32_t* __restrict__ p_eids, const int64_t* __restrict__ row_start,
                                                        unsigned long long* __restrict__ adj, int64_t n_active) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; v < n_active; v += warps) {
    const int64_t a = p_indptr[v], b = p_indptr[v + 1];
    int64_t out = row_start[v];
    for (int64_t i0 = a; i0 < b; i0 += 32) {
      const int64_t i = i0 + lane;
      const int32_t u = i < b ? p_indices[i] : 0x7fffffff;
      const bool keep = u < n_active;
      const unsigned m = __ballot_sync(0xffffffffu, keep);
      if (keep) {
        const int64_t at = out + __popc(m & ((1u << lane) - 1));
        adj[at] = ((unsigned long long)p_eids[i] << 32) | (uint32_t)u;
      }
      out += __popc(m);
    }
  }
}

}  // namespace ogl

using namespace ogl;

// ================================== host side ====================================================
struct ogl_graph {
  int64_t v_cap = 0, pool_cap = 0;
  int64_t n_vertices = 0, n_edges = 0;
  int64_t batch_cap = 0;   // stream edges per internal chunk
  int64_t* row_start = nullptr;
  int32_t *deg = nullptr, *cap = nullptr, *add = nullptr;
  unsigned long long* adj = nullptr;     // (eid << 32) | src
  GraphCtl* ctl = nullptr;
  GraphCtl* h_ctl = nullptr;     // pinned mirror
  int32_t *touched = nullptr, *tail_len = nullptr, *large = nullptr, *med = nullptr, *small = nullptr;
  ogl::MoveJob* jobs = nullptr;
  int* n_jobs = nullptr;               // [0] warp jobs (queue front), [1] big jobs (queue back)
  int jobs_cap = 0;
  unsigned long long* scr = nullptr;
  int64_t *stage_src = nullptr, *stage_dst = nullptr;   // host-insert staging
  int32_t* newcap = nullptr;
  int64_t* scan_scratch = nullptr;
  int64_t* total_dev = nullptr;
  int64_t* new_start = nullptr;
  // parent graph (vertex streams)
  int64_t* p_indptr = nullptr;
  int32_t* p_indices = nullptr;
  uint32_t* p_eids = nullptr;
  int64_t p_v = 0, p_e = 0;
  int64_t pool_used_host = 0, relocations = 0, compactions = 0;
  uint64_t generation = 1;
  int64_t src_bound = 0;                 // sources may be any id in [0, src_bound) (0: the graph's own vertex count): a shard of a
                                         // destination-range-partitioned CSR stores GLOBAL source ids in its local rows
  int fuse_small = 1;                    // snapshot-sized batches go through the single cooperative kernel (OGL_INSERT_FUSED=0: off)
  void* h_status = nullptr;              // pinned: FusedStatus written by the fused kernel
  unsigned int fused_seq = 0;
  int fused_dirty = 0;                   // per-batch device counters may be non-zero (the fused kernel expects and leaves them zero)
};

static int graph_alloc_pool(ogl_graph* g, int64_t cap) {
  g->generation++;
  OGL_CUDA(cudaMalloc(&g->adj, sizeof(unsigned long long) * (size_t)cap));
  g->pool_cap = cap;
  return OGL_OK;
}

extern "C" int ogl_graph_create(ogl_graph** out, int64_t v_cap, int64_t e_cap_directed) {
  OGL_TRY(require_device());
  OGL_ARG(out && v_cap > 0 && e_cap_directed >= 0, "ogl_graph_create: bad arguments");
  OGL_ARG(v_cap < 0x7fffffffLL, "ogl_graph_create: v_cap must fit int32");
  ogl_graph* g = new ogl_graph();
  g->v_cap = v_cap;
  if (const char* e = getenv("OGL_INSERT_FUSED")) g->fuse_small = atoi(e) != 0;
  g->batch_cap = 1 << 21;
  const int64_t pool = e_cap_directed * 3 + 1024;   // slack rows (x2) + relocation holes
  int r = graph_alloc_pool(g, pool);
  if (r != OGL_OK) { delete g; return r; }
#define A(ptr, bytes) OGL_CUDA(cudaMalloc(&(ptr), (size_t)(bytes)))
  A(g->row_start, sizeof(int64_t) * v_cap);
  A(g->deg, sizeof(int32_t) * v_cap);
  A(g->cap, sizeof(int32_t) * v_cap);
  A(g->add, sizeof(int32_t) * v_cap);
  A(g->newcap, sizeof(int32_t) * v_cap);
  A(g->new_start, sizeof(int64_t) * (v_cap + 1));
  A(g->ctl, sizeof(GraphCtl));
  A(g->touched, sizeof(int32_t) * 2 * g->batch_cap);
  A(g->tail_len, sizeof(int32_t) * 2 * g->batch_cap);
  A(g->large, sizeof(int32_t) * (2 * g->batch_cap / kMedTail + 64));
  A(g->med, sizeof(int32_t) * (2 * g->batch_cap / 32 + 64));
  A(g->small, sizeof(int32_t) * (g->batch_cap + 64));              // tails of >= 2 edges: at most tot / 2 rows
  g->jobs_cap = (int)((v_cap < 2 * g->batch_cap ? v_cap : 2 * g->batch_cap) + 64);   // <= one job per touched row
  A(g->jobs, sizeof(MoveJob) * g->jobs_cap);
  A(g->n_jobs, 2 * sizeof(int));
  A(g->scr, sizeof(unsigned long long) * 2 * g->batch_cap);
  A(g->stage_src, sizeof(int64_t) * g->batch_cap);
  A(g->stage_dst, sizeof(int64_t) * g->batch_cap);
  A(g->scan_scratch, sizeof(int64_t) * scan_scratch_elems(v_cap + 1));
  A(g->total_dev, sizeof(int64_t));
#undef A
  OGL_CUDA(cudaMallocHost(&g->h_ctl, sizeof(GraphCtl)));
  OGL_CUDA(cudaMallocHost(&g->h_status, 64));
  memset(g->h_status, 0, 64);
  OGL_CUDA(cudaFuncSetAttribute(k_fix_big, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kBigTail * sizeof(unsigned long long))));
  OGL_CUDA(cudaMemset(g->row_start, 0, sizeof(int64_t) * v_cap));
  OGL_CUDA(cudaMemset(g->deg, 0, sizeof(int32_t) * v_cap));
  OGL_CUDA(cudaMemset(g->cap, 0, sizeof(int32_t) * v_cap));
  OGL_CUDA(cudaMemset(g->add, 0, sizeof(int32_t) * v_cap));
  OGL_CUDA(cudaMemset(g->ctl, 0, sizeof(GraphCtl)));
  OGL_CUDA(cudaMemset(g->n_jobs, 0, 2 * sizeof(int)));      // (the fused insert expects and leaves the per-batch counters zero)
  *out = g;
  return OGL_OK;
}

extern "C" int ogl_graph_destroy(ogl_graph* g) {
  if (!g) return OGL_OK;
  void* ptrs[] = {g->row_start, g->deg, g->cap, g->add, g->adj, g->ctl, g->touched, g->tail_len, g->large, g->med, g->small, g->jobs, g->n_jobs,
                  g->scr, g->stage_src, g->stage_dst, g->newcap, g->scan_scratch, g->total_dev, g->new_start,
                  g->p_indptr, g->p_indices, g->p_eids};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (g->h_ctl) cudaFreeHost(g->h_ctl);
  if (g->h_status) cudaFreeHost(g->h_status);
  delete g;
  return OGL_OK;
}

extern "C" int ogl_graph_insert_vertices(ogl_graph* g, int64_t n, void* stream) {
  OGL_ARG(g && n >= 0, "ogl_graph_insert_vertices: bad arguments");
  if (g->n_vertices + n > g->v_cap) {
    set_error("ogl_graph_insert_vertices: %lld + %lld exceeds v_cap %lld", (long long)g->n_vertices, (long long)n, (long long)g->v_cap);
    return OGL_ERR_CAPACITY;
  }
  g->n_vertices += n;
  return OGL_OK;
}

// rewrite all rows into a pool of at least `min_cap` slots; caps become grow(deg + pending add)
static int graph_rebuild_pool(ogl_graph* g, int64_t extra, cudaStream_t s) {
  const int64_t V = g->n_vertices;
  OGL_LAUNCH(k_newcap, grid_for(V, kBlock), kBlock, 0, s, g->deg, g->add, g->newcap, V);
  OGL_TRY(exclusive_scan_i32_to_i64(g->newcap, g->new_start, V, g->scan_scratch, g->total_dev, s));
  int64_t total = 0;
  OGL_CUDA(cudaMemcpyAsync(&total, g->total_dev, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  OGL_CUDA(cudaStreamSynchronize(s));
  int64_t want = total + total / 2 + extra + 1024;
  if (want < g->pool_cap) want = g->pool_cap;
  unsigned long long* old_adj = g->adj;
  OGL_TRY(graph_alloc_pool(g, want));
  OGL_LAUNCH(k_move_rows, grid_for(V * 32, kBlock), kBlock, 0, s, g->row_start, g->new_start, g->deg, old_adj, g->adj, V);
  OGL_CUDA(cudaMemcpyAsync(g->row_start, g->new_start, sizeof(int64_t) * V, cudaMemcpyDeviceToDevice, s));
  OGL_CUDA(cudaMemcpyAsync(g->cap, g->newcap, sizeof(int32_t) * V, cudaMemcpyDeviceToDevice, s));
  unsigned long long top = (unsigned long long)total;
  OGL_CUDA(cudaMemcpyAsync(&g->ctl->pool_top, &top, sizeof(top), cudaMemcpyHostToDevice, s));
  OGL_CUDA(cudaStreamSynchronize(s));
  cudaFree(old_adj);
  g->pool_used_host = total;
  g->compactions++;
  return OGL_OK;
}

// one snapshot-sized batch through the single cooperative kernel; *done = 0 when the pool has no room (the general path rebuilds it)
static int graph_insert_fused(ogl_graph* g, const BatchEdges& b, int64_t tot, cudaStream_t s, int* done) {
  static int max_blocks = 0;
  if (max_blocks == 0) {
    int per_sm = 0;
    OGL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_insert_fused, kBlock, 0));
    max_blocks = per_sm * sm_count();
    if (max_blocks < 1) max_blocks = -1;
  }
  *done = 0;
  if (max_blocks < 0) return OGL_OK;
  int grid = (int)ceil_div(tot, kBlock);          // about one edge / one touched row per thread, at most one CTA per SM
  if (grid < 8) grid = 8;
  if (grid > sm_count()) grid = sm_count();
  if (grid > max_blocks) grid = max_blocks;
  if (g->fused_dirty) {                           // the general path (or k_fix_big) left per-batch counters behind
    OGL_CUDA(cudaMemsetAsync(&g->ctl->n_touched, 0, sizeof(GraphCtl) - offsetof(GraphCtl, n_touched), s));
    OGL_CUDA(cudaMemsetAsync(g->n_jobs, 0, 2 * sizeof(int), s));
    g->fused_dirty = 0;
  }
  BatchEdges bb = b;
  int64_t nv = g->n_vertices;
  int64_t ns = g->src_bound > 0 ? g->src_bound : g->n_vertices;
  uint32_t eid_base = (uint32_t)g->n_edges;
  long long pool_cap = g->pool_cap;
  FusedStatus* st = (FusedStatus*)g->h_status;
  unsigned int seq = ++g->fused_seq;
  void* args[] = {&bb, &g->add, &g->touched, &g->row_start, &g->deg, &g->cap, &g->tail_len, &g->adj, &g->jobs, &g->n_jobs, &g->jobs_cap,
                  &g->large, &g->ctl, &nv, &eid_base, &pool_cap, &st, &seq, &ns};
  OGL_CUDA(cudaLaunchCooperativeKernel((const void*)k_insert_fused, dim3((unsigned)grid), dim3(kBlock), args, 0, s));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  // the kernel's last act is to write its status into pinned host memory: spin on the sequence number (a launch failure or a
  // device fault shows up as an error of the stream query, never as an endless wait)
  for (unsigned spins = 0; st->seq != seq; ++spins) {
    if ((spins & 0x3ff) == 0x3ff) {
      const cudaError_t qe = cudaStreamQuery(s);
      if (qe != cudaSuccess && qe != cudaErrorNotReady) OGL_CUDA(qe);
      if (qe == cudaSuccess && st->seq != seq) OGL_CUDA(cudaStreamSynchronize(s));
    }
  }
  if (st->bad_id) {                               // (the kernel changed nothing)
    set_error("ogl_graph_insert_edges: vertex id out of range [0, %lld) (call insert_vertices first)", (long long)g->n_vertices);
    return OGL_ERR_ARG;
  }
  if (st->overflow) return OGL_OK;
  if (st->n_large > 0) {
    OGL_LAUNCH(k_fix_big, sm_count() * 2, 1024, kBigTail * sizeof(unsigned long long), s, g->touched, g->tail_len, g->row_start, g->deg,
               g->adj, g->scr, g->large, g->ctl);
    g->fused_dirty = 1;
  }
  g->n_edges += tot;
  *done = 1;
  return OGL_OK;
}

static int graph_insert_chunk(ogl_graph* g, const int64_t* src_dev, const int64_t* dst_dev, int64_t n, int symmetric, cudaStream_t s) {
  BatchEdges b{src_dev, dst_dev, n, symmetric};
  const int64_t tot = symmetric ? 2 * n : n;
  if (g->n_edges + tot > 0xffffffffLL) {
    set_error("ogl_graph_insert_edges: edge ids exceed 32 bits");
    return OGL_ERR_CAPACITY;
  }
  if (tot <= kFuseMaxEdges && g->fuse_small) {
    int done = 0;
    OGL_TRY(graph_insert_fused(g, b, tot, s, &done));
    if (done) return OGL_OK;
  }
  // reset the per-batch counters (pool_top / relocations persist)
  g->fused_dirty = 1;
  OGL_CUDA(cudaMemsetAsync(&g->ctl->n_touched, 0, sizeof(GraphCtl) - offsetof(GraphCtl, n_touched), s));
  const int64_t n_src = g->src_bound > 0 ? g->src_bound : g->n_vertices;
  OGL_LAUNCH(k_count, grid_for(tot, kBlock), kBlock, 0, s, b, g->add, g->touched, g->ctl, g->n_vertices, n_src);
  OGL_LAUNCH(k_need, grid_for(tot, kBlock), kBlock, 0, s, g->touched, g->add, g->deg, g->cap, g->ctl);
  OGL_CUDA(cudaMemcpyAsync(g->h_ctl, g->ctl, sizeof(GraphCtl), cudaMemcpyDeviceToHost, s));
  OGL_CUDA(cudaStreamSynchronize(s));
  if (g->h_ctl->bad_id) {
    // undo the counters so the graph stays usable
    OGL_CUDA(cudaMemsetAsync(g->add, 0, sizeof(int32_t) * g->v_cap, s));
    set_error("ogl_graph_insert_edges: vertex id out of range [0, %lld) (call insert_vertices first)", (long long)g->n_vertices);
    return OGL_ERR_ARG;
  }
  if ((int64_t)(g->h_ctl->pool_top + g->h_ctl->need) > g->pool_cap) {
    OGL_TRY(graph_rebuild_pool(g, tot, s));   // caps now cover the pending adds: nothing left to relocate
  }
  const int nt = g->h_ctl->n_touched;
  const int wgrid = grid_for((int64_t)nt * 32, kBlock);
  const int tgrid = grid_for(nt, kBlock);
  OGL_CUDA(cudaMemsetAsync(g->n_jobs, 0, 2 * sizeof(int), s));
  OGL_LAUNCH(k_reserve, tgrid, kBlock, 0, s, g->touched, g->add, g->row_start, g->deg, g->cap, g->tail_len, g->adj, g->jobs,
             g->n_jobs, g->jobs_cap, g->ctl);
  OGL_LAUNCH(k_move_jobs, sm_count() * 8, kBlock, 0, s, g->jobs, g->n_jobs, g->jobs_cap, g->adj);
  OGL_LAUNCH(k_place, grid_for(tot, kBlock), kBlock, 0, s, b, g->add, g->row_start, g->deg, g->adj,
             (uint32_t)g->n_edges, g->n_vertices, n_src);
  OGL_LAUNCH(k_fix, tgrid, kBlock, 0, s, g->touched, g->tail_len, g->deg, g->small, g->med, g->large, g->ctl);
  OGL_LAUNCH(k_fix_small, wgrid, kBlock, 0, s, g->touched, g->tail_len, g->row_start, g->deg, g->adj, g->small, g->ctl);
  OGL_LAUNCH(k_fix_med, grid_for((int64_t)nt * 4, kBlock, 4), kBlock, 0, s, g->touched, g->tail_len, g->row_start, g->deg, g->adj,
             g->med, g->ctl);
  OGL_LAUNCH(k_fix_big, sm_count() * 2, 1024, kBigTail * sizeof(unsigned long long), s, g->touched, g->tail_len, g->row_start, g->deg,
             g->adj, g->scr, g->large, g->ctl);
  g->n_edges += tot;
  return OGL_OK;
}

static int graph_insert(ogl_graph* g, const int64_t* src, const int64_t* dst, int64_t n, int symmetric, int on_host, void* stream) {
  OGL_ARG(g && n >= 0 && (n == 0 || (src && dst)), "ogl_graph_insert_edges: bad arguments");
  OGL_ARG(g->p_indptr == nullptr, "ogl_graph_insert_edges: graph is in vertex-stream (parent prefix) mode");
  cudaStream_t s = (cudaStream_t)stream;
  // edge ids inside one call are forward-then-reverse over the WHOLE call (dynamic_graph_edge.py:214-215), so a
  // symmetric call that does not fit one chunk is issued as forward chunks followed by reverse chunks.
  if (n == 0) return OGL_OK;
  OGL_TRY(readers_wait(g, s));                 // a prefetched minibatch may still be sampling this CSR on its plan's stream
  if (!symmetric || n <= g->batch_cap) {
    for (int64_t o = 0; o < n; o += g->batch_cap) {
      const int64_t m = (n - o < g->batch_cap) ? n - o : g->batch_cap;
      const int64_t *ps = src + o, *pd = dst + o;
      if (on_host) {
        OGL_CUDA(cudaMemcpyAsync(g->stage_src, ps, sizeof(int64_t) * m, cudaMemcpyHostToDevice, s));
        OGL_CUDA(cudaMemcpyAsync(g->stage_dst, pd, sizeof(int64_t) * m, cudaMemcpyHostToDevice, s));
        ps = g->stage_src; pd = g->stage_dst;
      }
      OGL_TRY(graph_insert_chunk(g, ps, pd, m, symmetric, s));
    }
    return OGL_OK;
  }
  OGL_TRY(graph_insert(g, src, dst, n, 0, on_host, stream));
  return graph_insert(g, dst, src, n, 0, on_host, stream);
}

extern "C" int ogl_graph_insert_edges(ogl_graph* g, const int64_t* src_dev, const int64_t* dst_dev, int64_t n, int symmetric, void* stream) {
  return graph_insert(g, src_dev, dst_dev, n, symmetric, 0, stream);
}
extern "C" int ogl_graph_insert_edges_host(ogl_graph* g, const int64_t* src_host, const int64_t* dst_host, int64_t n, int symmetric, void* stream) {
  return graph_insert(g, src_host, dst_host, n, symmetric, 1, stream);
}

extern "C" int ogl_graph_set_source_bound(ogl_graph* g, int64_t n_sources) {
  OGL_ARG(g && n_sources >= 0 && n_sources < 0xffffffffLL, "ogl_graph_set_source_bound: bad arguments");
  g->src_bound = n_sources;
  return OGL_OK;
}

extern "C" int ogl_graph_compact(ogl_graph* g, void* stream) {
  OGL_ARG(g, "ogl_graph_compact: null graph");
  if (g->p_indptr) return OGL_OK;
  OGL_TRY(readers_wait(g, (cudaStream_t)stream));
  return graph_rebuild_pool(g, 0, (cudaStream_t)stream);
}

extern "C" int ogl_graph_num_vertices(ogl_graph* g, int64_t* out) { OGL_ARG(g && out, "null"); *out = g->n_vertices; return OGL_OK; }
extern "C" int ogl_graph_num_edges(ogl_graph* g, int64_t* out) { OGL_ARG(g && out, "null"); *out = g->n_edges; return OGL_OK; }

extern "C" int ogl_graph_degrees(ogl_graph* g, int64_t* out_dev, void* stream) {
  OGL_ARG(g && out_dev, "ogl_graph_degrees: null");
  if (g->n_vertices == 0) return OGL_OK;
  OGL_LAUNCH(k_deg64, grid_for(g->n_vertices, kBlock), kBlock, 0, stream, g->deg, out_dev, g->n_vertices);
  return OGL_OK;
}

extern "C" int ogl_graph_export_csr(ogl_graph* g, int64_t* indptr_dev, int64_t* indices_dev, int64_t* eids_dev, void* stream) {
  OGL_ARG(g && indptr_dev && (indices_dev || g->n_edges == 0), "ogl_graph_export_csr: null");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t V = g->n_vertices;
  OGL_TRY(exclusive_scan_i32_to_i64(g->deg, indptr_dev, V, g->scan_scratch, g->total_dev, s));
  OGL_LAUNCH(k_set_last, 1, 1, 0, s, indptr_dev, g->total_dev, V);
  if (V > 0 && g->n_edges > 0)
    OGL_LAUNCH(k_export_rows, grid_for(V * 32, kBlock), kBlock, 0, s, g->row_start, g->deg, g->adj, indptr_dev,
               indices_dev, eids_dev, V);
  return OGL_OK;
}

extern "C" int ogl_graph_stats(ogl_graph* g, int64_t out[4]) {
  OGL_ARG(g && out, "null");
  GraphCtl c;
  OGL_CUDA(cudaMemcpy(&c, g->ctl, sizeof(c), cudaMemcpyDeviceToHost));
  out[0] = (int64_t)c.pool_top; out[1] = g->pool_cap; out[2] = (int64_t)c.relocations; out[3] = g->compactions;
  return OGL_OK;
}

extern "C" int ogl_graph_load_parent(ogl_graph* g, const int64_t* indptr_dev, const int64_t* indices_dev, const int64_t* eids_dev,
                                     int64_t n_vertices, void* stream) {
  OGL_ARG(g && indptr_dev && n_vertices > 0 && n_vertices <= g->v_cap, "ogl_graph_load_parent: bad arguments");
  OGL_ARG(g->n_edges == 0 && g->p_indptr == nullptr, "ogl_graph_load_parent: graph not empty");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t e = 0;
  OGL_CUDA(cudaMemcpyAsync(&e, indptr_dev + n_vertices, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  OGL_CUDA(cudaStreamSynchronize(s));
  OGL_ARG(e >= 0 && e <= 0xffffffffLL, "ogl_graph_load_parent: bad edge count");
  if (e > g->pool_cap) {
    cudaFree(g->adj);
    OGL_TRY(graph_alloc_pool(g, e + 1024));
  }
  OGL_CUDA(cudaMalloc(&g->p_indptr, sizeof(int64_t) * (n_vertices + 1)));
  OGL_CUDA(cudaMalloc(&g->p_indices, sizeof(int32_t) * (e + 1)));
  OGL_CUDA(cudaMalloc(&g->p_eids, sizeof(uint32_t) * (e + 1)));
  OGL_CUDA(cudaMemcpyAsync(g->p_indptr, indptr_dev, sizeof(int64_t) * (n_vertices + 1), cudaMemcpyDeviceToDevice, s));
  if (e > 0) OGL_LAUNCH(k_convert_parent, grid_for(e, kBlock), kBlock, 0, s, indices_dev, eids_dev, g->p_indices, g->p_eids, e);
  g->p_v = n_vertices;
  g->p_e = e;
  g->n_vertices = 0;
  return OGL_OK;
}

extern "C" int ogl_graph_set_active_prefix(ogl_graph* g, int64_t n_active, void* stream) {
  OGL_ARG(g && g->p_indptr, "ogl_graph_set_active_prefix: no parent graph loaded");
  OGL_ARG(n_active >= 0 && n_active <= g->p_v, "ogl_graph_set_active_prefix: n_active out of range");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t V = g->p_v;
  OGL_TRY(readers_wait(g, s));
  OGL_LAUNCH(k_prefix_count, grid_for(V * 32, kBlock), kBlock, 0, s, g->p_indptr, g->p_indices, g->deg, g->cap, n_active, V);
  OGL_TRY(exclusive_scan_i32_to_i64(g->deg, g->row_start, V, g->scan_scratch, g->total_dev, s));
  if (n_active > 0)
    OGL_LAUNCH(k_prefix_fill, grid_for(n_active * 32, kBlock), kBlock, 0, s, g->p_indptr, g->p_indices, g->p_eids, g->row_start,
               g->adj, n_active);
  int64_t total = 0;
  OGL_CUDA(cudaMemcpyAsync(&total, g->total_dev, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  OGL_CUDA(cudaStreamSynchronize(s));
  g->n_vertices = n_active;
  g->n_edges = total;
  return OGL_OK;
}

namespace ogl {
uint64_t graph_generation(const ogl_graph* g) { return g->generation; }
int64_t graph_num_edges(const ogl_graph* g) { return g->n_edges; }
int64_t graph_source_bound(const ogl_graph* g) { return g->src_bound; }
GraphView graph_view(const ogl_graph* g) {
  GraphView v;
  v.row_start = g->row_start; v.deg = g->deg; v.adj = g->adj; v.n_vertices = g->n_vertices;
  return v;
}
}  // namespace ogl
