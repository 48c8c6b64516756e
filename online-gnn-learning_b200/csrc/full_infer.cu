// Full-neighbourhood segment max: out[v] = max over EVERY in-edge (u -> v) of x[u], read straight from the streaming CSR
// (slack capacity, relocated rows and per-snapshot tails in place).  Memory-bound: each edge reads one [pitch] row of x.
//
// Degree skew is handled in three launches:
//   rows:    persistent warps take rows one at a time from a device cursor (power-law degrees make any static split uneven); a warp
//            walks the row's adjacency 32 entries at a time (one coalesced 256-byte load, sources broadcast by shuffle), each
//            lane owning one 16-byte column strip per pass, eight edge rows in flight.  A row of more than kSegmaxChunk edges is
//            a hub: the warp only reserves ceil(deg / kSegmaxChunk) chunk slots for it and moves on.
//   chunks:  persistent warps reduce one chunk of one hub each into a partial row.
//   combine: one warp per hub takes the max over its partial rows.
// Max is exact and order-free, so every split gives the same bits; the only races are on the work cursors.  The reduction uses the
// float max (fmaxf / __hmax2), not an integer compare of the bit patterns: no sign or NaN assumption on x.
//
// The in-neighbourhood frontier S u N_in(S) of a row list (k_frontier_*) reads the same CSR: it marks a bitmap, splitting hub rows
// into the same chunks, and compacts it to ascending ids.  Full inference of a short list runs its hidden layers on these rows only.
//
// The out-neighbourhood frontier S u N_out(S) (k_out_frontier_*) and the suffix max (k_suffix_rows: the max over the edges appended
// to a row since a refresh, folded into the row's stored max) serve incremental inference (StreamingInference, plan.cu).
//
// The per-vertex cross entropy over full-inference logits (k_full_xent) lives here too: one warp per row, the logsumexp of the
// training loss (warp_logsumexp, sage_kernels.cuh).
#include "full_infer.cuh"
#include "sage_kernels.cuh"
#include <algorithm>

namespace ogl {

namespace {

constexpr int kBlock = 256;
constexpr int kInFlight = 8;        // edge rows loaded before the first compare

template <typename T> struct Strip;
template <> struct Strip<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ uint4 neg_inf() { return make_uint4(0xFF800000u, 0xFF800000u, 0xFF800000u, 0xFF800000u); }
  static __device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) { return __float_as_uint(fmaxf(__uint_as_float(a), __uint_as_float(b))); }
};
template <> struct Strip<tf32_t> : Strip<float> {};
template <> struct Strip<__half> {
  static constexpr int N = 8;
  static __device__ __forceinline__ uint4 neg_inf() { return make_uint4(0xFC00FC00u, 0xFC00FC00u, 0xFC00FC00u, 0xFC00FC00u); }
  static __device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) {
    const __half2 r = __hmax2(*reinterpret_cast<const __half2*>(&a), *reinterpret_cast<const __half2*>(&b));
    return *reinterpret_cast<const uint32_t*>(&r);
  }
};
template <> struct Strip<__nv_bfloat16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ uint4 neg_inf() { return make_uint4(0xFF80FF80u, 0xFF80FF80u, 0xFF80FF80u, 0xFF80FF80u); }
  static __device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) {
    const __nv_bfloat162 r = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
    return *reinterpret_cast<const uint32_t*>(&r);
  }
};

template <typename T>
__device__ __forceinline__ uint4 vmax(uint4 a, uint4 b) {
  return make_uint4(Strip<T>::max2(a.x, b.x), Strip<T>::max2(a.y, b.y), Strip<T>::max2(a.z, b.z), Strip<T>::max2(a.w, b.w));
}

// one warp: o[strips] = max over the cnt adjacency entries adj[0..cnt) of x[src], 0 if cnt == 0.  Merge (the suffix max): unless
// `replace`, o = max(o, that max) instead, and o is left alone when cnt == 0
template <typename T, bool Merge = false>
__device__ __forceinline__ void warp_row_max(const T* __restrict__ x, int ld, int strips, const unsigned long long* __restrict__ adj,
                                             int cnt, T* __restrict__ o, int lane, bool replace = true) {
  constexpr int NV = Strip<T>::N;
  for (int s0 = 0; s0 < strips; s0 += 32) {
    const int st = s0 + lane;
    const bool act = st < strips;
    uint4 acc = Strip<T>::neg_inf();
    for (int j0 = 0; j0 < cnt; j0 += 32) {
      const int m = min(32, cnt - j0);
      const uint32_t my_src = lane < m ? (uint32_t)__ldg(adj + j0 + lane) : 0u;     // low word of (eid << 32) | src
      int j = 0;
      for (; j + kInFlight <= m; j += kInFlight) {
        uint4 v[kInFlight];
#pragma unroll
        for (int u = 0; u < kInFlight; ++u) {
          const uint32_t src = __shfl_sync(0xffffffffu, my_src, j + u);
          if (act) v[u] = __ldg(reinterpret_cast<const uint4*>(x + (int64_t)src * ld) + st);
        }
#pragma unroll
        for (int u = 0; u < kInFlight; ++u)
          if (act) acc = vmax<T>(acc, v[u]);
      }
      for (; j < m; ++j) {
        const uint32_t src = __shfl_sync(0xffffffffu, my_src, j);
        if (act) acc = vmax<T>(acc, __ldg(reinterpret_cast<const uint4*>(x + (int64_t)src * ld) + st));
      }
    }
    if (act) {
      uint4* po = reinterpret_cast<uint4*>(o + (int64_t)st * NV);
      if (!Merge || replace) *po = cnt > 0 ? acc : make_uint4(0u, 0u, 0u, 0u);
      else if (cnt > 0) *po = vmax<T>(*po, acc);
    }
  }
}

template <typename T>
__device__ __forceinline__ void warp_zero_row(T* __restrict__ o, int strips, int lane) {
  for (int st = lane; st < strips; st += 32) *reinterpret_cast<uint4*>(o + (int64_t)st * Strip<T>::N) = make_uint4(0u, 0u, 0u, 0u);
}

__device__ __forceinline__ int64_t warp_next(unsigned long long* cursor, int lane) {
  unsigned long long r = 0;
  if (lane == 0) r = atomicAdd(cursor, 1ull);
  return (int64_t)__shfl_sync(0xffffffffu, r, 0);
}

template <typename T, typename Idx>
__global__ void __launch_bounds__(kBlock) k_csr_segmax_rows(GraphView gv, const T* __restrict__ x, int ld, int strips,
                                                            const Idx* __restrict__ rows, int64_t row0, int64_t n_rows, T* __restrict__ out, int ldo,
                                                            unsigned long long* __restrict__ ctl, SegmaxHub* __restrict__ hubs, int64_t hub_cap,
                                                            int32_t* __restrict__ chunk_hub, int64_t chunk_cap) {
  const int lane = threadIdx.x & 31;
  for (;;) {
    const int64_t r = warp_next(ctl + 0, lane);
    if (r >= n_rows) break;
    const int64_t v = rows ? (int64_t)rows[r] : row0 + r;
    T* o = out + r * (int64_t)ldo;
    if (v < 0 || v >= gv.n_vertices) { warp_zero_row(o, strips, lane); continue; }
    const int deg = gv.deg[v];
    const unsigned long long* adj = gv.adj + gv.row_start[v];
    if (deg > kSegmaxChunk) {
      // hub: reserve a record and ceil(deg / chunk) partial rows; if either list is full (only possible when the request lists
      // the same hub many times over) this warp reduces the row itself
      const int nch = (deg + kSegmaxChunk - 1) / kSegmaxChunk;
      long long h = -1, base = -1;
      if (lane == 0) {
        h = (long long)atomicAdd(ctl + 1, 1ull);
        if (h < hub_cap) {
          base = (long long)atomicAdd(ctl + 2, (unsigned long long)nch);
          const bool ok = base + nch <= chunk_cap;
          hubs[h] = SegmaxHub{r, (int32_t)v, (int32_t)(ok ? base : 0), ok ? nch : 0, 0};
          if (!ok) {
            for (long long c = base; c < chunk_cap && c < base + nch; ++c) chunk_hub[c] = -1;
            base = -1;
          }
        }
      }
      base = __shfl_sync(0xffffffffu, base, 0);
      h = __shfl_sync(0xffffffffu, h, 0);
      if (base >= 0) {
        for (int c = lane; c < nch; c += 32) chunk_hub[base + c] = (int32_t)h;
        continue;
      }
    }
    warp_row_max(x, ld, strips, adj, deg, o, lane);
  }
}

// Suffix: the records are those of k_suffix_rows (r = the first edge of the suffix, the output row is the vertex)
template <typename T, bool Suffix = false>
__global__ void __launch_bounds__(kBlock) k_csr_segmax_chunks(GraphView gv, const T* __restrict__ x, int ld, int strips,
                                                              unsigned long long* __restrict__ ctl, const SegmaxHub* __restrict__ hubs,
                                                              const int32_t* __restrict__ chunk_hub, int64_t chunk_cap, T* __restrict__ partial,
                                                              int ldp) {
  const int lane = threadIdx.x & 31;
  const int64_t n = min((int64_t)ctl[2], chunk_cap);
  for (;;) {
    const int64_t c = warp_next(ctl + 3, lane);
    if (c >= n) break;
    const int h = chunk_hub[c];
    if (h < 0) continue;
    const SegmaxHub hb = hubs[h];
    const int64_t i = c - hb.base;
    const int deg = gv.deg[hb.v];
    const int e0 = (Suffix ? (int)hb.r : 0) + (int)(i * kSegmaxChunk);
    warp_row_max(x, ld, strips, gv.adj + gv.row_start[hb.v] + e0, min(kSegmaxChunk, deg - e0), partial + c * (int64_t)ldp, lane);
  }
}

// Suffix: the partial rows are combined into out[v] (kept unless the record's pad flag says the row is replaced)
template <typename T, bool Suffix = false>
__global__ void __launch_bounds__(kBlock) k_csr_segmax_combine(const unsigned long long* __restrict__ ctl, const SegmaxHub* __restrict__ hubs,
                                                               int64_t hub_cap, const T* __restrict__ partial, int ldp, int strips,
                                                               T* __restrict__ out, int ldo) {
  const int lane = threadIdx.x & 31;
  const int64_t n = min((int64_t)ctl[1], hub_cap);
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t h = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; h < n; h += warps) {
    const SegmaxHub hb = hubs[h];
    if (hb.n == 0) continue;
    uint4* o = reinterpret_cast<uint4*>(out + (Suffix ? (int64_t)hb.v : hb.r) * (int64_t)ldo);
    for (int st = lane; st < strips; st += 32) {
      uint4 acc = Strip<T>::neg_inf();
      for (int i = 0; i < hb.n; ++i)
        acc = vmax<T>(acc, __ldg(reinterpret_cast<const uint4*>(partial + (int64_t)(hb.base + i) * ldp) + st));
      if (Suffix && !hb.pad) acc = vmax<T>(acc, o[st]);
      o[st] = acc;
    }
  }
}

// ---- suffix segment max (csr_segmax_suffix): the rows pass of k_csr_segmax_rows over the edges [e0, deg) of each listed row, e0 =
// deg_prev[v] (0 and a replaced row when deg_prev[v] is 0 or past the degree).  A suffix of more than kSegmaxChunk edges goes to the
// chunk list as a hub record {r = e0, v, base, n, pad = replace}; the chunk and combine passes above then finish it.
template <typename T, typename Idx>
__global__ void __launch_bounds__(kBlock) k_suffix_rows(GraphView gv, const T* __restrict__ x, int ld, int strips, const Idx* __restrict__ rows,
                                                        int64_t row0, int64_t n_rows, const int64_t* __restrict__ deg_prev, T* __restrict__ acc,
                                                        int ldacc, unsigned long long* __restrict__ ctl, SegmaxHub* __restrict__ hubs,
                                                        int64_t hub_cap, int32_t* __restrict__ chunk_hub, int64_t chunk_cap) {
  const int lane = threadIdx.x & 31;
  for (;;) {
    const int64_t r = warp_next(ctl + 0, lane);
    if (r >= n_rows) break;
    const int64_t v = rows ? (int64_t)rows[r] : row0 + r;
    if (v < 0 || v >= gv.n_vertices) continue;
    const int deg = gv.deg[v];
    const int64_t prev = deg_prev[v];
    const bool replace = prev <= 0 || prev > deg;
    const int e0 = replace ? 0 : (int)prev, cnt = deg - e0;
    const unsigned long long* adj = gv.adj + gv.row_start[v] + e0;
    T* o = acc + v * (int64_t)ldacc;
    if (cnt > kSegmaxChunk) {
      const int nch = (cnt + kSegmaxChunk - 1) / kSegmaxChunk;
      long long h = -1, base = -1;
      if (lane == 0) {
        h = (long long)atomicAdd(ctl + 1, 1ull);
        if (h < hub_cap) {
          base = (long long)atomicAdd(ctl + 2, (unsigned long long)nch);
          const bool ok = base + nch <= chunk_cap;
          hubs[h] = SegmaxHub{e0, (int32_t)v, (int32_t)(ok ? base : 0), ok ? nch : 0, replace ? 1 : 0};
          if (!ok) {
            for (long long c = base; c < chunk_cap && c < base + nch; ++c) chunk_hub[c] = -1;
            base = -1;
          }
        }
      }
      base = __shfl_sync(0xffffffffu, base, 0);
      h = __shfl_sync(0xffffffffu, h, 0);
      if (base >= 0) {
        for (int c = lane; c < nch; c += 32) chunk_hub[base + c] = (int32_t)h;
        continue;
      }
    }
    warp_row_max<T, true>(x, ld, strips, adj, cnt, o, lane, replace);
  }
}

template <typename T>
int launch_suffix(const GraphView& gv, const void* x, int ld, int strips, const int32_t* rows32, const int64_t* rows64, int64_t row0,
                  int64_t n_rows, const int64_t* deg_prev, void* acc, int ldacc, SegmaxWs* ws, cudaStream_t s) {
  const int ldp = strips * Strip<T>::N;
  const int persistent = sm_count() * 8;
  const int rgrid = (int)std::min<int64_t>(persistent, ceil_div(n_rows, kBlock / 32));
  OGL_CUDA(cudaMemsetAsync(ws->ctl, 0, 4 * sizeof(unsigned long long), s));
  if (rows64)
    OGL_LAUNCH((k_suffix_rows<T, int64_t>), rgrid, kBlock, 0, s, gv, (const T*)x, ld, strips, rows64, row0, n_rows, deg_prev, (T*)acc, ldacc,
               ws->ctl, ws->hubs, ws->hub_cap, ws->chunk_hub, ws->chunk_cap);
  else
    OGL_LAUNCH((k_suffix_rows<T, int32_t>), rgrid, kBlock, 0, s, gv, (const T*)x, ld, strips, rows32, row0, n_rows, deg_prev, (T*)acc, ldacc,
               ws->ctl, ws->hubs, ws->hub_cap, ws->chunk_hub, ws->chunk_cap);
  OGL_LAUNCH((k_csr_segmax_chunks<T, true>), persistent, kBlock, 0, s, gv, (const T*)x, ld, strips, ws->ctl, ws->hubs, ws->chunk_hub,
             ws->chunk_cap, (T*)ws->partial, ldp);
  OGL_LAUNCH((k_csr_segmax_combine<T, true>), (int)std::min<int64_t>(persistent, ceil_div(ws->hub_cap, kBlock / 32)), kBlock, 0, s, ws->ctl,
             ws->hubs, ws->hub_cap, (const T*)ws->partial, ldp, strips, (T*)acc, ldacc);
  return OGL_OK;
}

template <typename T>
int launch_segmax(const GraphView& gv, const void* x, int ld, int strips, const int32_t* rows32, const int64_t* rows64, int64_t row0,
                  int64_t n_rows, void* out, int ldo, SegmaxWs* ws, cudaStream_t s) {
  const int ldp = strips * Strip<T>::N;
  const int persistent = sm_count() * 8;
  const int rgrid = (int)std::min<int64_t>(persistent, ceil_div(n_rows, kBlock / 32));
  OGL_CUDA(cudaMemsetAsync(ws->ctl, 0, 4 * sizeof(unsigned long long), s));
  if (rows64)
    OGL_LAUNCH((k_csr_segmax_rows<T, int64_t>), rgrid, kBlock, 0, s, gv, (const T*)x, ld, strips, rows64, row0, n_rows, (T*)out, ldo, ws->ctl,
               ws->hubs, ws->hub_cap, ws->chunk_hub, ws->chunk_cap);
  else
    OGL_LAUNCH((k_csr_segmax_rows<T, int32_t>), rgrid, kBlock, 0, s, gv, (const T*)x, ld, strips, rows32, row0, n_rows, (T*)out, ldo, ws->ctl,
               ws->hubs, ws->hub_cap, ws->chunk_hub, ws->chunk_cap);
  OGL_LAUNCH((k_csr_segmax_chunks<T>), persistent, kBlock, 0, s, gv, (const T*)x, ld, strips, ws->ctl, ws->hubs, ws->chunk_hub,
             ws->chunk_cap, (T*)ws->partial, ldp);
  OGL_LAUNCH((k_csr_segmax_combine<T>), (int)std::min<int64_t>(persistent, ceil_div(ws->hub_cap, kBlock / 32)), kBlock, 0, s, ws->ctl,
             ws->hubs, ws->hub_cap, (const T*)ws->partial, ldp, strips, (T*)out, ldo);
  return OGL_OK;
}

// ---- in-neighbourhood frontier S u N_in(S): mark a bitmap, then compact it to ascending ids (count -> scan -> ballot fill) ----
// seed: every listed row sets its bit; the lane that set it first owns the vertex and appends it to the distinct-row list, so a
// vertex listed many times is expanded once
template <typename Idx>
__global__ void __launch_bounds__(kBlock) k_frontier_seed(const Idx* __restrict__ rows, int64_t n, int64_t n_vertices, uint32_t* __restrict__ bits,
                                                          int32_t* __restrict__ uniq, unsigned long long* __restrict__ ctl) {
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); i0 < n; i0 += stride) {
    const int64_t i = i0 + lane;
    int64_t v = -1;
    bool first = false;
    if (i < n) {
      v = (int64_t)rows[i];
      if (v >= 0 && v < n_vertices) {
        const uint32_t b = 1u << (v & 31);
        first = !(atomicOr(bits + (v >> 5), b) & b);
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, first);
    if (!m) continue;
    unsigned long long base = 0;
    if (lane == __ffs(m) - 1) base = atomicAdd(ctl + 0, (unsigned long long)__popc(m));
    base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
    if (first) uniq[base + __popc(m & ((1u << lane) - 1))] = (int32_t)v;
  }
}

// one warp sets the bits of the sources adj[0..cnt); a bit already set costs a load, not an atomic (hub sources recur)
__device__ __forceinline__ void warp_mark_sources(const unsigned long long* __restrict__ adj, int cnt, uint32_t* __restrict__ bits, int lane) {
  for (int j = lane; j < cnt; j += 32) {
    const uint32_t u = (uint32_t)__ldg(adj + j);
    const uint32_t b = 1u << (u & 31);
    if (!(__ldcg(bits + (u >> 5)) & b)) atomicOr(bits + (u >> 5), b);
  }
}

// rows: persistent warps take distinct rows from a cursor and mark their sources; a row of more than kSegmaxChunk edges is a hub
// whose chunks go to the chunk list (if the list is full the warp marks the row itself)
__global__ void __launch_bounds__(kBlock) k_frontier_rows(GraphView gv, uint32_t* __restrict__ bits, const int32_t* __restrict__ uniq,
                                                          unsigned long long* __restrict__ ctl, int2* __restrict__ chunks, int64_t chunk_cap) {
  const int lane = threadIdx.x & 31;
  const int64_t n = (int64_t)ctl[0];
  for (;;) {
    const int64_t i = warp_next(ctl + 1, lane);
    if (i >= n) break;
    const int v = uniq[i];
    const int deg = gv.deg[v];
    const unsigned long long* adj = gv.adj + gv.row_start[v];
    if (deg > kSegmaxChunk) {
      const int nch = (deg + kSegmaxChunk - 1) / kSegmaxChunk;
      long long base = 0;
      if (lane == 0) base = (long long)atomicAdd(ctl + 2, (unsigned long long)nch);
      base = __shfl_sync(0xffffffffu, base, 0);
      const bool ok = base + nch <= chunk_cap;
      for (int c = lane; c < nch && base + c < chunk_cap; c += 32) chunks[base + c] = make_int2(ok ? v : -1, c * kSegmaxChunk);
      if (ok) continue;
    }
    warp_mark_sources(adj, deg, bits, lane);
  }
}

__global__ void __launch_bounds__(kBlock) k_frontier_chunks(GraphView gv, uint32_t* __restrict__ bits, unsigned long long* __restrict__ ctl,
                                                            const int2* __restrict__ chunks, int64_t chunk_cap) {
  const int lane = threadIdx.x & 31;
  const int64_t n = min((int64_t)ctl[2], chunk_cap);
  for (;;) {
    const int64_t c = warp_next(ctl + 3, lane);
    if (c >= n) break;
    const int2 ch = chunks[c];
    if (ch.x < 0) continue;
    warp_mark_sources(gv.adj + gv.row_start[ch.x] + ch.y, min(kSegmaxChunk, gv.deg[ch.x] - ch.y), bits, lane);
  }
}

__global__ void __launch_bounds__(kBlock) k_frontier_count(const uint32_t* __restrict__ bits, int64_t words, int32_t* __restrict__ counts) {
  for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < words; w += (int64_t)gridDim.x * blockDim.x) counts[w] = __popc(bits[w]);
}

// one warp per bitmap word, lane = bit: set bits go to out[offs[word] + rank among the word's set bits]; *cost += deg + 1 of each
template <typename OutIdx>
__global__ void __launch_bounds__(kBlock) k_frontier_fill(const uint32_t* __restrict__ bits, const int32_t* __restrict__ offs, int64_t words,
                                                          const int32_t* __restrict__ deg, OutIdx* __restrict__ out,
                                                          unsigned long long* __restrict__ cost) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  unsigned long long c = 0;
  for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < words; w += warps) {
    const uint32_t word = bits[w];
    if (!((word >> lane) & 1u)) continue;
    const int v = (int)(w * 32 + lane);
    out[offs[w] + __popc(word & ((1u << lane) - 1))] = (OutIdx)v;
    c += (unsigned long long)deg[v] + 1ull;
  }
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0 && c) atomicAdd(cost, c);
}

// ---- out-neighbourhood frontier S u N_out(S) (out_frontier): the CSR holds in-edges only, so every row outside S scans its own
// sources against the bitmap of S and joins the result bitmap (seeded with S) at the first hit.  Four 32-entry groups of the
// adjacency are loaded before the vote, then the warp stops if any lane hit.
__device__ __forceinline__ bool warp_any_source(const unsigned long long* __restrict__ adj, int cnt, const uint32_t* __restrict__ in, int lane) {
  constexpr int kGroups = 4;
  for (int j0 = 0; j0 < cnt; j0 += 32 * kGroups) {
    uint32_t u[kGroups];
#pragma unroll
    for (int k = 0; k < kGroups; ++k) {
      const int j = j0 + 32 * k + lane;
      u[k] = j < cnt ? (uint32_t)__ldg(adj + j) : 0xffffffffu;
    }
    bool hit = false;
#pragma unroll
    for (int k = 0; k < kGroups; ++k)
      if (u[k] != 0xffffffffu) hit |= (__ldg(in + (u[k] >> 5)) >> (u[k] & 31)) & 1u;
    if (__any_sync(0xffffffffu, hit)) return true;
  }
  return false;
}

// rows: persistent warps take every vertex from a cursor; a row of more than kSegmaxChunk edges is a hub whose chunks go to the chunk
// list (if the list is full the warp scans the row itself)
__global__ void __launch_bounds__(kBlock) k_out_frontier_rows(GraphView gv, const uint32_t* __restrict__ in, uint32_t* __restrict__ out,
                                                              unsigned long long* __restrict__ ctl, int2* __restrict__ chunks, int64_t chunk_cap) {
  const int lane = threadIdx.x & 31;
  for (;;) {
    const int64_t v = warp_next(ctl + 1, lane);
    if (v >= gv.n_vertices) break;
    if ((__ldg(in + (v >> 5)) >> (v & 31)) & 1u) continue;       // in S: already in the result
    const int deg = gv.deg[v];
    const unsigned long long* adj = gv.adj + gv.row_start[v];
    if (deg > kSegmaxChunk) {
      const int nch = (deg + kSegmaxChunk - 1) / kSegmaxChunk;
      long long base = 0;
      if (lane == 0) base = (long long)atomicAdd(ctl + 2, (unsigned long long)nch);
      base = __shfl_sync(0xffffffffu, base, 0);
      const bool ok = base + nch <= chunk_cap;
      for (int c = lane; c < nch && base + c < chunk_cap; c += 32) chunks[base + c] = make_int2(ok ? (int)v : -1, c * kSegmaxChunk);
      if (ok) continue;
    }
    if (warp_any_source(adj, deg, in, lane) && lane == 0) atomicOr(out + (v >> 5), 1u << (v & 31));
  }
}

__global__ void __launch_bounds__(kBlock) k_out_frontier_chunks(GraphView gv, const uint32_t* __restrict__ in, uint32_t* __restrict__ out,
                                                                unsigned long long* __restrict__ ctl, const int2* __restrict__ chunks,
                                                                int64_t chunk_cap) {
  const int lane = threadIdx.x & 31;
  const int64_t n = min((int64_t)ctl[2], chunk_cap);
  for (;;) {
    const int64_t c = warp_next(ctl + 3, lane);
    if (c >= n) break;
    const int2 ch = chunks[c];
    if (ch.x < 0) continue;
    const uint32_t b = 1u << (ch.x & 31);
    if (__ldcg(out + (ch.x >> 5)) & b) continue;                 // another chunk of the row already hit
    if (warp_any_source(gv.adj + gv.row_start[ch.x] + ch.y, min(kSegmaxChunk, gv.deg[ch.x] - ch.y), in, lane) && lane == 0)
      atomicOr(out + (ch.x >> 5), b);
  }
}

// loss[r] = logsumexp(logits[r, :C]) - logits[r, y], y = labels[v_r], v_r = rows[r] | row0 + r.  A v_r outside [0, n_vertices) reads
// vertex 0's label and sets bit 0 of *err; a label outside [0, C) gives NaN and sets bit 1.
template <typename Idx>
__global__ void __launch_bounds__(kBlock) k_full_xent(const float* __restrict__ logits, int ld, int C, const int32_t* __restrict__ labels,
                                                      const Idx* __restrict__ rows, int64_t row0, int64_t n, int64_t n_vertices,
                                                      float* __restrict__ loss, uint32_t* __restrict__ err) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
    int64_t v = rows ? (int64_t)rows[r] : row0 + r;
    uint32_t bits = 0;
    if (v < 0 || v >= n_vertices) {
      v = 0;
      bits |= 1u;
    }
    const float* l = logits + r * (int64_t)ld;
    const float lse = warp_logsumexp(l, C, lane);
    const int y = labels[v];
    const bool ok = y >= 0 && y < C;
    if (!ok) bits |= 2u;
    if (lane == 0) {
      loss[r] = ok ? lse - l[y] : __int_as_float(0x7fc00000);
      if (bits) atomicOr(err, bits);
    }
  }
}

}  // namespace

int full_xent(const float* logits, int ld, int C, const int32_t* labels, const int32_t* rows32, const int64_t* rows64, int64_t row0,
              int64_t n, int64_t n_vertices, float* loss, uint32_t* err, cudaStream_t s) {
  if (n <= 0) return OGL_OK;
  const int grid = (int)std::min<int64_t>(ceil_div(n, kBlock / 32), (int64_t)sm_count() * 16);
  if (rows64)
    OGL_LAUNCH(k_full_xent<int64_t>, grid, kBlock, 0, s, logits, ld, C, labels, rows64, row0, n, n_vertices, loss, err);
  else
    OGL_LAUNCH(k_full_xent<int32_t>, grid, kBlock, 0, s, logits, ld, C, labels, rows32, row0, n, n_vertices, loss, err);
  return OGL_OK;
}

void frontier_ws_free(FrontierWs* ws) {
  for (void* q : {(void*)ws->bits, (void*)ws->bits_in, (void*)ws->uniq, (void*)ws->counts, (void*)ws->offs, (void*)ws->scan, (void*)ws->chunks, (void*)ws->ctl,
                  (void*)ws->out})
    cudaFree(q);
  *ws = FrontierWs();
}

int frontier_ws_reserve(FrontierWs* ws, int64_t n_vertices, int64_t n_edges) {
  const int64_t chunk_cap = 2 * (n_edges / kSegmaxChunk) + 64;
  if (ws->ctl && ws->v_cap >= n_vertices && ws->chunk_cap >= chunk_cap) return OGL_OK;
  const int64_t vc = std::max(n_vertices, ws->v_cap), cc = std::max(chunk_cap, ws->chunk_cap), words = ceil_div(vc, 32) + 1;
  frontier_ws_free(ws);
  if (cudaMalloc(&ws->bits, sizeof(uint32_t) * words) != cudaSuccess || cudaMalloc(&ws->bits_in, sizeof(uint32_t) * words) != cudaSuccess ||
      cudaMalloc(&ws->uniq, sizeof(int32_t) * vc) != cudaSuccess ||
      cudaMalloc(&ws->counts, sizeof(int32_t) * words) != cudaSuccess || cudaMalloc(&ws->offs, sizeof(int32_t) * words) != cudaSuccess ||
      cudaMalloc(&ws->scan, sizeof(int32_t) * scan_scratch_elems(words)) != cudaSuccess ||
      cudaMalloc(&ws->chunks, sizeof(int2) * cc) != cudaSuccess || cudaMalloc(&ws->ctl, 4 * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMalloc(&ws->out, sizeof(FrontierOut)) != cudaSuccess) {
    cudaGetLastError();
    frontier_ws_free(ws);
    set_error("in-neighbourhood frontier: cannot allocate the workspace of %lld vertices", (long long)vc);
    return OGL_ERR_CAPACITY;
  }
  ws->v_cap = vc; ws->chunk_cap = cc;
  return OGL_OK;
}

int in_frontier(const GraphView& gv, int64_t n_edges, const int32_t* rows32, const int64_t* rows64, int64_t n, int32_t* out_rows,
                FrontierWs* ws, cudaStream_t s) {
  OGL_TRY(frontier_ws_reserve(ws, gv.n_vertices, n_edges));
  const int64_t words = ceil_div(gv.n_vertices, 32);
  OGL_CUDA(cudaMemsetAsync(ws->bits, 0, sizeof(uint32_t) * words, s));
  OGL_CUDA(cudaMemsetAsync(ws->ctl, 0, 4 * sizeof(unsigned long long), s));
  OGL_CUDA(cudaMemsetAsync(ws->out, 0, sizeof(FrontierOut), s));
  if (n > 0) {
    const int persistent = sm_count() * 8;
    if (rows64)
      OGL_LAUNCH(k_frontier_seed<int64_t>, grid_for(n, kBlock), kBlock, 0, s, rows64, n, gv.n_vertices, ws->bits, ws->uniq, ws->ctl);
    else
      OGL_LAUNCH(k_frontier_seed<int32_t>, grid_for(n, kBlock), kBlock, 0, s, rows32, n, gv.n_vertices, ws->bits, ws->uniq, ws->ctl);
    OGL_LAUNCH(k_frontier_rows, (int)std::min<int64_t>(persistent, ceil_div(n, kBlock / 32)), kBlock, 0, s, gv, ws->bits, ws->uniq, ws->ctl,
               ws->chunks, ws->chunk_cap);
    OGL_LAUNCH(k_frontier_chunks, persistent, kBlock, 0, s, gv, ws->bits, ws->ctl, ws->chunks, ws->chunk_cap);
  }
  if (words == 0) return OGL_OK;
  OGL_LAUNCH(k_frontier_count, grid_for(words, kBlock), kBlock, 0, s, ws->bits, words, ws->counts);
  OGL_TRY(exclusive_scan_i32(ws->counts, ws->offs, words, ws->scan, &ws->out->n, s));
  OGL_LAUNCH(k_frontier_fill<int32_t>, grid_for(words * 32, kBlock), kBlock, 0, s, ws->bits, ws->offs, words, gv.deg, out_rows, &ws->out->cost);
  return OGL_OK;
}

int out_frontier(const GraphView& gv, int64_t n_edges, const int64_t* rows64, int64_t n, int32_t* out_rows32, int64_t* out_rows64,
                 FrontierWs* ws, cudaStream_t s) {
  OGL_TRY(frontier_ws_reserve(ws, gv.n_vertices, n_edges));
  const int64_t words = ceil_div(gv.n_vertices, 32);
  OGL_CUDA(cudaMemsetAsync(ws->bits_in, 0, sizeof(uint32_t) * words, s));
  OGL_CUDA(cudaMemsetAsync(ws->ctl, 0, 4 * sizeof(unsigned long long), s));
  OGL_CUDA(cudaMemsetAsync(ws->out, 0, sizeof(FrontierOut), s));
  if (words == 0) return OGL_OK;
  if (n > 0)
    OGL_LAUNCH(k_frontier_seed<int64_t>, grid_for(n, kBlock), kBlock, 0, s, rows64, n, gv.n_vertices, ws->bits_in, ws->uniq, ws->ctl);
  OGL_CUDA(cudaMemcpyAsync(ws->bits, ws->bits_in, sizeof(uint32_t) * words, cudaMemcpyDeviceToDevice, s));
  if (n > 0) {
    const int persistent = sm_count() * 8;
    OGL_LAUNCH(k_out_frontier_rows, persistent, kBlock, 0, s, gv, ws->bits_in, ws->bits, ws->ctl, ws->chunks, ws->chunk_cap);
    OGL_LAUNCH(k_out_frontier_chunks, persistent, kBlock, 0, s, gv, ws->bits_in, ws->bits, ws->ctl, ws->chunks, ws->chunk_cap);
  }
  OGL_LAUNCH(k_frontier_count, grid_for(words, kBlock), kBlock, 0, s, ws->bits, words, ws->counts);
  OGL_TRY(exclusive_scan_i32(ws->counts, ws->offs, words, ws->scan, &ws->out->n, s));
  if (out_rows64)
    OGL_LAUNCH(k_frontier_fill<int64_t>, grid_for(words * 32, kBlock), kBlock, 0, s, ws->bits, ws->offs, words, gv.deg, out_rows64,
               &ws->out->cost);
  else
    OGL_LAUNCH(k_frontier_fill<int32_t>, grid_for(words * 32, kBlock), kBlock, 0, s, ws->bits, ws->offs, words, gv.deg, out_rows32,
               &ws->out->cost);
  return OGL_OK;
}

void segmax_ws_free(SegmaxWs* ws) {
  cudaFree(ws->ctl); cudaFree(ws->hubs); cudaFree(ws->chunk_hub); cudaFree(ws->partial);
  *ws = SegmaxWs();
}

int segmax_ws_reserve(SegmaxWs* ws, int64_t n_edges, int64_t row_bytes) {
  // distinct hubs have > kSegmaxChunk edges each, and a hub of d edges takes ceil(d / chunk) <= 2 d / chunk slots
  const int64_t hub_cap = n_edges / kSegmaxChunk + 64, chunk_cap = 2 * (n_edges / kSegmaxChunk) + 64;
  if (ws->ctl && ws->hub_cap >= hub_cap && ws->chunk_cap >= chunk_cap && ws->row_bytes >= row_bytes) return OGL_OK;
  const int64_t hc = std::max(hub_cap, ws->hub_cap), cc = std::max(chunk_cap, ws->chunk_cap), rb = std::max(row_bytes, ws->row_bytes);
  segmax_ws_free(ws);
  if (cudaMalloc(&ws->ctl, 4 * sizeof(unsigned long long)) != cudaSuccess || cudaMalloc(&ws->hubs, sizeof(SegmaxHub) * hc) != cudaSuccess ||
      cudaMalloc(&ws->chunk_hub, sizeof(int32_t) * cc) != cudaSuccess || cudaMalloc(&ws->partial, (size_t)(cc * rb)) != cudaSuccess) {
    cudaGetLastError();
    segmax_ws_free(ws);
    set_error("segment max: cannot allocate the hub workspace (%lld partial rows of %lld bytes)", (long long)cc, (long long)rb);
    return OGL_ERR_CAPACITY;
  }
  ws->hub_cap = hc; ws->chunk_cap = cc; ws->row_bytes = rb;
  return OGL_OK;
}

int csr_segmax(int mode, const GraphView& gv, int64_t n_edges, const void* x, int ld, int cols, const int32_t* rows32,
               const int64_t* rows64, int64_t row0, int64_t n_rows, void* out, int ldo, SegmaxWs* ws, cudaStream_t s) {
  if (n_rows <= 0) return OGL_OK;
  const int nv = mode_vec(mode);
  const int strips = (cols + nv - 1) / nv;
  OGL_TRY(segmax_ws_reserve(ws, n_edges, (int64_t)strips * 16));
  OGL_MODE_DISPATCH(mode, OGL_TRY(launch_segmax<T>(gv, x, ld, strips, rows32, rows64, row0, n_rows, out, ldo, ws, s)));
  return OGL_OK;
}

int csr_segmax_suffix(int mode, const GraphView& gv, int64_t n_edges, const void* x, int ld, int cols, const int32_t* rows32,
                      const int64_t* rows64, int64_t row0, int64_t n, const int64_t* deg_prev, void* acc, int ldacc, SegmaxWs* ws, cudaStream_t s) {
  if (n <= 0) return OGL_OK;
  const int nv = mode_vec(mode);
  const int strips = (cols + nv - 1) / nv;
  OGL_TRY(segmax_ws_reserve(ws, n_edges, (int64_t)strips * 16));
  OGL_MODE_DISPATCH(mode, OGL_TRY(launch_suffix<T>(gv, x, ld, strips, rows32, rows64, row0, n, deg_prev, acc, ldacc, ws, s)));
  return OGL_OK;
}

}  // namespace ogl

using namespace ogl;

extern "C" int ogl_graph_segment_max(ogl_graph* g, int mode, const void* x_dev, int ld, int cols, const int64_t* rows_dev, int64_t n_rows,
                                     void* out_dev, int ldo, void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(g && mode_valid(mode), "ogl_graph_segment_max: bad arguments");
  OGL_ARG(graph_source_bound(g) == 0, "ogl_graph_segment_max: the graph is a destination shard (ogl_graph_set_source_bound): its sources "
          "are not rows of x");
  const GraphView gv = graph_view(g);
  OGL_ARG(rows_dev || n_rows == gv.n_vertices, "ogl_graph_segment_max: without a row list n_rows must be the vertex count %lld",
          (long long)gv.n_vertices);
  OGL_ARG(n_rows >= 0, "ogl_graph_segment_max: n_rows < 0");
  if (n_rows == 0) return OGL_OK;
  const int nv = mode_vec(mode);
  OGL_ARG(x_dev && out_dev && cols > 0 && cols <= ld && ld % nv == 0 && ldo % nv == 0 && (cols + nv - 1) / nv * nv <= ldo &&
              ((uintptr_t)x_dev & 15) == 0 && ((uintptr_t)out_dev & 15) == 0,
          "ogl_graph_segment_max: x / out must be 16-byte aligned with pitches ld, ldo multiples of %d elements and ldo >= cols rounded up to %d",
          nv, nv);
  cudaStream_t s = (cudaStream_t)stream;
  SegmaxWs ws;
  int r = csr_segmax(mode, gv, graph_num_edges(g), x_dev, ld, cols, nullptr, rows_dev, 0, n_rows, out_dev, ldo, &ws, s);
  if (r == OGL_OK && cudaStreamSynchronize(s) != cudaSuccess) {          // (the workspace is freed below)
    set_error("ogl_graph_segment_max: %s", cudaGetErrorString(cudaGetLastError()));
    r = OGL_ERR_CUDA;
  }
  segmax_ws_free(&ws);
  return r;
}

extern "C" int ogl_graph_in_frontier(ogl_graph* g, const int64_t* rows_dev, int64_t n, int32_t* out_rows_dev, int64_t* out_n,
                                     int64_t* out_edge_cost, void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(g && out_n && out_edge_cost && n >= 0 && (rows_dev || n == 0), "ogl_graph_in_frontier: bad arguments");
  OGL_ARG(graph_source_bound(g) == 0, "ogl_graph_in_frontier: the graph is a destination shard (ogl_graph_set_source_bound): its sources "
          "are not its rows");
  const GraphView gv = graph_view(g);
  OGL_ARG(out_rows_dev || gv.n_vertices == 0, "ogl_graph_in_frontier: null out_rows");
  cudaStream_t s = (cudaStream_t)stream;
  FrontierWs ws;
  FrontierOut h{};
  int r = in_frontier(gv, graph_num_edges(g), nullptr, rows_dev, n, out_rows_dev, &ws, s);
  if (r == OGL_OK && (cudaMemcpyAsync(&h, ws.out, sizeof(h), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
                      cudaStreamSynchronize(s) != cudaSuccess)) {
    set_error("ogl_graph_in_frontier: %s", cudaGetErrorString(cudaGetLastError()));
    r = OGL_ERR_CUDA;
  }
  frontier_ws_free(&ws);
  *out_n = h.n;
  *out_edge_cost = (int64_t)h.cost;
  return r;
}

extern "C" int ogl_graph_out_frontier(ogl_graph* g, const int64_t* rows_dev, int64_t n, int32_t* out_rows_dev, int64_t* out_n,
                                      int64_t* out_edge_cost, void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(g && out_n && out_edge_cost && n >= 0 && (rows_dev || n == 0), "ogl_graph_out_frontier: bad arguments");
  OGL_ARG(graph_source_bound(g) == 0, "ogl_graph_out_frontier: the graph is a destination shard (ogl_graph_set_source_bound): its sources "
          "are not its rows");
  const GraphView gv = graph_view(g);
  OGL_ARG(out_rows_dev || gv.n_vertices == 0, "ogl_graph_out_frontier: null out_rows");
  cudaStream_t s = (cudaStream_t)stream;
  FrontierWs ws;
  FrontierOut h{};
  int r = out_frontier(gv, graph_num_edges(g), rows_dev, n, out_rows_dev, nullptr, &ws, s);
  if (r == OGL_OK && (cudaMemcpyAsync(&h, ws.out, sizeof(h), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
                      cudaStreamSynchronize(s) != cudaSuccess)) {
    set_error("ogl_graph_out_frontier: %s", cudaGetErrorString(cudaGetLastError()));
    r = OGL_ERR_CUDA;
  }
  frontier_ws_free(&ws);
  *out_n = h.n;
  *out_edge_cost = (int64_t)h.cost;
  return r;
}

extern "C" int ogl_graph_segment_max_suffix(ogl_graph* g, int mode, const void* x_dev, int ld, int cols, const int64_t* rows_dev, int64_t n,
                                            const int64_t* deg_prev_dev, void* acc_dev, int ldacc, void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(g && mode_valid(mode) && n >= 0 && (rows_dev || n == 0) && (deg_prev_dev || n == 0), "ogl_graph_segment_max_suffix: bad arguments");
  OGL_ARG(graph_source_bound(g) == 0, "ogl_graph_segment_max_suffix: the graph is a destination shard (ogl_graph_set_source_bound): its "
          "sources are not rows of x");
  if (n == 0) return OGL_OK;
  const int nv = mode_vec(mode);
  OGL_ARG(x_dev && acc_dev && cols > 0 && cols <= ld && ld % nv == 0 && ldacc % nv == 0 && (cols + nv - 1) / nv * nv <= ldacc &&
              ((uintptr_t)x_dev & 15) == 0 && ((uintptr_t)acc_dev & 15) == 0,
          "ogl_graph_segment_max_suffix: x / acc must be 16-byte aligned with pitches ld, ldacc multiples of %d elements and ldacc >= cols "
          "rounded up to %d", nv, nv);
  cudaStream_t s = (cudaStream_t)stream;
  SegmaxWs ws;
  int r = csr_segmax_suffix(mode, graph_view(g), graph_num_edges(g), x_dev, ld, cols, nullptr, rows_dev, 0, n, deg_prev_dev, acc_dev, ldacc,
                            &ws, s);
  if (r == OGL_OK && cudaStreamSynchronize(s) != cudaSuccess) {          // (the workspace is freed below)
    set_error("ogl_graph_segment_max_suffix: %s", cudaGetErrorString(cudaGetLastError()));
    r = OGL_ERR_CUDA;
  }
  segmax_ws_free(&ws);
  return r;
}
