// Memory-bound kernels of the GraphSAGE-pool layer: feature gather, segment max with argmax
// capture, argmax gradient scatter, bias-gradient column sums, cross-entropy, Adam.
// All are HBM-bound: 128-bit coalesced row accesses, device-side row counts (no host sync),
// grids sized from the SM count.
#include "sage_kernels.cuh"

namespace ogl {

constexpr int kBlock = 256;

template <typename T> struct Vec;           // 16-byte vector of T
template <> struct Vec<float> { static constexpr int N = 4; };
template <> struct Vec<__nv_bfloat16> { static constexpr int N = 8; };
template <> struct Vec<__half> { static constexpr int N = 8; };
template <> struct Vec<tf32_t> { static constexpr int N = 4; };

// two 16-bit elements in one register (the 16-bit storage types): the segment max and the max-pool backward are ISSUE-bound when they
// treat the eight elements of a strip one by one (ncu: 65-67 % issue-active, L2 / DRAM at 20-30 %), so they work on pairs
template <typename T> struct Pair;
template <> struct Pair<__half> {
  using type = __half2;
  static __device__ __forceinline__ type from_bits(uint32_t w) { return *reinterpret_cast<const type*>(&w); }
  static __device__ __forceinline__ uint32_t bits(type v) { return *reinterpret_cast<const uint32_t*>(&v); }
  static __device__ __forceinline__ float2 to_float2(uint32_t w) { return __half22float2(from_bits(w)); }
  static constexpr uint32_t kNegInf2 = 0xFC00FC00u;
};
template <> struct Pair<__nv_bfloat16> {
  using type = __nv_bfloat162;
  static __device__ __forceinline__ type from_bits(uint32_t w) { return *reinterpret_cast<const type*>(&w); }
  static __device__ __forceinline__ uint32_t bits(type v) { return *reinterpret_cast<const uint32_t*>(&v); }
  static __device__ __forceinline__ float2 to_float2(uint32_t w) { return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u)); }
  static constexpr uint32_t kNegInf2 = 0xFF80FF80u;
};

__device__ __forceinline__ int dyn_count(const int32_t* n_dev, int n_max) { return n_dev ? min(*n_dev, n_max) : n_max; }
__device__ __forceinline__ int pad128(int n, int n_max) { return min((n + 127) / 128 * 128, n_max); }

// ---- feature store -------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kBlock) k_feat_write(const float* __restrict__ src, const int64_t* __restrict__ src_rows, int64_t n, int F,
                                                       T* __restrict__ dst, int pitch, int64_t row0, float scale) {
  // one warp per row; fp32 -> T (times `scale`: the loss scale of mode OGL_FP16 when the rows are gradients), zero the pad columns
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
    const float* s = src + (src_rows ? src_rows[r] : r) * (int64_t)F;
    T* d = dst + (row0 + r) * (int64_t)pitch;
    for (int c = lane; c < pitch; c += 32) d[c] = from_f32<T>(c < F ? s[c] * scale : 0.f);
  }
}

__global__ void __launch_bounds__(kBlock) k_label_write(const int64_t* __restrict__ src, const int64_t* __restrict__ src_rows, int64_t n,
                                                        int32_t* __restrict__ dst, int64_t row0) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dst[row0 + i] = (int32_t)src[src_rows ? src_rows[i] : i];
}

// out[r, :] = table[nodes[r], :] for r < n; zero rows [n, pad128(n))
template <typename T>
__global__ void __launch_bounds__(kBlock) k_gather_rows(const T* __restrict__ table, int pitch, const int32_t* __restrict__ nodes,
                                                        const int32_t* __restrict__ n_dev, int n_max, T* __restrict__ out) {
  const int n = dyn_count(n_dev, n_max);
  const int np = pad128(n, n_max);
  const int vpr = pitch / Vec<T>::N;            // 16-byte vectors per row
  const int64_t total = (int64_t)np * vpr;
  const uint4* tb = reinterpret_cast<const uint4*>(table);
  uint4* ob = reinterpret_cast<uint4*>(out);
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(t / vpr), c = (int)(t % vpr);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (r < n) v = __ldg(tb + (int64_t)nodes[r] * vpr + c);
    ob[t] = v;
  }
}

// table[nodes[r], :] = rows[r, :] for r < n: the inverse of k_gather_rows (distinct nodes: no two rows race)
template <typename T>
__global__ void __launch_bounds__(kBlock) k_scatter_rows(const T* __restrict__ rows, int pitch, const int32_t* __restrict__ nodes, int n,
                                                         T* __restrict__ table) {
  const int vpr = pitch / Vec<T>::N;
  const int64_t total = (int64_t)n * vpr;
  const uint4* rb = reinterpret_cast<const uint4*>(rows);
  uint4* tb = reinterpret_cast<uint4*>(table);
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(t / vpr), c = (int)(t % vpr);
    tb[(int64_t)nodes[r] * vpr + c] = __ldg(rb + t);
  }
}

// ---- feat_drop: dropout of a layer's input rows, in place (training mode) ----------------------------------------------------
// graphsage_dgl.py:41-46 hands `dropout` to SAGEConv(feat_drop=...): the layer input is dropped ONCE and the same dropped rows
// feed h_self and fc_pool.  keep(r, c) = philox4x32_10(counter = (c >> 2, r, 0xD0 + layer, optimiser step), key = seed)[c & 3]
// >= p * 2^32; kept values are scaled by 1 / (1 - p) (torch.nn.Dropout).  oracle/sage.py:dropout_keep is the numpy twin.
template <typename T>
__global__ void __launch_bounds__(kBlock) k_feat_drop(T* __restrict__ x, int pitch, int cols, const int32_t* __restrict__ n_dev, int n_max,
                                                      uint32_t thresh, float scale, uint2 key, const uint32_t* __restrict__ step_dev,
                                                      uint32_t layer) {
  const int n = dyn_count(n_dev, n_max);
  const int qpr = (cols + 3) >> 2;
  const uint32_t step = *step_dev;
  const int64_t total = (int64_t)n * qpr;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(t / qpr), q = (int)(t % qpr);
    const uint4 w = philox4x32_10(make_uint4((uint32_t)q, (uint32_t)r, 0xD0u + layer, step), key);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = q * 4 + i;
      if (c < cols) {
        T* at = x + (int64_t)r * pitch + c;
        *at = from_f32<T>(pick4(w, i) >= thresh ? to_f32<T>(*at) * scale : 0.f);
      }
    }
  }
}

// ---- segment max over the fixed-fanout block (ELL layout), first-slot-wins argmax -----------------
template <typename T>
__global__ void __launch_bounds__(kBlock) k_segmax_fwd(const T* __restrict__ hp, int pitch, const int32_t* __restrict__ edge_lid, int fanout,
                                                       const int32_t* __restrict__ n_dst_dev, int n_dst_max, T* __restrict__ ng,
                                                       uint8_t* __restrict__ arg) {
  constexpr int NV = Vec<T>::N;
  const int n = dyn_count(n_dst_dev, n_dst_max);
  const int np = pad128(n, n_dst_max);
  const int vpr = pitch / NV;
  const int64_t total = (int64_t)np * vpr;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int d = (int)(t / vpr), c = (int)(t % vpr);
    if constexpr (NV == 8) {
      // 16-bit storage: pairs of elements per instruction -- mask = (x > best), best = max(best, x), slot = mask ? j : slot
      using P = Pair<T>;
      uint32_t best2[4], slot2[4];                 // slot2: one 16-bit lane per element
#pragma unroll
      for (int q = 0; q < 4; ++q) { best2[q] = P::kNegInf2; slot2[q] = 0x00ff00ffu; }
      bool any = false;
      if (d < n) {
        const int32_t* el = edge_lid + (int64_t)d * fanout;
        constexpr int kSlots = 5;
        for (int j0 = 0; j0 < fanout; j0 += kSlots) {
          int lid[kSlots];
          uint4 raw[kSlots];
#pragma unroll
          for (int u = 0; u < kSlots; ++u) lid[u] = (j0 + u < fanout) ? __ldg(el + j0 + u) : -1;
#pragma unroll
          for (int u = 0; u < kSlots; ++u)
            if (lid[u] >= 0) raw[u] = __ldg(reinterpret_cast<const uint4*>(hp + (int64_t)lid[u] * pitch) + c);
#pragma unroll
          for (int u = 0; u < kSlots; ++u) {
            if (lid[u] < 0) continue;
            const uint32_t jj = (uint32_t)(j0 + u) * 0x00010001u;
            const uint32_t w[4] = {raw[u].x, raw[u].y, raw[u].z, raw[u].w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const typename P::type x2 = P::from_bits(w[q]), b2 = P::from_bits(best2[q]);
              const uint32_t m = __hgt2_mask(x2, b2);        // strict >: the first slot attaining the maximum keeps it
              best2[q] = P::bits(__hmax2(b2, x2));
              slot2[q] = (slot2[q] & ~m) | (jj & m);
            }
            any = true;
          }
        }
      }
      if (!any) {
#pragma unroll
        for (int q = 0; q < 4; ++q) { best2[q] = 0u; slot2[q] = 0x00ff00ffu; }
      }
      *reinterpret_cast<uint4*>(ng + (int64_t)d * pitch + c * NV) = make_uint4(best2[0], best2[1], best2[2], best2[3]);
      if (d < n)
        *reinterpret_cast<uint2*>(arg + (int64_t)d * pitch + c * NV) =
            make_uint2(__byte_perm(slot2[0], slot2[1], 0x6420), __byte_perm(slot2[2], slot2[3], 0x6420));
    } else {
    float best[NV];
    uint8_t slot[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) { best[i] = 0.f; slot[i] = 255; }
    if (d < n) {
      bool any = false;
      const int32_t* el = edge_lid + (int64_t)d * fanout;
      // slots in chunks of kSlots: the chunk's row ids, then ALL of its row loads, are issued before the first compare (a thread's
      // loads are otherwise a chain of `fanout` dependent L2 round trips); slots are still compared in ascending order
      constexpr int kSlots = 5;
      for (int j0 = 0; j0 < fanout; j0 += kSlots) {
        int lid[kSlots];
        uint4 raw[kSlots];
#pragma unroll
        for (int u = 0; u < kSlots; ++u) lid[u] = (j0 + u < fanout) ? __ldg(el + j0 + u) : -1;
#pragma unroll
        for (int u = 0; u < kSlots; ++u)
          if (lid[u] >= 0) raw[u] = __ldg(reinterpret_cast<const uint4*>(hp + (int64_t)lid[u] * pitch) + c);
#pragma unroll
        for (int u = 0; u < kSlots; ++u) {
          if (lid[u] < 0) continue;
          const T* v = reinterpret_cast<const T*>(&raw[u]);
#pragma unroll
          for (int i = 0; i < NV; ++i) {
            const float x = to_f32<T>(v[i]);
            if (!any || x > best[i]) { best[i] = x; slot[i] = (uint8_t)(j0 + u); }
          }
          any = true;
        }
      }
    }
    T o[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) o[i] = from_f32<T>(best[i]);
    *reinterpret_cast<uint4*>(ng + (int64_t)d * pitch + c * NV) = *reinterpret_cast<const uint4*>(o);
    if (d < n) *reinterpret_cast<uint32_t*>(arg + (int64_t)d * pitch + c * NV) = *reinterpret_cast<const uint32_t*>(slot);
    }
  }
}

// Backward of the max-pool, source side:  dhp[s, f] = sum over sampled edges e = (d, slot j) with src(e) = s of
// (arg[d, f] == j) * dng[d, f].   The ReLU mask of hp is already folded into dng (dneigh GEMM epilogue, mask =
// neigh: neigh[d, f] is exactly hp[src(arg), f]).  Instead of scattering with atomics into an fp32 buffer and
// converting afterwards, every source row GATHERS over its reverse edge list (built at sampling time): dhp is
// written once, in the arithmetic type, with no atomics.  One thread per (row, 16-byte column strip); the dng /
// arg rows it re-reads (each destination row is visited once per slot) stay L2-resident.  Rows [n, pad128) = 0.
// (The fc_pool bias gradient needs no pass over dhp at all: every dng[d, f] lands in exactly one source row, so
// colsum(dhp) == colsum(dng).)
template <typename T>
__global__ void __launch_bounds__(kBlock) k_pool_bwd(const T* __restrict__ dng, int pitch, const uint8_t* __restrict__ arg,
                                                     const int32_t* __restrict__ rev_ptr, const int32_t* __restrict__ rev_edge, int fanout,
                                                     const int32_t* __restrict__ n_src_dev, int n_src_max, T* __restrict__ dhp) {
  constexpr int NV = Vec<T>::N;
  const int n = dyn_count(n_src_dev, n_src_max);
  const int np = pad128(n, n_src_max);
  const int vpr = pitch / NV;
  const int64_t total = (int64_t)np * vpr;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(t / vpr), strip = (int)(t % vpr);
    float sum[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) sum[i] = 0.f;
    if (r < n) {
      const int e0 = __ldg(rev_ptr + r), e1 = __ldg(rev_ptr + r + 1);
      // the list walk is a chain of dependent loads (offset -> edge -> rows): two edges are kept in flight at a time
      auto fetch = [&](int e, uint4& graw, uint2& sl, int& j) {      // sl: the strip's argmax slots, one byte per element
        const int d = e >> 8;                      // entry = (destination row << 8) | slot
        j = e & 255;
        const int64_t at = (int64_t)d * pitch + strip * NV;
        graw = __ldg(reinterpret_cast<const uint4*>(dng + at));
        if (NV == 8) sl = __ldg(reinterpret_cast<const uint2*>(arg + at));
        else sl = make_uint2(__ldg(reinterpret_cast<const uint32_t*>(arg + at)), 0u);
      };
      auto add = [&](const uint4& graw, const uint2& sl, int j) {
        // (packed variants -- byte-parallel slot compare, match flags widened to lane masks, pairs converted after an AND -- were
        // measured: 97-99 us against 87 us for this loop.  The conversions and fp32 adds are the same count either way, and the SIMD
        // video compares are emulated on this architecture)
        const T* gv = reinterpret_cast<const T*>(&graw);
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const uint32_t si = ((i < 4 ? sl.x : sl.y) >> (8 * (i & 3))) & 255u;
          if (si == (uint32_t)j) sum[i] += to_f32<T>(gv[i]);
        }
      };
      int k = e0;
      for (; k + 1 < e1; k += 2) {
        const int ea = __ldg(rev_edge + k), eb = __ldg(rev_edge + k + 1);
        uint4 ga, gb;
        uint2 sa, sb;
        int ja, jb;
        fetch(ea, ga, sa, ja);
        fetch(eb, gb, sb, jb);
        add(ga, sa, ja);
        add(gb, sb, jb);
      }
      if (k < e1) {
        uint4 ga;
        uint2 sa;
        int ja;
        fetch(__ldg(rev_edge + k), ga, sa, ja);
        add(ga, sa, ja);
      }
    }
    T o[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) o[i] = from_f32<T>(sum[i]);
    *reinterpret_cast<uint4*>(dhp + t * NV) = *reinterpret_cast<const uint4*>(o);
  }
}

// ---- bias gradient: deterministic two-phase column sum -------------------------------------------
// phase 1: a block covers 32 16-byte column strips x kColRows rows; warp w takes rows w, w+8, ...; the 8 warps are
// combined in shared memory in a fixed order.  phase 2 sums the per-chunk partials in ascending chunk order.
constexpr int kColRows = 256;
template <typename T>
__global__ void __launch_bounds__(kBlock) k_colsum_partial(const T* __restrict__ x, int pitch, int cols, const int32_t* __restrict__ n_dev,
                                                           int n_max, float* __restrict__ partial) {
  constexpr int NV = Vec<T>::N;
  __shared__ float sm[8][32][NV + 1];
  const int n = dyn_count(n_dev, n_max);
  const int chunk = blockIdx.y;
  const int r0 = chunk * kColRows, r1 = min(r0 + kColRows, n);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int strip = blockIdx.x * 32 + lane;
  const int vpr = pitch / NV;
  float acc[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) acc[i] = 0.f;
  if (strip < vpr) {
    for (int r = r0 + warp; r < r1; r += 8) {
      const uint4 raw = __ldg(reinterpret_cast<const uint4*>(x + (int64_t)r * pitch) + strip);
      const T* v = reinterpret_cast<const T*>(&raw);
#pragma unroll
      for (int i = 0; i < NV; ++i) acc[i] += to_f32<T>(v[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < NV; ++i) sm[warp][lane][i] = acc[i];
  __syncthreads();
  // 32 strips x NV columns = up to 256 outputs: one per thread
  const int o_strip = threadIdx.x / NV, o_i = threadIdx.x % NV;
  if (o_strip < 32) {
    const int c = (blockIdx.x * 32 + o_strip) * NV + o_i;
    if (c < cols) {
      float s_ = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) s_ += sm[w][o_strip][o_i];
      partial[(int64_t)chunk * cols + c] = s_;
    }
  }
}
__global__ void __launch_bounds__(1024) k_colsum_final(const float* __restrict__ partial, int cols, const int32_t* __restrict__ n_dev,
                                                       int n_max, float* __restrict__ out, float* __restrict__ out2, float alpha) {
  __shared__ float sm[32][33];
  const int n = dyn_count(n_dev, n_max);
  const int chunks = (n + kColRows - 1) / kColRows;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (c < cols)
    for (int k = warp; k < chunks; k += 32) s += partial[(int64_t)k * cols + c];
  sm[warp][lane] = s;
  __syncthreads();
  if (warp == 0 && c < cols) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 32; ++w) t += sm[w][lane];
    t *= alpha;                                   // (mode OGL_FP16: undoes the loss scale, a power of two)
    out[c] = t;
    if (out2) out2[c] = t;
  }
}

// ---- cross entropy: per-vertex loss + dlogits (rows >= n zeroed up to the padded count); one warp per row -------
template <typename T>
__global__ void __launch_bounds__(kBlock) k_xent(const float* __restrict__ logits, int ldl, int C, const int32_t* __restrict__ labels,
                                                 const int32_t* __restrict__ nodes, const int32_t* __restrict__ n_dev, int n_max,
                                                 int rows_buf, float scale,
                                                 float* __restrict__ per_loss, T* __restrict__ dlogits, int ldd, int want_grad) {
  const int n = dyn_count(n_dev, n_max);
  const int nz = want_grad ? pad128(n, rows_buf) : n;
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < max(n, nz); r += warps) {
    if (r < n) {
      const float* l = logits + (int64_t)r * ldl;
      const float lse = warp_logsumexp(l, C, lane);
      const int y = labels[nodes[r]];
      if (per_loss && lane == 0) per_loss[r] = lse - l[y];
      if (want_grad) {
        T* d = dlogits + (int64_t)r * ldd;
        for (int c = lane; c < ldd; c += 32) {
          float g = 0.f;
          if (c < C) g = (expf(l[c] - lse) - (c == y ? 1.f : 0.f)) * scale;
          d[c] = from_f32<T>(g);
        }
      }
    } else if (want_grad) {
      T* d = dlogits + (int64_t)r * ldd;
      for (int c = lane; c < ldd; c += 32) d[c] = from_f32<T>(0.f);
    }
  }
}

// single CTA, fixed order: deterministic sum of the per-vertex losses
__global__ void __launch_bounds__(1024) k_sum_f32(const float* __restrict__ x, const int32_t* __restrict__ n_dev, int n_max, float* __restrict__ out) {
  __shared__ float s[32];
  const int n = dyn_count(n_dev, n_max);
  float a = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) a += x[i];
  for (int o = 16; o > 0; o >>= 1) a += __shfl_down_sync(0xffffffffu, a, o);
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x < 32) {
    a = s[threadIdx.x];
    for (int o = 16; o > 0; o >>= 1) a += __shfl_down_sync(0xffffffffu, a, o);
    if (threadIdx.x == 0) *out = a;
  }
}

// ---- Adam (torch.optim.Adam defaults, pytorch/model.py:25) on the flat fp32 buffers ---------------
__global__ void __launch_bounds__(kBlock) k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                                 int64_t n, float lr, float b1, float b2, float eps, uint32_t* __restrict__ t_dev) {
  const uint32_t t = *t_dev + 1;
  const float bc1 = 1.f - powf(b1, (float)t), bc2 = 1.f - powf(b2, (float)t);
  const float step = lr / bc1, isq = rsqrtf(bc2);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i];
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] -= step * mi / (sqrtf(vi) * isq + eps);
  }
}
// Adam + refresh of the arithmetic-type weight shadows (W [out, pitch(in)] and W^T [in, pitch(out)]) in one pass over
// the flat parameter buffer: the updated value is written to its shadow slots straight from the register.
template <typename T>
__global__ void __launch_bounds__(kBlock) k_adam_shadow(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                        float* __restrict__ v, int64_t lo, int64_t n, float lr, float b1, float b2, float eps,
                                                        const uint32_t* __restrict__ t_dev, const ShadowSeg* __restrict__ segs, int n_segs) {
  __shared__ ShadowSeg ss[48];
  for (int i = threadIdx.x; i < n_segs; i += blockDim.x) ss[i] = segs[i];
  __syncthreads();
  const uint32_t t = *t_dev + 1;
  const float bc1 = 1.f - powf(b1, (float)t), bc2 = 1.f - powf(b2, (float)t);
  const float step = lr / bc1, isq = rsqrtf(bc2);
  for (int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i];
    float mi = m[i], vi = v[i];
    const float pi = adam_math(gi, mi, vi, p[i], b1, b2, eps, step, isq);
    m[i] = mi;
    v[i] = vi;
    p[i] = pi;
    int sg = 0;
    while (sg < n_segs && i >= ss[sg].end) ++sg;
    if (sg < n_segs && i >= ss[sg].begin) {
      const ShadowSeg& q = ss[sg];
      const int64_t r = i - q.begin;
      const int o = (int)(r / q.in), c = (int)(r % q.in);
      ((T*)q.ws)[(int64_t)o * q.pitch_in + c] = from_f32<T>(pi);
      ((T*)q.wt)[(int64_t)c * q.pitch_out + o] = from_f32<T>(pi);
    }
  }
}
__global__ void k_bump(uint32_t* a, uint32_t* b) {
  if (a) *a += 1;
  if (b) *b += 1;
}

// weight shadows in the arithmetic type: W [out, pitch(in)] and W^T [in, pitch(out)]
template <typename T>
__global__ void __launch_bounds__(kBlock) k_weight_shadow(const float* __restrict__ w, int out, int in, T* __restrict__ ws, int pitch_in,
                                                          T* __restrict__ wt, int pitch_out) {
  const int64_t total = (int64_t)out * pitch_in;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int o = (int)(t / pitch_in), i = (int)(t % pitch_in);
    const float x = i < in ? w[(int64_t)o * in + i] : 0.f;
    ws[t] = from_f32<T>(x);
    if (wt && i < in) wt[(int64_t)i * pitch_out + o] = from_f32<T>(x);
  }
}

template <typename T>
__global__ void __launch_bounds__(kBlock) k_unpad_copy(const float* __restrict__ src, int lds, int n_rows_max, const int32_t* n_dev, int cols, float* __restrict__ dst) {
  const int n = dyn_count(n_dev, n_rows_max);
  const int64_t total = (int64_t)n * cols;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x)
    dst[t] = src[(t / cols) * lds + (t % cols)];
}

// ================================ host wrappers ====================================================
// mode: OGL_F32 (exact fp32), OGL_BF16, OGL_FP16, OGL_TF32 (fp32 storage, values rounded to TF32 where a GEMM operand is produced)
#define L2(K, grid, s, ...)                                                                      \
  do {                                                                                           \
    if (mode == OGL_BF16) OGL_LAUNCH((K<__nv_bfloat16>), grid, kBlock, 0, s, __VA_ARGS__);       \
    else if (mode == OGL_FP16) OGL_LAUNCH((K<__half>), grid, kBlock, 0, s, __VA_ARGS__);         \
    else if (mode == OGL_TF32) OGL_LAUNCH((K<tf32_t>), grid, kBlock, 0, s, __VA_ARGS__);         \
    else OGL_LAUNCH((K<float>), grid, kBlock, 0, s, __VA_ARGS__);                                \
  } while (0)
// the same with typed views of the void* arguments (T names the element type inside CALL)
#define L2T(K, grid, s, CALL)                                                                    \
  do {                                                                                           \
    if (mode == OGL_BF16) { using T = __nv_bfloat16; OGL_LAUNCH((K<T>), grid, kBlock, 0, s, CALL); } \
    else if (mode == OGL_FP16) { using T = __half; OGL_LAUNCH((K<T>), grid, kBlock, 0, s, CALL); }   \
    else if (mode == OGL_TF32) { using T = tf32_t; OGL_LAUNCH((K<T>), grid, kBlock, 0, s, CALL); }   \
    else { using T = float; OGL_LAUNCH((K<T>), grid, kBlock, 0, s, CALL); }                      \
  } while (0)
#define ARGS(...) __VA_ARGS__

int feat_write(int mode, const float* src, const int64_t* src_rows, int64_t n, int F, void* dst, int pitch, int64_t row0, cudaStream_t s,
               float scale) {
  if (n <= 0) return OGL_OK;
  const int grid = grid_for(n * 32, kBlock);
  L2T(k_feat_write, grid, s, ARGS(src, src_rows, n, F, (T*)dst, pitch, row0, scale));
  return OGL_OK;
}
int label_write(const int64_t* src, const int64_t* src_rows, int64_t n, int32_t* dst, int64_t row0, cudaStream_t s) {
  if (n <= 0) return OGL_OK;
  OGL_LAUNCH(k_label_write, grid_for(n, kBlock), kBlock, 0, s, src, src_rows, n, dst, row0);
  return OGL_OK;
}
int gather_rows(int mode, const void* table, int pitch, const int32_t* nodes, const int32_t* n_dev, int n_max, void* out, cudaStream_t s) {
  const int grid = grid_for((int64_t)n_max * pitch / 8, kBlock, 16);
  L2T(k_gather_rows, grid, s, ARGS((const T*)table, pitch, nodes, n_dev, n_max, (T*)out));
  return OGL_OK;
}
int scatter_rows(int mode, const void* rows, int pitch, const int32_t* nodes, int n, void* table, cudaStream_t s) {
  if (n <= 0) return OGL_OK;
  const int grid = grid_for((int64_t)n * pitch / 8, kBlock, 16);
  L2T(k_scatter_rows, grid, s, ARGS((const T*)rows, pitch, nodes, n, (T*)table));
  return OGL_OK;
}
int feat_drop(int mode, void* x, int pitch, int cols, const int32_t* n_dev, int n_max, float p, uint64_t seed, const uint32_t* step_dev,
              int layer, cudaStream_t s) {
  if (!(p > 0.f)) return OGL_OK;
  OGL_ARG(p < 1.f, "feat_drop: dropout probability must be in [0, 1)");
  const uint32_t thresh = (uint32_t)fmin(4294967295.0, floor((double)p * 4294967296.0));
  const float scale = 1.f / (1.f - p);
  const uint2 key = make_uint2((uint32_t)(seed & 0xffffffffu), (uint32_t)(seed >> 32));
  const int grid = grid_for((int64_t)n_max * ((cols + 3) / 4), kBlock, 16);
  L2T(k_feat_drop, grid, s, ARGS((T*)x, pitch, cols, n_dev, n_max, thresh, scale, key, step_dev, (uint32_t)layer));
  return OGL_OK;
}
int segmax_fwd(int mode, const void* hp, int pitch, const int32_t* edge_lid, int fanout, const int32_t* n_dst_dev, int n_dst_max, void* ng,
               uint8_t* arg, cudaStream_t s) {
  const int grid = grid_for((int64_t)n_dst_max * pitch / 8, kBlock, 16);
  L2T(k_segmax_fwd, grid, s, ARGS((const T*)hp, pitch, edge_lid, fanout, n_dst_dev, n_dst_max, (T*)ng, arg));
  return OGL_OK;
}
int pool_bwd(int mode, const void* dng, int pitch, const uint8_t* arg, const int32_t* rev_ptr, const int32_t* rev_edge, int fanout,
             const int32_t* n_src_dev, int n_src_max, void* dhp, cudaStream_t s) {
  const int grid = grid_for((int64_t)round_up(n_src_max, 128) * pitch / mode_vec(mode), kBlock, 32);
  L2T(k_pool_bwd, grid, s, ARGS((const T*)dng, pitch, arg, rev_ptr, rev_edge, fanout, n_src_dev, n_src_max, (T*)dhp));
  return OGL_OK;
}
int64_t colsum_partial_elems(int n_max, int cols) { return ceil_div(n_max, kColRows) * (int64_t)cols; }
int colsum(int mode, const void* x, int pitch, int cols, const int32_t* n_dev, int n_max, float* partial, float* out, float* out2, cudaStream_t s,
           float alpha) {
  dim3 grid((unsigned)ceil_div(pitch / mode_vec(mode), 32), (unsigned)ceil_div(n_max, kColRows));
  L2T(k_colsum_partial, grid, s, ARGS((const T*)x, pitch, cols, n_dev, n_max, partial));
  OGL_LAUNCH(k_colsum_final, (unsigned)ceil_div(cols, 32), 1024, 0, s, partial, cols, n_dev, n_max, out, out2, alpha);
  return OGL_OK;
}
int xent(int mode, const float* logits, int ldl, int C, const int32_t* labels, const int32_t* nodes, const int32_t* n_dev, int n_max,
         int rows_buf, float scale, float* per_loss, void* dlogits, int ldd, int want_grad, cudaStream_t s) {
  const int grid = grid_for((int64_t)(rows_buf > n_max ? rows_buf : n_max) * 32, kBlock);
  L2T(k_xent, grid, s, ARGS(logits, ldl, C, labels, nodes, n_dev, n_max, rows_buf, scale, per_loss, (T*)dlogits, ldd, want_grad));
  return OGL_OK;
}
int sum_f32(const float* x, const int32_t* n_dev, int n_max, float* out, cudaStream_t s) {
  OGL_LAUNCH(k_sum_f32, 1, 1024, 0, s, x, n_dev, n_max, out);
  return OGL_OK;
}
int adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float b1, float b2, float eps, uint32_t* t_dev, cudaStream_t s) {
  OGL_LAUNCH(k_adam, grid_for(n, kBlock), kBlock, 0, s, p, g, m, v, n, lr, b1, b2, eps, t_dev);
  return OGL_OK;
}
int adam_shadow(int mode, float* p, const float* g, float* m, float* v, int64_t lo, int64_t hi, float lr, float b1, float b2, float eps,
                uint32_t* t_dev, const ShadowSeg* segs_dev, int n_segs, cudaStream_t s) {
  OGL_ARG(n_segs <= 48, "adam_shadow: too many weight segments");
  OGL_ARG(lo >= 0 && hi > lo, "adam_shadow: empty range");
  const int grid = grid_for(hi - lo, kBlock);
  L2(k_adam_shadow, grid, s, p, g, m, v, lo, hi, lr, b1, b2, eps, t_dev, segs_dev, n_segs);
  return OGL_OK;
}
int bump(uint32_t* a, uint32_t* b, cudaStream_t s) {
  OGL_LAUNCH(k_bump, 1, 1, 0, s, a, b);
  return OGL_OK;
}
int weight_shadow(int mode, const float* w, int out, int in, void* ws, int pitch_in, void* wt, int pitch_out, cudaStream_t s) {
  const int grid = grid_for((int64_t)out * pitch_in, kBlock);
  L2T(k_weight_shadow, grid, s, ARGS(w, out, in, (T*)ws, pitch_in, (T*)wt, pitch_out));
  return OGL_OK;
}
int unpad_copy(const float* src, int lds, int n_rows_max, const int32_t* n_dev, int cols, float* dst, cudaStream_t s) {
  OGL_LAUNCH((k_unpad_copy<float>), grid_for((int64_t)n_rows_max * cols, kBlock), kBlock, 0, s, src, lds, n_rows_max, n_dev, cols, dst);
  return OGL_OK;
}

}  // namespace ogl

// ---- evaluation metrics on the device (train/graphsage/model.py:60-95: argmax -> confusion matrix -> macro-F1) -----------------
// one warp per vertex: argmax over the C logits with numpy's tie rule (first maximum), one atomic into cm[label][pred].
// Labels outside [0, C) (the "unknown" -1 of Elliptic) are skipped and counted in cm[C * C].
namespace ogl {
__global__ void __launch_bounds__(kBlock) k_eval_confusion(const float* __restrict__ logits, int ld, int64_t n, int C,
                                                           const int64_t* __restrict__ labels, unsigned long long* __restrict__ cm) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
    const float* l = logits + r * ld;
    float best = -INFINITY;
    int arg = 0x7fffffff;
    for (int c = lane; c < C; c += 32) {
      const float x = l[c];
      if (x > best || (arg == 0x7fffffff && !(x < best))) { best = x; arg = c; }      // strict >: the first maximum of this lane
    }
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
      if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
    }
    if (lane == 0) {
      const int64_t y = labels[r];
      if (y >= 0 && y < C && arg < C) atomicAdd(&cm[y * C + arg], 1ull);
      else atomicAdd(&cm[(int64_t)C * C], 1ull);
    }
  }
}
}  // namespace ogl

extern "C" int ogl_eval_confusion(const float* logits_dev, int ld, int64_t n, int n_classes, const int64_t* labels_dev,
                                  int64_t* cm_dev, void* stream) {
  OGL_TRY(ogl::require_device());
  OGL_ARG(n >= 0 && n_classes > 0 && ld >= n_classes && cm_dev && (n == 0 || (logits_dev && labels_dev)), "ogl_eval_confusion: bad arguments");
  if (n == 0) return OGL_OK;
  OGL_LAUNCH(ogl::k_eval_confusion, ogl::grid_for(n * 32, ogl::kBlock), ogl::kBlock, 0, stream, logits_dev, ld, n, n_classes, labels_dev,
             (unsigned long long*)cm_dev);
  return OGL_OK;
}
