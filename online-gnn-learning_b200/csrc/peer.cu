// Gradient exchange of the data-parallel step over NVLink peer memory, fused with Adam (SURVEY 8(e): the only collective
// of the path is the sum of the flat fp32 gradient buffer over the ranks, followed by the replicated Adam update).
//
// Every rank keeps its gradient buffer in a device allocation of this library that every other rank of the box maps into its
// own address space (CUDA IPC over NVLink / NVSwitch).  ONE kernel per gradient bucket then does, on every rank:
//     arrive barrier (flags in peer memory)  ->  g[i] = sum over ranks r = 0 .. W-1 of grads_r[i]  (P2P loads, fixed rank order,
//     so every replica computes bit-identical weights)  ->  Adam on the local fp32 parameters + refresh of the bf16 W / W^T
//     shadows from the register  ->  "done reading" flags back to the peers.
// No NCCL call, no intermediate reduced buffer, no separate optimiser pass; the kernel uses no shared memory worth mentioning
// and few CTAs, so it is resident NEXT to the weight-gradient GEMM it overlaps (an NCCL all-reduce kernel takes whole SMs and
// pushes 3 of that GEMM's 135 one-wave CTAs into a second wave).
//
// Hazards: (1) a rank may only read its peers' gradients after they are final -> arrive barrier at kernel start, written with
// release / read with acquire at system scope after a __threadfence_system; (2) a rank may only overwrite its gradients (next
// step's backward) after every peer has finished reading them -> every kernel ends by publishing done[rank] = epoch to all
// peers, and ogl_peer_wait_readers (a one-warp kernel the caller enqueues before the next backward) waits for them.
#include "common.cuh"
#include "sage_kernels.cuh"
#include "peer.cuh"

namespace ogl {

namespace {

constexpr int kMaxWorld = 8;
constexpr int kFlagWords = 64;                    // per rank: arrive[8] | pad | done[8] | pad | cta counter
constexpr int kArrive = 0, kDone = 16, kCounter = 32, kEpoch = 34;
// kEpoch: exchanges this rank has completed.  The kernels take their epoch from this word (every CTA of a launch reads it before the
// launch's last CTA advances it), not from a kernel argument: an exchange can then sit inside a captured CUDA graph that is
// replayed every step
constexpr long long kSpinLimit = 20000000000ll;   // ~10 s of SM clocks: a missing peer traps instead of hanging the box

struct PeerView {
  const float* grads[kMaxWorld];
  uint32_t* flags[kMaxWorld];
  int rank, world;
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float ld_peer(const float* p) {       // never served from a stale line of this SM's L1
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_peer4(const float* p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void spin_until(const uint32_t* flag, uint32_t epoch) {
  const long long t0 = clock64();
  while ((int32_t)(ld_acquire_sys(flag) - epoch) < 0) {
    __nanosleep(40);
    if (clock64() - t0 > kSpinLimit) __trap();
  }
}

template <typename T>
__device__ __forceinline__ void shadow_one(int64_t i, float pi, const ShadowSeg* ss, int n_segs) {
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
// grads of [lo, hi): summed over the ranks in rank order, Adam (same arithmetic as k_adam_shadow) on the local replica.  Every rank
// loads every peer's gradients itself (W - 1 remote loads per element, one flag barrier).
template <typename T>
__global__ void __launch_bounds__(256) k_peer_sum_adam(const PeerView pv, int64_t lo, int64_t hi, float* __restrict__ p,
                                                       float* __restrict__ m, float* __restrict__ v, float lr, float b1, float b2, float eps,
                                                       const uint32_t* __restrict__ t_dev, const ShadowSeg* __restrict__ segs, int n_segs,
                                                       float* __restrict__ reduced_out) {
  __shared__ ShadowSeg ss[48];
  for (int i = threadIdx.x; i < n_segs; i += blockDim.x) ss[i] = segs[i];
  const uint32_t epoch = *((volatile const uint32_t*)(pv.flags[pv.rank] + kEpoch)) + 1u;
  // ---- arrive: my gradients are final (stream order) -> tell every peer, then wait for every peer
  if (blockIdx.x == 0 && threadIdx.x < pv.world) {
    __threadfence_system();
    st_release_sys(pv.flags[threadIdx.x] + kArrive + pv.rank, epoch);
  }
  if (threadIdx.x < pv.world) spin_until(pv.flags[pv.rank] + kArrive + threadIdx.x, epoch);
  __syncthreads();
  const uint32_t t = *t_dev + 1;
  const float bc1 = 1.f - powf(b1, (float)t), bc2 = 1.f - powf(b2, (float)t);
  const float step = lr / bc1, isq = rsqrtf(bc2);
  const int W = pv.world;
  // 16-byte body between the aligned bounds, scalar head / tail.  All W peer loads of a quad (and its m / v / p quads) are in flight
  // together: an NVLink round trip is paid once per quad, not once per rank
  const int64_t lo4 = (lo + 3) & ~(int64_t)3, hi4 = hi & ~(int64_t)3;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
  if (lo4 < hi4) {
    for (int64_t q = lo4 / 4 + tid; q < hi4 / 4; q += nth) {
      float4 gr[kMaxWorld];
#pragma unroll
      for (int r = 0; r < kMaxWorld; ++r)
        if (r < W) gr[r] = ld_peer4(pv.grads[r] + q * 4);
      float4 g = gr[0];
#pragma unroll
      for (int r = 1; r < kMaxWorld; ++r)
        if (r < W) { g.x += gr[r].x; g.y += gr[r].y; g.z += gr[r].z; g.w += gr[r].w; }
      float4 m4 = *reinterpret_cast<const float4*>(m + q * 4);
      float4 v4 = *reinterpret_cast<const float4*>(v + q * 4);
      float4 p4 = *reinterpret_cast<const float4*>(p + q * 4);
      if (reduced_out) *reinterpret_cast<float4*>(reduced_out + q * 4) = g;
      p4.x = adam_math(g.x, m4.x, v4.x, p4.x, b1, b2, eps, step, isq);
      p4.y = adam_math(g.y, m4.y, v4.y, p4.y, b1, b2, eps, step, isq);
      p4.z = adam_math(g.z, m4.z, v4.z, p4.z, b1, b2, eps, step, isq);
      p4.w = adam_math(g.w, m4.w, v4.w, p4.w, b1, b2, eps, step, isq);
      *reinterpret_cast<float4*>(m + q * 4) = m4;
      *reinterpret_cast<float4*>(v + q * 4) = v4;
      *reinterpret_cast<float4*>(p + q * 4) = p4;
      shadow_one<T>(q * 4 + 0, p4.x, ss, n_segs);
      shadow_one<T>(q * 4 + 1, p4.y, ss, n_segs);
      shadow_one<T>(q * 4 + 2, p4.z, ss, n_segs);
      shadow_one<T>(q * 4 + 3, p4.w, ss, n_segs);
    }
  }
  const int64_t head_end = lo4 < hi ? lo4 : hi, tail_begin = hi4 > head_end ? hi4 : head_end;
  for (int part = 0; part < 2; ++part) {
    const int64_t b0 = part ? tail_begin : lo, b1e = part ? hi : head_end;
    for (int64_t i = b0 + tid; i < b1e; i += nth) {
      float g = ld_peer(pv.grads[0] + i);
      for (int r = 1; r < W; ++r) g += ld_peer(pv.grads[r] + i);
      if (reduced_out) reduced_out[i] = g;
      float mi = m[i], vi = v[i];
      const float pi = adam_math(g, mi, vi, p[i], b1, b2, eps, step, isq);
      m[i] = mi; v[i] = vi; p[i] = pi;
      shadow_one<T>(i, pi, ss, n_segs);
    }
  }
  // ---- done: the last CTA of this rank tells every peer that their gradients have been read
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t* counter = pv.flags[pv.rank] + kCounter;
    __threadfence();
    const uint32_t old = atomicAdd(counter, 1u);
    if (old == gridDim.x - 1) {
      *counter = 0;
      pv.flags[pv.rank][kEpoch] = epoch;           // (every CTA of this launch has read the old value: they have all finished)
      __threadfence_system();
      for (int r = 0; r < W; ++r) st_release_sys(pv.flags[r] + kDone + pv.rank, epoch);
    }
  }
}

__global__ void k_peer_wait_done(const uint32_t* my_flags, int world) {
  const uint32_t epoch = *((volatile const uint32_t*)(my_flags + kEpoch));      // exchanges this rank has completed
  if (epoch != 0 && threadIdx.x < world) spin_until(my_flags + kDone + threadIdx.x, epoch);
}

}  // namespace

}  // namespace ogl

using namespace ogl;

struct ogl_peer {
  int rank = 0, world = 1;
  int64_t n_floats = 0;
  void* base = nullptr;                 // local allocation: [n_floats fp32 gradients | kFlagWords uint32 flags]
  size_t flags_off = 0;
  void* peer_base[kMaxWorld] = {};      // mapped peers (own slot = base)
  int opened[kMaxWorld] = {};
  int connected = 0;
  PeerView view;
};

extern "C" int ogl_peer_create(ogl_peer** out, int rank, int world, int64_t n_floats) {
  OGL_TRY(require_device());
  OGL_ARG(out && world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world && n_floats > 0,
          "ogl_peer_create: need 0 <= rank < world <= %d and n_floats > 0", kMaxWorld);
  ogl_peer* p = new ogl_peer();
  p->rank = rank; p->world = world; p->n_floats = n_floats;
  p->flags_off = ((size_t)n_floats * 4 + 255) / 256 * 256;
  OGL_CUDA(cudaMalloc(&p->base, p->flags_off + kFlagWords * 4));
  OGL_CUDA(cudaMemset(p->base, 0, p->flags_off + kFlagWords * 4));
  OGL_CUDA(cudaDeviceSynchronize());
  p->peer_base[rank] = p->base;
  if (world == 1) {
    p->connected = 1;
    p->view.rank = 0; p->view.world = 1;
    p->view.grads[0] = (const float*)p->base;
    p->view.flags[0] = (uint32_t*)((char*)p->base + p->flags_off);
  }
  *out = p;
  return OGL_OK;
}

extern "C" int ogl_peer_destroy(ogl_peer* p) {
  if (!p) return OGL_OK;
  cudaDeviceSynchronize();
  for (int r = 0; r < p->world; ++r)
    if (p->opened[r]) cudaIpcCloseMemHandle(p->peer_base[r]);
  cudaFree(p->base);
  delete p;
  return OGL_OK;
}

extern "C" int ogl_peer_handle(ogl_peer* p, void* handle64) {
  OGL_ARG(p && handle64, "ogl_peer_handle: null");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  OGL_CUDA(cudaIpcGetMemHandle(&h, p->base));
  memcpy(handle64, &h, 64);
  return OGL_OK;
}

static void finish_connect(ogl_peer* p) {
  p->view.rank = p->rank; p->view.world = p->world;
  for (int r = 0; r < p->world; ++r) {
    p->view.grads[r] = (const float*)p->peer_base[r];
    p->view.flags[r] = (uint32_t*)((char*)p->peer_base[r] + p->flags_off);
  }
  p->connected = 1;
}

extern "C" int ogl_peer_connect(ogl_peer* p, const void* handles) {
  OGL_ARG(p && handles, "ogl_peer_connect: null");
  for (int r = 0; r < p->world; ++r) {
    if (r == p->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)handles + 64 * r, 64);
    OGL_CUDA(cudaIpcOpenMemHandle(&p->peer_base[r], h, cudaIpcMemLazyEnablePeerAccess));
    p->opened[r] = 1;
  }
  finish_connect(p);
  return OGL_OK;
}

// ranks living in ONE process (tests on a single GPU, or one process driving several GPUs with peer access enabled)
extern "C" int ogl_peer_connect_local(ogl_peer* p, ogl_peer* const* all) {
  OGL_ARG(p && all, "ogl_peer_connect_local: null");
  for (int r = 0; r < p->world; ++r) {
    OGL_ARG(all[r] && all[r]->world == p->world && all[r]->rank == r && all[r]->n_floats == p->n_floats,
            "ogl_peer_connect_local: peer %d does not match", r);
    p->peer_base[r] = all[r]->base;
  }
  finish_connect(p);
  return OGL_OK;
}

extern "C" int ogl_peer_buffer(ogl_peer* p, float** grads_dev) {
  OGL_ARG(p && grads_dev, "ogl_peer_buffer: null");
  *grads_dev = (float*)p->base;
  return OGL_OK;
}

extern "C" int ogl_peer_wait_readers(ogl_peer* p, void* stream) {
  OGL_ARG(p && p->connected, "ogl_peer_wait_readers: not connected");
  OGL_LAUNCH(k_peer_wait_done, 1, 32, 0, stream, p->view.flags[p->rank], p->world);
  return OGL_OK;
}

namespace ogl {
int peer_wait_readers(ogl_peer* p, cudaStream_t s) { return ogl_peer_wait_readers(p, s); }
}

namespace ogl {

int peer_sum_adam(ogl_peer* p, const PeerAdamArgs& a, int64_t lo, int64_t hi, cudaStream_t s) {
  OGL_ARG(p && p->connected, "ogl_plan_peer_adam: peer group not connected");
  OGL_ARG(0 <= lo && lo < hi && hi <= p->n_floats, "ogl_plan_peer_adam: range [%lld, %lld) outside the %lld gradients", (long long)lo,
          (long long)hi, (long long)p->n_floats);
  OGL_ARG(a.grads == (const float*)p->base, "ogl_plan_peer_adam: the plan's gradient buffer is not this peer group's buffer");
  OGL_ARG(a.n_segs <= 48, "ogl_plan_peer_adam: too many weight segments");
  // at most 2 CTAs per SM: 2 KB of shared memory and 78 registers per thread, so the whole grid is resident NEXT to the
  // weight-gradient GEMM it overlaps (that kernel leaves ~35 KB of shared memory and 4/5 of the registers free)
  const int64_t quads = (hi - lo + 3) / 4;
  int grid = (int)ceil_div(quads, 256);
  if (grid > 2 * sm_count()) grid = 2 * sm_count();
  if (grid < 1) grid = 1;
  OGL_MODE_DISPATCH(a.mode, OGL_LAUNCH((k_peer_sum_adam<T>), grid, 256, 0, s, p->view, lo, hi, a.params, a.m, a.v, a.lr, a.b1, a.b2, a.eps,
                                       a.t_dev, a.segs, a.n_segs, a.reduced_out));
  return OGL_OK;
}

}  // namespace ogl
