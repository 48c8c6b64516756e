// Shared host/device utilities for the ogl_b200 library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>
#include "../../include/ogl_b200.h"

namespace ogl {

// ---- error plumbing (no exception crosses the C ABI) ---------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;

#define OGL_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      ogl::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return OGL_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

#define OGL_TRY(expr)               \
  do {                              \
    int _r = (expr);                \
    if (_r != OGL_OK) return _r;    \
  } while (0)

#define OGL_ARG(cond, ...)           \
  do {                               \
    if (!(cond)) {                   \
      ogl::set_error(__VA_ARGS__);   \
      return OGL_ERR_ARG;            \
    }                                \
  } while (0)

// launch + count + check
#define OGL_LAUNCH(kernel, grid, block, smem, stream, ...)                     \
  do {                                                                         \
    kernel<<<(grid), (block), (smem), (cudaStream_t)(stream)>>>(__VA_ARGS__);  \
    ogl::g_launches.fetch_add(1, std::memory_order_relaxed);                   \
    OGL_CUDA(cudaGetLastError());                                              \
  } while (0)

int require_device();   // OGL_OK iff an sm_100 device is current

// ---- readers of a graph / feature store that run on a stream of their own --------------------------------------------------
// A prefetched minibatch (plan.cu: ogl_plan_prefetch) samples the CSR and gathers feature rows on the plan's private stream,
// possibly long after the call returned.  It registers its completion event against the handles it reads; every entry point
// that MUTATES such a handle (edge / vertex insert, prefix activation, compaction, feature writes) first makes its own stream
// wait for the registered events, so a snapshot's evolve() can never run under a pending prefetch's feet.
void readers_add(const void* res_a, const void* res_b, cudaEvent_t ev, const void* owner);
void readers_remove(cudaEvent_t ev);
void readers_remove_owner(const void* owner);
int readers_wait(const void* res, cudaStream_t s);
int sm_count();

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int round_up(int a, int b) { return (a + b - 1) / b * b; }

// grid for an element-parallel kernel over n items: enough CTAs to cover, capped so that
// grid-stride loops run on a multiple of the SM count
static inline int grid_for(int64_t n, int block, int ctas_per_sm = 8) {
  int64_t need = ceil_div(n > 0 ? n : 1, block);
  int64_t cap = (int64_t)sm_count() * ctas_per_sm;
  return (int)(need < cap ? need : cap);
}

// ---- Philox4x32-10 (device twin of oracle/philox.py) ----------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += W0;
    k.y += W1;
  }
  return c;
}
__device__ __forceinline__ uint32_t pick4(const uint4& v, int i) {
  return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w));
}

// ---- device exclusive scan over int32 (3-phase, deterministic) ------------------------
// scratch must hold scan_scratch_elems(n_max) int32.
int64_t scan_scratch_elems(int64_t n_max);
// out[i] = sum_{j<i} in[j] for i < n (n static upper bound; caller zero-pads), total -> *total_dev (may be null)
int exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, int32_t* scratch, int32_t* total_dev, cudaStream_t s);
// 64-bit variant (graph compaction: offsets can exceed 2^31)
int exclusive_scan_i32_to_i64(const int32_t* in, int64_t* out, int64_t n, int64_t* scratch, int64_t* total_dev, cudaStream_t s);

// ---- dtype helpers ---------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
// mode OGL_FP16: fp16 storage (10 explicit mantissa bits, like TF32; overflow gives inf on purpose -- it must be loud)
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

// mode OGL_TF32: fp32 storage whose VALUE is rounded to TF32 (10 explicit mantissa bits, round to nearest) wherever a GEMM
// operand is produced, so that tcgen05.mma.kind::tf32 -- which drops the low 13 mantissa bits of what it reads -- sees it exactly
// (truncating unrounded fp32 inside the tensor core would bias every product towards zero by ~2^-11)
struct tf32_t { float v; };
__device__ __forceinline__ float round_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
template <> __device__ __forceinline__ float to_f32<tf32_t>(tf32_t v) { return v.v; }
template <> __device__ __forceinline__ tf32_t from_f32<tf32_t>(float v) { return tf32_t{round_tf32(v)}; }

// the arithmetic modes and their storage types: element bytes / elements per 16-byte vector
static inline int mode_valid(int mode) { return mode == OGL_F32 || mode == OGL_BF16 || mode == OGL_TF32 || mode == OGL_FP16; }
static inline int mode_is_16bit(int mode) { return mode == OGL_BF16 || mode == OGL_FP16; }
static inline int mode_bytes(int mode) { return mode_is_16bit(mode) ? 2 : 4; }
static inline int mode_vec(int mode) { return mode_is_16bit(mode) ? 8 : 4; }

// runs the statement(s) with T = the storage element type of mode: float (OGL_F32), __nv_bfloat16, __half, tf32_t (OGL_TF32)
#define OGL_MODE_DISPATCH(mode, ...)                                   \
  do {                                                                 \
    switch (mode) {                                                    \
      case OGL_BF16: { using T = __nv_bfloat16; __VA_ARGS__; } break;  \
      case OGL_FP16: { using T = __half; __VA_ARGS__; } break;         \
      case OGL_TF32: { using T = ogl::tf32_t; __VA_ARGS__; } break;    \
      default: { using T = float; __VA_ARGS__; } break;                \
    }                                                                  \
  } while (0)

}  // namespace ogl
