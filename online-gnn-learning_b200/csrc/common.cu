// Error plumbing, device checks and the deterministic 3-phase exclusive scan.
#include "common.cuh"
#include <stdarg.h>
#include <mutex>
#include <vector>

namespace ogl {

static thread_local char t_err[1024] = "";
std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_err, sizeof(t_err), fmt, ap);
  va_end(ap);
}

namespace {
struct Reader { const void *a, *b; cudaEvent_t ev; const void* owner; };
std::mutex g_readers_mu;
std::vector<Reader> g_readers;
}  // namespace
void readers_add(const void* res_a, const void* res_b, cudaEvent_t ev, const void* owner) {
  std::lock_guard<std::mutex> lk(g_readers_mu);
  for (auto& r : g_readers)
    if (r.ev == ev) { r.a = res_a; r.b = res_b; r.owner = owner; return; }
  g_readers.push_back({res_a, res_b, ev, owner});
}
void readers_remove(cudaEvent_t ev) {
  std::lock_guard<std::mutex> lk(g_readers_mu);
  for (size_t i = 0; i < g_readers.size(); ++i)
    if (g_readers[i].ev == ev) { g_readers.erase(g_readers.begin() + i); return; }
}
void readers_remove_owner(const void* owner) {
  std::lock_guard<std::mutex> lk(g_readers_mu);
  for (size_t i = g_readers.size(); i-- > 0;)
    if (g_readers[i].owner == owner) g_readers.erase(g_readers.begin() + i);
}
int readers_wait(const void* res, cudaStream_t s) {
  std::lock_guard<std::mutex> lk(g_readers_mu);
  for (auto& r : g_readers)
    if (r.a == res || r.b == res) OGL_CUDA(cudaStreamWaitEvent(s, r.ev, 0));
  return OGL_OK;
}

static int g_sm_count = 0;
int sm_count() {
  if (g_sm_count == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      g_sm_count = n;
    else
      return 148;
  }
  return g_sm_count;
}

int require_device() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    set_error("no CUDA device: %s (ogl_b200 has no CPU fallback)", cudaGetErrorString(e));
    return OGL_ERR_NODEVICE;
  }
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess || major != 10) {
    set_error("device %d is not sm_100 (compute capability major %d); ogl_b200 is built for sm_100a only", dev, major);
    return OGL_ERR_NODEVICE;
  }
  return OGL_OK;
}

// ---------------------------------------------------------------------------------------
// Exclusive scan: tiles of 2048 (256 threads x 8).  phase 1 tile sums, phase 2 scan of the
// sums (recursive), phase 3 tile scan + offset.  Deterministic (integer adds).
// ---------------------------------------------------------------------------------------
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

template <typename TO>
__device__ __forceinline__ TO block_exclusive_scan(TO v, TO* total, TO* smem /*>=9*/) {
  // exclusive scan of one value per thread across a 256-thread block
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  TO inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    TO t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) smem[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    TO w = lane < (kScanThreads / 32) ? smem[lane] : (TO)0;
    TO winc = w;
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
      TO t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    if (lane < (kScanThreads / 32)) smem[lane] = winc - w;
    if (lane == (kScanThreads / 32) - 1) smem[8] = winc;
  }
  __syncthreads();
  TO res = smem[warp] + inc - v;
  *total = smem[8];
  __syncthreads();
  return res;
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(kScanThreads) k_scan_tile_sums(const TI* __restrict__ in, TO* __restrict__ sums, int64_t n) {
  __shared__ TO smem[9];
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  TO acc = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < n) acc += (TO)in[base + i];
  TO total;
  block_exclusive_scan<TO>(acc, &total, smem);
  if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(kScanThreads) k_scan_tiles(const TI* in, TO* out,
                                                              const TO* offsets, int64_t n, TO* total_out) {
  __shared__ TO smem[9];
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  TO v[kScanItems];
  TO acc = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    v[i] = (base + i < n) ? (TO)in[base + i] : (TO)0;
    acc += v[i];
  }
  TO total;
  TO ex = block_exclusive_scan<TO>(acc, &total, smem);
  TO off = offsets ? offsets[blockIdx.x] : (TO)0;
  TO run = ex + off;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) out[base + i] = run;
    run += v[i];
  }
  if (total_out && blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) *total_out = off + total;
}

int64_t scan_scratch_elems(int64_t n_max) {
  int64_t total = 0, n = n_max;
  while (n > kScanTile) {
    n = ceil_div(n, kScanTile);
    total += n + 16;
  }
  return total + 16;
}

template <typename TI, typename TO>
static int scan_impl(const TI* in, TO* out, int64_t n, TO* scratch, TO* total_dev, cudaStream_t s) {
  if (n <= 0) {
    if (total_dev) OGL_CUDA(cudaMemsetAsync(total_dev, 0, sizeof(TO), s));
    return OGL_OK;
  }
  const int64_t nb = ceil_div(n, kScanTile);
  if (nb == 1) {
    OGL_LAUNCH((k_scan_tiles<TI, TO>), 1, kScanThreads, 0, s, in, out, (const TO*)nullptr, n, total_dev);
    return OGL_OK;
  }
  TO* sums = scratch;
  OGL_LAUNCH((k_scan_tile_sums<TI, TO>), (unsigned)nb, kScanThreads, 0, s, in, sums, n);
  // scan the sums in place (exclusive)
  OGL_TRY((scan_impl<TO, TO>(sums, sums, nb, scratch + nb + 16, nullptr, s)));
  OGL_LAUNCH((k_scan_tiles<TI, TO>), (unsigned)nb, kScanThreads, 0, s, in, out, (const TO*)sums, n, total_dev);
  return OGL_OK;
}

int exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, int32_t* scratch, int32_t* total_dev, cudaStream_t s) {
  return scan_impl<int32_t, int32_t>(in, out, n, scratch, total_dev, s);
}
int exclusive_scan_i32_to_i64(const int32_t* in, int64_t* out, int64_t n, int64_t* scratch, int64_t* total_dev, cudaStream_t s) {
  return scan_impl<int32_t, int64_t>(in, out, n, scratch, total_dev, s);
}

}  // namespace ogl

extern "C" {
const char* ogl_last_error(void) { return ogl::t_err; }
int ogl_version(void) { return 105; }
int64_t ogl_kernel_launches(void) { return (int64_t)ogl::g_launches.load(); }
}
