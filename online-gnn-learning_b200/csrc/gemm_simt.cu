// SIMT (FFMA) GEMMs with fp32 accumulation: the exact-arithmetic path (mode OGL_F32, rtol 1e-5)
// and the cross-check for the tcgen05 kernels (tests force it with gemm_impl=1).
#include "gemm.cuh"

namespace ogl {

constexpr int BM = 64, BN = 64, BK = 16, TM = 4, TN_ = 4;

template <typename T> __device__ __forceinline__ float ldf(const void* p, int64_t i) { return to_f32<T>(((const T*)p)[i]); }

template <typename TI, typename TO>
__global__ void __launch_bounds__(256) k_gemm_nt(GemmNT g) {
  __shared__ float As[BK][BM + 4];
  __shared__ float Bs[BK][BN + 4];
  const int m_dyn = g.m_dev ? min(*g.m_dev, g.m_max) : g.m_max;
  const int m_pad = g.zero_tail ? min((m_dyn + 127) / 128 * 128, g.m_max) : m_dyn;
  const int row0 = blockIdx.y * BM, col0 = blockIdx.x * BN;
  if (row0 >= m_pad) return;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  float acc[TM][TN_];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN_; ++j) acc[i][j] = 0.f;

  for (int seg = 0; seg < g.n_seg; ++seg) {
    const int K = g.k[seg];
    const int rows_valid = g.a_rows_dev[seg] ? min(*g.a_rows_dev[seg], m_dyn) : m_dyn;
    if (row0 >= rows_valid) continue;
    const void* A = g.a[seg];
    const void* B = g.b[seg];
    const int lda = g.lda[seg], ldb = g.ldb[seg];
    for (int k0 = 0; k0 < K; k0 += BK) {
      // 64x16 tile of A and of B, 4 elements per thread, k fastest
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int idx = threadIdx.x * 4 + e;
        const int r = idx / BK, kk = idx % BK;
        const int gm = row0 + r, gk = k0 + kk;
        As[kk][r] = (gm < rows_valid && gk < K) ? ldf<TI>(A, (int64_t)gm * lda + gk) : 0.f;
        const int gn = col0 + r;
        Bs[kk][r] = (gn < g.n && gk < K) ? ldf<TI>(B, (int64_t)gn * ldb + gk) : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < BK; ++kk) {
        float a[TM], b[TN_];
#pragma unroll
        for (int i = 0; i < TM; ++i) a[i] = As[kk][ty * TM + i];
#pragma unroll
        for (int j = 0; j < TN_; ++j) b[j] = Bs[kk][tx * TN_ + j];
#pragma unroll
        for (int i = 0; i < TM; ++i)
#pragma unroll
          for (int j = 0; j < TN_; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int gm = row0 + ty * TM + i;
    if (gm >= m_pad) continue;
#pragma unroll
    for (int j = 0; j < TN_; ++j) {
      const int gn = col0 + tx * TN_ + j;
      if (gn >= g.n) continue;
      float v = 0.f;
      if (gm < m_dyn) {
        v = acc[i][j] * g.alpha;
        if (g.bias) v += g.bias[gn];
        if (g.bias2) v += g.bias2[gn];
        if (g.relu) v = fmaxf(v, 0.f);
        if (g.mask && !(ldf<TI>(g.mask, (int64_t)gm * g.ldmask + gn) > 0.f)) v = 0.f;
      }
      ((TO*)g.c)[(int64_t)gm * g.ldc + gn] = from_f32<TO>(v);
    }
  }
}

// C[n,k] partial over a slice of rows m; gridDim.z = splits
template <typename TI>
__global__ void __launch_bounds__(256) k_gemm_tn(GemmTN g, int rows_per_split, float* __restrict__ out, int64_t out_stride) {
  __shared__ float As[BK][BM + 4];
  __shared__ float Bs[BK][BN + 4];
  const int m_dyn = g.m_dev ? min(*g.m_dev, g.m_max) : g.m_max;
  const int n0 = blockIdx.y * BM, k0 = blockIdx.x * BN;
  const int m_begin = blockIdx.z * rows_per_split;
  const int m_end = min(m_begin + rows_per_split, m_dyn);
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  float acc[TM][TN_];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN_; ++j) acc[i][j] = 0.f;
  for (int m0 = m_begin; m0 < m_end; m0 += BK) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = threadIdx.x * 4 + e;
      const int mm = idx / BM, c = idx % BM;      // c fastest: coalesced along n / k
      const int gm = m0 + mm;
      As[mm][c] = (gm < m_end && n0 + c < g.n) ? ldf<TI>(g.a, (int64_t)gm * g.lda + n0 + c) : 0.f;
      Bs[mm][c] = (gm < m_end && k0 + c < g.k) ? ldf<TI>(g.b, (int64_t)gm * g.ldb + k0 + c) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int mm = 0; mm < BK; ++mm) {
      float a[TM], b[TN_];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = As[mm][ty * TM + i];
#pragma unroll
      for (int j = 0; j < TN_; ++j) b[j] = Bs[mm][tx * TN_ + j];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN_; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* o = out + (int64_t)blockIdx.z * out_stride;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int gn = n0 + ty * TM + i;
    if (gn >= g.n) continue;
#pragma unroll
    for (int j = 0; j < TN_; ++j) {
      const int gk = k0 + tx * TN_ + j;
      if (gk < g.k) o[(int64_t)gn * g.k + gk] = acc[i][j];
    }
  }
}

// deterministic reduction of the split partials: c[n, ldc] = sum_z partial[z][n][k] (z ascending)
__global__ void __launch_bounds__(256) k_reduce_splits(const float* __restrict__ partial, int splits, int n, int k, float* __restrict__ c, int ldc,
                                                       float alpha) {
  const int64_t total = (int64_t)n * k;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int z = 0; z < splits; ++z) s += partial[(int64_t)z * total + i];
    c[(i / k) * ldc + (i % k)] = s * alpha;
  }
}

// partials with a padded row pitch ldp (tcgen05 TN kernel)
__global__ void __launch_bounds__(256) k_reduce_splits_ld(const float* __restrict__ partial, int splits, int n, int k, int ldp,
                                                          float* __restrict__ c, int ldc) {
  const int64_t total = (int64_t)n * k;
  const int64_t stride = (int64_t)n * ldp;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / k, col = i % k;
    float s = 0.f;
    for (int z = 0; z < splits; ++z) s += partial[(int64_t)z * stride + r * ldp + col];
    c[r * ldc + col] = s;
  }
}

// grouped form: blockIdx.y = problem; 16-byte loads of the partial rows (pitch % 4 == 0), fixed summation order
__global__ void __launch_bounds__(256) k_reduce_splits_group(const ReduceGroup g) {
  const ReduceGroup::Problem& q = g.pr[blockIdx.y];
  const int quads = q.ldp / 4;
  const int64_t total = (int64_t)q.n * quads;
  const int64_t stride = (int64_t)q.n * q.ldp;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / quads;
    const int col = (int)(i % quads) * 4;
    if (col >= q.k) continue;
    const float* src = q.partial + r * q.ldp + col;
    float4 acc = __ldcs(reinterpret_cast<const float4*>(src));
    for (int z = 1; z < g.splits; ++z) {
      const float4 x = __ldcs(reinterpret_cast<const float4*>(src + (int64_t)z * stride));
      acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
    }
    float* dst = q.c + r * q.ldc + col;
    const float al = q.alpha;
    dst[0] = acc.x * al;
    if (col + 1 < q.k) dst[1] = acc.y * al;
    if (col + 2 < q.k) dst[2] = acc.z * al;
    if (col + 3 < q.k) dst[3] = acc.w * al;
  }
}

int reduce_splits_group(const ReduceGroup& g, cudaStream_t s) {
  int64_t most = 1;
  for (int i = 0; i < g.count; ++i) {
    const int64_t t = (int64_t)g.pr[i].n * (g.pr[i].ldp / 4);
    if (t > most) most = t;
  }
  dim3 grid((unsigned)grid_for(most, 256), (unsigned)g.count);
  OGL_LAUNCH(k_reduce_splits_group, grid, 256, 0, s, g);
  return OGL_OK;
}

int reduce_splits_ld(const float* partial, int splits, int n, int k, int ldp, float* c, int ldc, cudaStream_t s) {
  OGL_LAUNCH(k_reduce_splits_ld, grid_for((int64_t)n * k, 256), 256, 0, s, partial, splits, n, k, ldp, c, ldc);
  return OGL_OK;
}

int reduce_splits(const float* partial, int splits, int n, int k, float* c, int ldc, cudaStream_t s, float alpha) {
  OGL_LAUNCH(k_reduce_splits, grid_for((int64_t)n * k, 256), 256, 0, s, partial, splits, n, k, c, ldc, alpha);
  return OGL_OK;
}

int gemm_nt_simt(const GemmNT& g, cudaStream_t s) {
  dim3 grid((unsigned)ceil_div(g.n, BN), (unsigned)ceil_div(g.m_max, BM));
  OGL_MODE_DISPATCH(g.mode, if (g.out_f32) OGL_LAUNCH((k_gemm_nt<T, float>), grid, 256, 0, s, g);
                            else OGL_LAUNCH((k_gemm_nt<T, T>), grid, 256, 0, s, g));
  return OGL_OK;
}

int gemm_tn_simt(const GemmTN& g, cudaStream_t s) {
  const int tiles = (int)(ceil_div(g.n, BM) * ceil_div(g.k, BN));
  int splits = (int)ceil_div(4 * sm_count(), tiles);
  const int max_by_rows = (int)ceil_div(g.m_max, 256);
  if (splits > max_by_rows) splits = max_by_rows;
  const int64_t per = (int64_t)g.n * g.k;
  if ((int64_t)splits * per > g.partial_elems) splits = (int)(g.partial_elems / per);
  if (splits < 1) { set_error("gemm_tn_simt: split workspace too small"); return OGL_ERR_ARG; }
  if (splits > 64) splits = 64;
  int rows_per_split = (int)ceil_div(g.m_max, splits);
  rows_per_split = (rows_per_split + BK - 1) / BK * BK;
  dim3 grid((unsigned)ceil_div(g.k, BN), (unsigned)ceil_div(g.n, BM), (unsigned)splits);
  OGL_MODE_DISPATCH(g.mode, OGL_LAUNCH((k_gemm_tn<T>), grid, 256, 0, s, g, rows_per_split, g.partial, per));
  return reduce_splits(g.partial, splits, g.n, g.k, g.c, g.ldc, s, g.alpha);
}

}  // namespace ogl
