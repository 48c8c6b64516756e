// Host wrappers of the memory-bound GraphSAGE-pool kernels (see sage_kernels.cu).
#pragma once
#include "common.cuh"

namespace ogl {

// one weight matrix inside the flat fp32 parameter buffer and its shadows (ascending, non-overlapping)
struct ShadowSeg {
  int64_t begin, end;     // [begin, end) in the flat buffer = W [out, in] row-major
  int out, in, pitch_in, pitch_out;
  void* ws;               // W   [out, pitch_in]
  void* wt;               // W^T [in, pitch_out]
};

#ifdef __CUDACC__
// one element of Adam (torch.optim.Adam defaults as the reference uses them, pytorch/model.py:22-25); shared by the single-GPU
// kernel (sage_kernels.cu) and the peer-memory data-parallel kernel (peer.cu) so that both round identically
__device__ __forceinline__ float adam_math(float gi, float& mi, float& vi, float pi, float b1, float b2, float eps, float step, float isq) {
  mi = b1 * mi + (1.f - b1) * gi;
  vi = b2 * vi + (1.f - b2) * gi * gi;
  return pi - step * mi / (sqrtf(vi) * isq + eps);
}
// one warp: logsumexp of the row l[0..C), the same value on every lane; shared by the training loss (k_xent, sage_kernels.cu) and
// the full-inference loss (k_full_xent, full_infer.cu) so that equal logits give bit-equal losses
__device__ __forceinline__ float warp_logsumexp(const float* l, int C, int lane) {
  float mx = -INFINITY;
  for (int c = lane; c < C; c += 32) mx = fmaxf(mx, l[c]);
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float se = 0.f;
  for (int c = lane; c < C; c += 32) se += expf(l[c] - mx);
  for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
  return mx + logf(se);
}
#endif

int feat_write(int mode, const float* src, const int64_t* src_rows, int64_t n, int F, void* dst, int pitch, int64_t row0, cudaStream_t s,
               float scale = 1.f);
int label_write(const int64_t* src, const int64_t* src_rows, int64_t n, int32_t* dst, int64_t row0, cudaStream_t s);
int gather_rows(int mode, const void* table, int pitch, const int32_t* nodes, const int32_t* n_dev, int n_max, void* out, cudaStream_t s);
// table[nodes[r], :] = rows[r, :] for r < n (rows [n, pitch], table [*, pitch], both in the storage type; nodes distinct)
int scatter_rows(int mode, const void* rows, int pitch, const int32_t* nodes, int n, void* table, cudaStream_t s);
// in-place dropout of a layer's input rows (no-op for p == 0); step_dev = the optimiser step counter
int feat_drop(int mode, void* x, int pitch, int cols, const int32_t* n_dev, int n_max, float p, uint64_t seed, const uint32_t* step_dev,
              int layer, cudaStream_t s);
int segmax_fwd(int mode, const void* hp, int pitch, const int32_t* edge_lid, int fanout, const int32_t* n_dst_dev, int n_dst_max, void* ng,
               uint8_t* arg, cudaStream_t s);
int pool_bwd(int mode, const void* dng, int pitch, const uint8_t* arg, const int32_t* rev_ptr, const int32_t* rev_edge, int fanout,
             const int32_t* n_src_dev, int n_src_max, void* dhp, cudaStream_t s);
int64_t colsum_partial_elems(int n_max, int cols);
// out (and out2) = alpha * column sums
int colsum(int mode, const void* x, int pitch, int cols, const int32_t* n_dev, int n_max, float* partial, float* out, float* out2, cudaStream_t s,
           float alpha = 1.f);
int xent(int mode, const float* logits, int ldl, int C, const int32_t* labels, const int32_t* nodes, const int32_t* n_dev, int n_max,
         int rows_buf, float scale, float* per_loss, void* dlogits, int ldd, int want_grad, cudaStream_t s);
int sum_f32(const float* x, const int32_t* n_dev, int n_max, float* out, cudaStream_t s);
int adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float b1, float b2, float eps, uint32_t* t_dev, cudaStream_t s);
// Adam over the parameter range [lo, hi) (the step counter *t_dev is read, not advanced)
int adam_shadow(int mode, float* p, const float* g, float* m, float* v, int64_t lo, int64_t hi, float lr, float b1, float b2, float eps, uint32_t* t_dev,
                const ShadowSeg* segs_dev, int n_segs, cudaStream_t s);
int bump(uint32_t* a, uint32_t* b, cudaStream_t s);
int weight_shadow(int mode, const float* w, int out, int in, void* ws, int pitch_in, void* wt, int pitch_out, cudaStream_t s);
int unpad_copy(const float* src, int lds, int n_rows_max, const int32_t* n_dev, int cols, float* dst, cudaStream_t s);
int reduce_splits(const float* partial, int splits, int n, int k, float* c, int ldc, cudaStream_t s, float alpha = 1.f);
int reduce_splits_ld(const float* partial, int splits, int n, int k, int ldp, float* c, int ldc, cudaStream_t s);

}  // namespace ogl
