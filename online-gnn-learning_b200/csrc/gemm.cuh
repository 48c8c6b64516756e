// Dense GEMM entry points of the GraphSAGE-pool path (SIMT fp32-accumulate + tcgen05 bf16 / fp16 / tf32).
// Operands are in the storage type of the arithmetic mode (common.cuh); in mode OGL_TF32 that is fp32 holding TF32-rounded values,
// which tcgen05 kind::tf32 reads exactly, as the SIMT path does.
#pragma once
#include "common.cuh"

namespace ogl {

// C[m, n] = act( sum_seg sum_k A_seg[m, k] * B_seg[n, k] + bias[n] ) , optional relu / mask.
// A, B row-major with the contraction index contiguous ("NT").  Up to two (A, B, K) segments
// accumulate into the same output (used for [h_self | neigh] x [W_self | W_neigh]^T).
//
// Rows read: with m = min(*m_dev, m_max) and rv_s = min(*a_rows_dev[s], m), segment s counts for rows m' < rv_s.  Rows
// [rv_s, round_up(rv_s, 128)) of A_s must be zero (the tile holding row rv_s multiplies them); rows at or past round_up(rv_s, 128)
// are never read, whatever they hold (a CTA pair whose second 128-row tile lies there loads it as zeros).  Columns >= k of A and
// B and rows >= n of B are never read either.
// Rows written: [0, m) the result, [m, round_up(m, 128)) zeros when zero_tail (clamped to m_max).  The tcgen05 epilogues that
// leave through TMA stores (16-bit outputs, TF32 activations) store whole 128-row tiles, 256-row tiles of a CTA pair: the rows past
// the zero tail up to round_up(that, 256) may receive zeros as well; rows past that are never written.  Columns [n, ldc) are not
// part of the result: the tcgen05 epilogues store zeros into those their 32- or 64-column boxes cover (all of them when
// ldc <= round_up(n, 32)), the SIMT kernel leaves them alone.
struct GemmNT {
  const void* a[2] = {nullptr, nullptr};   // element type = the mode's storage type
  int lda[2] = {0, 0};
  const void* b[2] = {nullptr, nullptr};
  int ldb[2] = {0, 0};
  int k[2] = {0, 0};
  int n_seg = 1;
  const int32_t* a_rows_dev[2] = {nullptr, nullptr};  // rows of segment s valid for m < *a_rows_dev[s] (nullptr: all)
  int a_rows_max[2] = {0, 0};      // rows that exist in segment s's buffer (0: m_max); reads beyond are zero-filled (TMA)
  int force_cg = 0;                // tcgen05 path: 0 = auto, 1 = single CTA, 2 = CTA pairs (cta_group::2)
  const float* bias = nullptr;     // [n] fp32 (nullable)
  const float* bias2 = nullptr;    // second bias added too (fc_self.bias + fc_neigh.bias)
  int relu = 0;
  float alpha = 1.f;               // scales the accumulated product before the bias (feat_drop's 1 / (1 - p) in the backward pass)
  const void* mask = nullptr;      // same shape/type as A-typed [m, ldmask]: out = mask>0 ? out : 0
  int ldmask = 0;
  void* c = nullptr;               // out_f32 ? f32 : the mode's storage type
  int ldc = 0;
  int m_max = 0;                   // static row bound (grid size)
  const int32_t* m_dev = nullptr;  // dynamic row count on device (nullptr: m_max)
  int n = 0;
  int mode = OGL_F32;              // arithmetic mode (OGL_F32 | OGL_BF16 | OGL_TF32 | OGL_FP16)
  int out_f32 = 0;                 // 1: plain fp32 output (logits); 0: the mode's storage type (OGL_TF32: TF32-rounded, a later operand)
  int zero_tail = 1;               // write zeros to rows [m, round_up(m, 128)) (contraction padding for later TN GEMMs)
};

// C[n, k] = sum_{m < *m_dev} A[m, n] * B[m, k]   (fp32 out; weight gradients)
// The tcgen05 kernel contracts whole 64-row blocks (32 in mode OGL_TF32): rows [m, round_up(m, 64)) of A must be zero (B may hold
// any finite values there); rows past round_up(m, 128), columns >= n of A and >= k of B are never read.
struct GemmTN {
  const void* a = nullptr;   // [m, lda], n contiguous
  int lda = 0;
  const void* b = nullptr;   // [m, ldb], k contiguous
  int ldb = 0;
  float* c = nullptr;        // [n, ldc]
  int ldc = 0;
  int n = 0, k = 0;
  int m_max = 0;
  const int32_t* m_dev = nullptr;
  int mode = OGL_F32;        // arithmetic mode: the operands' storage type
  float alpha = 1.f;         // C = alpha * A^T B (mode OGL_FP16: undoes the loss scale carried by the activation gradients)
  float* partial = nullptr;  // split workspace [splits, n, k]
  int64_t partial_elems = 0;
};

// tcgen05 when the mode has tensor-core operands (not OGL_F32), SIMT is not forced (force_simt: ogl_plan_config.gemm_impl != 0) and
// the driver supports it; the SIMT kernels otherwise
int gemm_nt(const GemmNT& g, int force_simt, cudaStream_t s);
// up to 4 weight-gradient GEMMs that contract over the same rows: one launch on the tcgen05 path
int gemm_tn_group(const GemmTN* g, int count, int force_simt, cudaStream_t s);
static inline int gemm_tn(const GemmTN& g, int force_simt, cudaStream_t s) { return gemm_tn_group(&g, 1, force_simt, s); }

int gemm_nt_simt(const GemmNT& g, cudaStream_t s);
int gemm_tn_simt(const GemmTN& g, cudaStream_t s);

// tcgen05 / TMA / TMEM versions (bf16, fp16 or tf32 operands, fp32 accumulate); same contracts
int gemm_nt_tc(const GemmNT& g, cudaStream_t s);
int gemm_tn_tc(const GemmTN& g, cudaStream_t s);
// up to 4 weight-gradient GEMMs contracting over the same rows (same m_dev / m_max) in one launch; g[0].partial is the workspace
int gemm_tn_tc_group(const GemmTN* g, int count, cudaStream_t s);

// deterministic reduction of the split partials of up to 4 problems in one launch: c = sum over z (ascending) of partial[z]
struct ReduceGroup {
  struct Problem { const float* partial; float* c; int n, k, ldp, ldc; float alpha; } pr[4];
  int count, splits;
};
int reduce_splits_group(const ReduceGroup& g, cudaStream_t s);
bool gemm_tc_available();

}  // namespace ogl
