// tcgen05 / TMA / TMEM GEMMs of the GraphSAGE-pool path (bf16, fp16 or tf32 operands, fp32 accumulation in tensor memory).
// Template parameter KIND: 0 = bf16, 2 = fp16 (both tcgen05.mma.kind::f16; only the operand-format field of the instruction
// descriptor and the epilogue's pack / mask conversions differ), 1 = tcgen05.mma.kind::tf32 on fp32 operands (mode OGL_TF32; `TF`
// inside the kernels): a 128-byte swizzle row then holds 32 contraction elements instead of 64 and one MMA contracts 8 instead of
// 16, so stages, descriptors and barriers are byte-identical.
//
// Two warp-specialised kernels: 128-byte-wide contraction stages moved by TMA (SWIZZLE_128B) into a shared-memory ring, producer and
// MMA warps that run warp-uniform loops and issue through elect.sync (see elect_one), tcgen05.mma with accumulators in TMEM
// (cta_group::2 CTA pairs for the large NT shapes), epilogue warps reading them back with tcgen05.ld and leaving through TMA stores:
//
//   k_gemm_nt_tc   C[m, n] = act(sum_seg A_seg[m, :] . B_seg[n, :] + bias)    both operands K-major.  Persistent CTAs
//                  (one per SM), two 256-column TMEM accumulators so the epilogue of tile i overlaps the MMAs of
//                  tile i+1.  Used for fc_pool (+bias+ReLU), [h_self | neigh] x [W_self | W_neigh]^T (two
//                  contraction segments into one accumulator), and the activation-gradient GEMMs (+ReLU mask).
//   k_gemm_tn_tc   C[n, k] = sum_m A[m, n] . B[m, k]   both operands MN-major (the contraction runs over the
//                  rows of two activation matrices): the weight-gradient GEMMs.  Split over m across CTAs, fp32
//                  partials reduced in a fixed order (deterministic).
//
// Row counts are read from device memory (no host sync); tiles beyond the dynamic row count are skipped.
// Descriptor encodings follow the PTX ISA "tcgen05 matrix / instruction descriptor" tables.
#include "gemm.cuh"
#include "sage_kernels.cuh"
#include <cuda.h>

namespace ogl {

namespace {

constexpr int BM = 128;          // UMMA M (rows of the output tile)
constexpr int BK = 64;           // contraction elements per stage = one 128-byte swizzle row of bf16
constexpr int BN_MAX = 256;      // UMMA N upper bound
constexpr int STAGES = 4;
constexpr int A_STAGE_BYTES = BM * BK * 2;        // 16 KB
constexpr int B_STAGE_BYTES = BN_MAX * BK * 2;    // 32 KB
constexpr int RING_BYTES = STAGES * (A_STAGE_BYTES + B_STAGE_BYTES);   // 192 KB
constexpr int STORE_BOX_BYTES = 32 * 128;                              // one TMA-store box: 32 rows x 128 B
constexpr int STORE_BYTES = 4 /*warps*/ * 2 /*buffers*/ * STORE_BOX_BYTES;   // 32 KB epilogue staging
constexpr int BIAS_BYTES = 2 * BN_MAX * 4;                              // per-accumulator bias slice
constexpr int TAIL_BYTES = 256;                                         // barriers + tmem slot
constexpr int SMEM_NT1 = RING_BYTES + STORE_BYTES + BIAS_BYTES + TAIL_BYTES;
// cta_group::2 variant of the NT kernel: a CTA pair shares one B tile (each CTA stages half of it), so a stage is
// 16 KB of A + 16 KB of B per CTA.  FIVE stages (160 KB): together with the staging boxes the CTA then leaves ~33 KB of
// the SM's shared memory free, so the small kernels of the side / prefetch streams (sampling, to_block, scans, column sums;
// all <= 9 KB) can be resident next to it instead of waiting for the GEMM to leave the SM
constexpr int STAGES2 = 5;
constexpr int B2_STAGE_BYTES = (BN_MAX / 2) * BK * 2;    // 16 KB
constexpr int RING2_BYTES = STAGES2 * (A_STAGE_BYTES + B2_STAGE_BYTES);
constexpr int SMEM_NT2 = RING2_BYTES + STORE_BYTES + BIAS_BYTES + TAIL_BYTES;
static_assert(SMEM_NT2 <= 232448, "exceeds the 227 KB per-CTA shared memory of sm_100");
// TN kernel: its epilogue starts after the last MMA has retired, so its staging boxes alias the (then idle) operand ring
constexpr int SMEM_TN = RING_BYTES + TAIL_BYTES;
static_assert(SMEM_NT1 <= 232448, "exceeds the 227 KB per-CTA shared memory of sm_100");
constexpr int THREADS = 288;     // TN kernel: warps 0, 6 (A halves) and 7, 8 (B halves) TMA producers, warp 1 MMA issuer + TMEM owner, warps 2-5 epilogue
constexpr int THREADS_NT = 384;  // NT kernel: the same roles with EIGHT epilogue warps (two per TMEM lane quarter, each taking
                                 // every other 64-column box) so that draining a tile stays well below the tile's MMA time,
                                 // and a second TMA producer (warp 10; see k_gemm_nt_tc)

// ------------------------------------------------------------------ PTX wrappers ----------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(a), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(map), "r"(smem_u32(src)), "r"(c0),
               "r"(c1), "r"(c2)
               : "memory");
}
// programmatic dependent launch: a GEMM launched with the attribute may start (barrier init, TMEM allocation, descriptor prefetch) while
// the kernel before it in the stream is still draining; everything that touches that kernel's results comes after this wait
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {     // descriptor fetch off the first load's critical path
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, 256;" ::: "memory"); }   // the 8 epilogue warps (NT kernel)
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// One elected lane of a CONVERGED warp (CUTLASS's elect_one_sync).  The producer and MMA warps run their loops with all 32 lanes
// and warp-uniform values and predicate only the asynchronous instructions with this: UTMALDG / UTCHMMA take their descriptors,
// coordinates and addresses from UNIFORM registers, and for code the compiler sees as thread-divergent (`if (lane == 0) { ... }`)
// it wraps every such instruction in a waterfall loop (ELECT + seven R2UR.BROADCAST + branch, ~140 clocks per MMA measured with
// the loads and the epilogue switched off -- more than the 128 clocks a 256 x 256 x 16 MMA takes, and ~500 per 16 KB TMA box:
// the "30 B/clk per issuing thread" of tools/exp/ingest_probe.cu).  With uniform control flow the operands stay in uniform
// registers and an issue costs a few clocks.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// a value the compiler can prove warp-uniform (lane 0's copy): loads from global / shared memory and inline-asm outputs are not
__device__ __forceinline__ int uniform(int v) { return __shfl_sync(0xffffffffu, v, 0); }
__device__ __forceinline__ uint32_t uniform(uint32_t v) { return __shfl_sync(0xffffffffu, v, 0); }

// ---- cta_group::2 (CTA pair) variants ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// both CTAs of the pair load into their own shared memory; the transaction bytes complete on the LEADER's barrier
// (shared::cluster address of the same offset in CTA rank 0: peer bit 24 cleared)
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {      // arrives on the barrier at this offset in BOTH CTAs
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_mma_tf32_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// one MMA of the kernel's flavour: CG = CTAs per tile (cta_group), TF = tf32 operands
template <int CG, int TF>
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (CG == 2) {
    if constexpr (TF) tc_mma_tf32_pair(d_tmem, a_desc, b_desc, idesc, accumulate);
    else tc_mma_bf16_pair(d_tmem, a_desc, b_desc, idesc, accumulate);
  } else {
    if constexpr (TF) tc_mma_tf32(d_tmem, a_desc, b_desc, idesc, accumulate);
    else tc_mma_bf16(d_tmem, a_desc, b_desc, idesc, accumulate);
  }
}
__device__ __forceinline__ void mbar_arrive_on_cta(uint64_t* bar, uint32_t cta) {   // arrive on the same-offset barrier of CTA `cta`
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(smem_u32(bar)), "r"(cta)
      : "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* slot) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(COLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_free_pair(uint32_t base) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS) : "memory");
}

__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n\t"
      "tcgen05.wait::ld.sync.aligned;"      // same asm block: consumers of r[] cannot be scheduled before the wait
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(COLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_free(uint32_t base) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS) : "memory");
}

// shared-memory matrix descriptor (sm_100 format: version 1 at bit 46, SWIZZLE_128B = 2 at bits 61-63)
//   K-major : rows of 128 B (64 bf16 of the contraction), 8-row groups 1024 B apart (SBO); LBO unused (1)
//   MN-major: 64-element (128 B) chunks of the M/N index, contraction rows 128 B apart, 8-row groups 1024 B
//             apart (SBO), next 64-element chunk `lbo` bytes apart
//   MN-major 32-bit (tf32) operands exist in ONE layout only: SWIZZLE_128B_BASE32B = 1 at bits 61-63 -- 128-byte rows swizzled in
//             32-byte units over groups of FOUR contraction rows (TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B); SBO = distance of the
//             4-row groups (512 B for dense rows), LBO = distance of the 32-element chunks
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type = 2) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | ((uint64_t)layout_type << 61);
}
// instruction descriptor for kind::f16 / kind::tf32: D = f32 (bits 4-5 = 1), A / B format at bits 7-9 / 10-12 (kind::f16: 0 = fp16,
// 1 = bf16; kind::tf32: 2 = tf32), majors at bits 15 / 16 (0 = K-major, 1 = MN-major), N >> 3 at bits 17-22, M >> 4 at bits 24-28.
// kind: the kernels' KIND (0 = bf16, 1 = tf32, 2 = fp16)
__device__ __forceinline__ uint32_t instr_desc(int m, int n, int a_mn_major, int b_mn_major, int kind = 0) {
  const uint32_t fmt = kind == 1 ? 2u : (kind == 2 ? 0u : 1u);
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

struct SmemLayout {
  uint8_t* a0;           // stage i of A at a0 + i * A_STAGE_BYTES
  uint8_t* b0;
  int b_stage_bytes;
  __device__ __forceinline__ uint8_t* a(int i) const { return a0 + i * A_STAGE_BYTES; }
  __device__ __forceinline__ uint8_t* b(int i) const { return b0 + i * b_stage_bytes; }
  uint8_t* store;        // [4 warps][2][STORE_BOX_BYTES] epilogue staging for TMA stores
  float* bias;           // [2][BN_MAX]
  uint64_t* full;        // [STAGES]
  uint64_t* empty;       // [STAGES]
  uint64_t* acc_full;    // [2]
  uint64_t* acc_empty;   // [2]
  uint32_t* tmem_slot;
};
__device__ __forceinline__ SmemLayout carve(uint8_t* base, int n_stages = STAGES, int b_stage_bytes = B_STAGE_BYTES,
                                            int ring_bytes = RING_BYTES, bool store_in_ring = false) {
  // the dynamic shared window of a kernel without static __shared__ starts 1024-byte aligned (SWIZZLE_128B atoms
  // need it); checked at run time instead of paying 1 KB of slack
  if ((smem_u32(base) & 1023u) != 0) __trap();
  SmemLayout s;
  s.a0 = base;
  s.b0 = base + n_stages * A_STAGE_BYTES;
  s.b_stage_bytes = b_stage_bytes;
  s.store = store_in_ring ? base : base + ring_bytes;
  uint8_t* tail = base + ring_bytes + (store_in_ring ? 0 : STORE_BYTES);
  s.bias = (float*)tail;                                   // (unused when store_in_ring: the TN kernel has no bias)
  uint64_t* bars = (uint64_t*)(tail + (store_in_ring ? 0 : BIAS_BYTES));
  s.full = bars;
  s.empty = bars + n_stages;
  s.acc_full = bars + 2 * n_stages;
  s.acc_empty = bars + 2 * n_stages + 2;
  s.tmem_slot = (uint32_t*)(bars + 2 * n_stages + 4);
  return s;
}

template <int KIND>
__device__ __forceinline__ uint32_t pack16(float lo, float hi) {          // two outputs in the 16-bit storage type of KIND
  if constexpr (KIND == 2) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  } else {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
}
template <int KIND>
__device__ __forceinline__ bool positive16(uint16_t bits) {              // value > 0 (NaN: false), bf16 and fp16 alike
  return (bits & 0x8000u) == 0 && (bits & 0x7fffu) != 0 && (bits & 0x7fffu) <= (KIND == 2 ? 0x7c00u : 0x7f80u);
}

// ------------------------------------------------------------------ NT kernel --------------------
struct NtParams {
  CUtensorMap ta[2], tb[2];
  CUtensorMap tc;               // bf16 output [m_max, ldc], box 64 x 32 (TMA store); unused for fp32 output
  int k[2];
  int n_seg;
  const int32_t* a_rows_dev[2];
  const int32_t* m_dev;
  int m_max;
  int n, bn, n_tiles;           // bn = TMA box rows of B / width of a full tile; the last tile may be narrower
  const float* bias;
  const float* bias2;
  int relu;
  float alpha;
  const void* mask;             // operand-typed (bf16 | fp32) [m, ldmask]
  int ldmask;
  void* c;
  int ldc;
  int out_bf16;                 // bf16 output through TMA stores
  int out_f32_tma;              // TF kernels: fp32 output through TMA stores (activations), rounded to TF32 if round_out
  int round_out;
  int zero_tail;
};

// CG = 1: one CTA per 128-row tile.  CG = 2: a CTA pair (cluster of 2, tcgen05 cta_group::2) computes a 256-row super
// tile: each CTA stages its own 128 rows of A and HALF of the B tile, the leader CTA issues UMMA M = 256 that reads
// both halves, each CTA keeps the accumulator of its own rows in its own TMEM and runs its own epilogue.  Per CTA a
// k-block then moves 32 KB instead of 48 KB through L2 -> SM, the limiter of the single-CTA kernel.
template <int CG, int KIND>
__global__ void __launch_bounds__(THREADS_NT, 1) k_gemm_nt_tc(const __grid_constant__ NtParams p) {
  constexpr int TF = KIND == 1 ? 1 : 0;
  constexpr int NST = CG == 2 ? STAGES2 : STAGES;
  constexpr int BKE = TF ? 32 : 64;               // contraction elements per stage = one 128-byte swizzle row
  constexpr int KI = TF ? 8 : 16;                 // contraction elements per tcgen05.mma
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const SmemLayout s = carve(smem_raw, NST, CG == 2 ? B2_STAGE_BYTES : B_STAGE_BYTES, CG == 2 ? RING2_BYTES : RING_BYTES);
  const int warp = uniform((int)(threadIdx.x >> 5)), lane = threadIdx.x & 31;
  const int rank = CG == 2 ? uniform((int)cluster_ctarank()) : 0;          // CTA rank inside the pair
  const int unit = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int n_units = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  const int m_dyn = uniform(p.m_dev ? min(*p.m_dev, p.m_max) : p.m_max);
  const int m_pad = p.zero_tail ? min((m_dyn + 127) / 128 * 128, p.m_max) : m_dyn;
  const int m_tiles = ((m_pad + BM - 1) / BM + CG - 1) / CG;      // row blocks of CG * 128 rows
  const int total_tiles = m_tiles * p.n_tiles;
  // i-th tile of this unit -> (row block mt, column tile nb), round robin over all (row block, column tile) pairs; false past the
  // unit's last tile
  auto tile_at = [&](int i, int& mt, int& nb) -> bool {
    const int t = unit + i * n_units;
    if (t >= total_tiles) return false;
    mt = t / p.n_tiles; nb = t % p.n_tiles;
    return true;
  };
  int rows_valid[2];
  rows_valid[0] = uniform(p.a_rows_dev[0] ? min(*p.a_rows_dev[0], m_dyn) : m_dyn);
  rows_valid[1] = uniform(p.n_seg > 1 ? (p.a_rows_dev[1] ? min(*p.a_rows_dev[1], m_dyn) : m_dyn) : 0);

  if (threadIdx.x == 32) {                        // (a lane of the MMA warp: off the barrier-initialising thread)
    for (int i = 0; i < p.n_seg; ++i) { prefetch_tensormap(&p.ta[i]); prefetch_tensormap(&p.tb[i]); }
    if (p.out_bf16 || p.out_f32_tma) prefetch_tensormap(&p.tc);
  }
  if (threadIdx.x == 0) {
    // full[]: two TMA producers (A | B), one expect_tx arrival each
    for (int i = 0; i < NST; ++i) { mbar_init(&s.full[i], 2); mbar_init(&s.empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&s.acc_full[i], 1); mbar_init(&s.acc_empty[i], 8 * CG); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (CG == 2) tmem_alloc_pair<512>(s.tmem_slot);
    else tmem_alloc<512>(s.tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();       // the peer's barriers are initialised before any remote arrive / TMA completes on them
  tc_fence_after();
  const uint32_t tmem_base = uniform(*s.tmem_slot);
  pdl_wait();                            // operands (and the output buffer's previous readers) belong to the preceding kernel
  pdl_trigger();                         // a GEMM behind this one cannot share an SM with it (shared memory): it takes each SM as this
                                         // kernel's CTA leaves it, instead of waiting for the whole grid

  // ===== TMA producers (in pair mode: in both CTAs, each for its own shared memory) =====
  // The A and the B boxes of a stage are issued by two producer warps (0 and 10), each with its own expect_tx arrival on the stage's
  // full barrier.  That split dates from the thread-divergent issue path, where every TMA instruction cost ~500 clocks of waterfall
  // (the "30 B/clk per issuing thread" of tools/exp/ingest_probe.cu); with elect_one() one producer does as well, the second is kept
  // because it costs nothing.  Warp 11 is idle.
  // (run by ALL lanes of a producer warp, converged; the copies themselves are issued by the elected lane)
  auto tma_producer = [&](bool a_boxes) {
    int stage = 0;
    uint32_t phase = 0;
    // bytes this producer lands per stage on the barrier the MMA issuer waits on (pair mode: both CTAs' boxes, on the leader's)
    const uint32_t tx = a_boxes ? (uint32_t)(CG * A_STAGE_BYTES) : (CG == 2 ? (uint32_t)(2 * (p.bn / 2) * 128) : (uint32_t)(p.bn * 128));
    int mt, nb;
    for (int it = 0; tile_at(it, mt, nb); ++it) {
      const int mb = mt * CG + rank;
      const int bn_tile = (nb == p.n_tiles - 1) ? ((p.n - nb * BN_MAX + 15) / 16 * 16) : p.bn;
      for (int seg = 0; seg < p.n_seg; ++seg) {
        if (mt * CG * BM >= rows_valid[seg]) continue;          // (pair-uniform: decided on the pair's first row)
        const int nkb = (p.k[seg] + BKE - 1) / BKE;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&s.empty[stage], phase ^ 1);
          if (elect_one()) {
            if (CG == 2) {
              if (rank == 0) mbar_expect_tx(&s.full[stage], tx);
              if (a_boxes) tma_load_2d_pair(s.a(stage), &p.ta[seg], &s.full[stage], kb * BKE, mb * BM);
              else tma_load_2d_pair(s.b(stage), &p.tb[seg], &s.full[stage], kb * BKE, nb * BN_MAX + rank * (bn_tile / 2));
            } else {
              mbar_expect_tx(&s.full[stage], tx);
              if (a_boxes) tma_load_2d(s.a(stage), &p.ta[seg], &s.full[stage], kb * BKE, mb * BM);
              else tma_load_2d(s.b(stage), &p.tb[seg], &s.full[stage], kb * BKE, nb * BN_MAX);
            }
          }
          __syncwarp();
          if (++stage == NST) { stage = 0; phase ^= 1; }
        }
      }
    }
  };
  if (warp == 0) {
    tma_producer(true);
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer (pair mode: the leader CTA only): the whole warp runs the loop, the elected lane issues =====
    if (rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      const int b_stage_bytes = CG == 2 ? B2_STAGE_BYTES : B_STAGE_BYTES;
      const uint64_t a_desc0 = smem_desc(smem_u32(s.a(0)), 16, 1024), b_desc0 = smem_desc(smem_u32(s.b(0)), 16, 1024);
      int mt, nb;
      for (int it = 0; tile_at(it, mt, nb); ++it) {
        const int bn_tile = (nb == p.n_tiles - 1) ? ((p.n - nb * BN_MAX + 15) / 16 * 16) : p.bn;
        const uint32_t idesc = instr_desc(BM * CG, bn_tile, 0, 0, KIND);
        mbar_wait(&s.acc_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN_MAX);
        uint32_t accumulate = 0;
        for (int seg = 0; seg < p.n_seg; ++seg) {
          if (mt * CG * BM >= rows_valid[seg]) continue;
          const int K = p.k[seg];
          const int nkb = (K + BKE - 1) / BKE;
          for (int kb = 0; kb < nkb; ++kb) {
            mbar_wait(&s.full[stage], phase);
            tc_fence_after();
            // descriptors of this stage: the 14-bit address field advances by 2 (= 32 bytes) per k step of one MMA (16 bf16 /
            // 8 tf32 elements); the issue loop is kept branch-free for full k-blocks so that the tensor pipe never waits on this thread
            const uint64_t ad = a_desc0 + (uint64_t)(stage * (A_STAGE_BYTES >> 4));
            const uint64_t bd = b_desc0 + (uint64_t)(stage * (b_stage_bytes >> 4));
            const int k_left = K - kb * BKE;
            if (elect_one()) {
              if (k_left >= BKE) {
                tc_mma<CG, TF>(d_tmem, ad, bd, idesc, accumulate);
                tc_mma<CG, TF>(d_tmem, ad + 2, bd + 2, idesc, 1);
                tc_mma<CG, TF>(d_tmem, ad + 4, bd + 4, idesc, 1);
                tc_mma<CG, TF>(d_tmem, ad + 6, bd + 6, idesc, 1);
              } else {
                const int n_ki = (k_left + KI - 1) / KI;
                for (int ki = 0; ki < n_ki; ++ki) tc_mma<CG, TF>(d_tmem, ad + 2 * ki, bd + 2 * ki, idesc, ki ? 1u : accumulate);
              }
              if (CG == 2) tc_commit_pair(&s.empty[stage]);
              else tc_commit(&s.empty[stage]);
            }
            __syncwarp();
            accumulate = 1;
            if (++stage == NST) { stage = 0; phase ^= 1; }
          }
        }
        if (elect_one()) {
          if (CG == 2) tc_commit_pair(&s.acc_full[acc]);
          else tc_commit(&s.acc_full[acc]);
        }
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp >= 10) {
    // ===== second TMA producer (warp 10): the B boxes =====
    if (warp == 10) tma_producer(false);
    __syncwarp();
  } else {
    // ===== epilogue: TMEM -> registers -> bias / ReLU / mask -> swizzled smem box -> TMA store =====
    const int quarter = warp & 3;                 // TMEM lanes [32*quarter, +32) are this warp's
    const int parity = (warp - 2) >> 2;           // which of the two warps of that quarter: takes boxes box_idx % 2 == parity
    const int epi_tid = (warp - 2) * 32 + lane;
    uint8_t* const buf = s.store + (warp - 2) * STORE_BOX_BYTES;      // one staging box per warp
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t boxes_issued = 0;
    int mt_e, nb;
    for (int it = 0; tile_at(it, mt_e, nb); ++it) {
      const int mb = mt_e * CG + rank;
      const int bn_tile = (nb == p.n_tiles - 1) ? ((p.n - nb * BN_MAX + 15) / 16 * 16) : p.bn;
      const int gm = mb * BM + quarter * 32 + lane;
      const bool row_store = gm < m_pad;
      const bool row_live = gm < m_dyn;
      const bool tile_live = mb * BM + BM <= m_dyn;
      const float relu_lo = p.relu ? 0.f : -INFINITY;
      const float alpha = p.alpha;
      // bias slice of this tile -> shared (broadcast reads below); double-buffered with the accumulator
      float* bias_s = s.bias + acc * BN_MAX;
      for (int j = epi_tid; j < bn_tile; j += 256) {
        const int gn = nb * BN_MAX + j;
        float bv = 0.f;
        if (gn < p.n) {
          if (p.bias) bv += __ldg(p.bias + gn);
          if (p.bias2) bv += __ldg(p.bias2 + gn);
        }
        bias_s[j] = bv;
      }
      epi_barrier();
      mbar_wait(&s.acc_full[acc], acc_phase);
      tc_fence_after();
      if (TF && p.out_f32_tma) {
        // fp32 activations of the tf32 mode: one 32 x 32 fp32 box (32 rows of 128 bytes) per step, TF32-rounded, TMA store
        for (int c0 = parity * 32; c0 < bn_tile; c0 += 64) {
          if (boxes_issued >= 1) {
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
          }
          if (p.mask) {                            // 32 x 32 fp32 mask box staged with coalesced 512-byte warp loads (see the bf16 path)
            const int rbase = mb * BM + quarter * 32, cbase = nb * BN_MAX + c0 + (lane & 7) * 4;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int r = i * 4 + (lane >> 3);
              uint4 mraw = make_uint4(0u, 0u, 0u, 0u);
              if (rbase + r < m_dyn && cbase < p.ldmask)
                mraw = __ldg(reinterpret_cast<const uint4*>((const float*)p.mask + (int64_t)(rbase + r) * p.ldmask + cbase));
              *reinterpret_cast<uint4*>(buf + r * 128 + (((lane & 7) ^ (r & 7)) << 4)) = mraw;
            }
            __syncwarp();
          }
          uint32_t r[32];
          tc_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN_MAX + c0), r);
          const int gn0 = nb * BN_MAX + c0;
          float v[32];
          if (tile_live && gn0 + 32 <= p.n) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 b4 = *reinterpret_cast<const float4*>(bias_s + c0 + q * 4);
              v[q * 4 + 0] = fmaxf(fmaf(__uint_as_float(r[q * 4 + 0]), alpha, b4.x), relu_lo);
              v[q * 4 + 1] = fmaxf(fmaf(__uint_as_float(r[q * 4 + 1]), alpha, b4.y), relu_lo);
              v[q * 4 + 2] = fmaxf(fmaf(__uint_as_float(r[q * 4 + 2]), alpha, b4.z), relu_lo);
              v[q * 4 + 3] = fmaxf(fmaf(__uint_as_float(r[q * 4 + 3]), alpha, b4.w), relu_lo);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              float x = 0.f;
              if (row_live && gn0 + j < p.n) x = fmaxf(fmaf(__uint_as_float(r[j]), alpha, bias_s[c0 + j]), relu_lo);
              v[j] = x;
            }
          }
          if (p.mask) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 mv = *reinterpret_cast<const float4*>(buf + lane * 128 + ((q ^ (lane & 7)) << 4));
              if (!(mv.x > 0.f)) v[q * 4 + 0] = 0.f;
              if (!(mv.y > 0.f)) v[q * 4 + 1] = 0.f;
              if (!(mv.z > 0.f)) v[q * 4 + 2] = 0.f;
              if (!(mv.w > 0.f)) v[q * 4 + 3] = 0.f;
            }
          }
          if (p.round_out) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = round_tf32(v[j]);
          }
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(buf + lane * 128 + ((q ^ (lane & 7)) << 4)) = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
          fence_async_smem();
          __syncwarp();
          if (elect_one()) {
            tma_store_2d(&p.tc, buf, nb * BN_MAX + c0, mb * BM + quarter * 32);
            tma_store_commit();
          }
          __syncwarp();
          ++boxes_issued;
        }
      } else if (!TF && p.out_bf16) {
        for (int c0 = parity * 64; c0 < bn_tile; c0 += 128) {
          if (boxes_issued >= 1) {                 // this warp's previous store has finished reading the staging box
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
          }
          if (p.mask) {
            // the 32 x 64 mask box of this warp goes through the staging buffer first: 8 fully coalesced 512-byte
            // warp loads (4 rows x 128 B each) instead of 32-sector row-per-thread loads; same XOR swizzle, and each
            // thread later overwrites only the chunks of its own row that it has already consumed
            const int rbase = mb * BM + quarter * 32, cbase = nb * BN_MAX + c0 + (lane & 7) * 8;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int r = i * 4 + (lane >> 3);
              uint4 mraw = make_uint4(0u, 0u, 0u, 0u);
              if (rbase + r < m_dyn && cbase < p.ldmask)
                mraw = __ldg(reinterpret_cast<const uint4*>((const __nv_bfloat16*)p.mask + (int64_t)(rbase + r) * p.ldmask + cbase));
              *reinterpret_cast<uint4*>(buf + r * 128 + (((lane & 7) ^ (r & 7)) << 4)) = mraw;
            }
            __syncwarp();
          }
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int cc = c0 + half * 32;
            if (cc >= bn_tile) break;              // columns >= bn_tile >= ldc are clipped by the TMA store
            uint32_t r[32];
            tc_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN_MAX + cc), r);
            const int gn0 = nb * BN_MAX + cc;
            float v[32];
            if (tile_live && gn0 + 32 <= p.n) {
              // interior chunk (every row live, every column < n): branch-free, bias through 16-byte shared loads
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float4 b4 = *reinterpret_cast<const float4*>(bias_s + cc + q * 4);
                v[q * 4 + 0] = fmaxf(fmaf(__uint_as_float(r[q * 4 + 0]), alpha, b4.x), relu_lo);
                v[q * 4 + 1] = fmaxf(fmaf(__uint_as_float(r[q * 4 + 1]), alpha, b4.y), relu_lo);
                v[q * 4 + 2] = fmaxf(fmaf(__uint_as_float(r[q * 4 + 2]), alpha, b4.z), relu_lo);
                v[q * 4 + 3] = fmaxf(fmaf(__uint_as_float(r[q * 4 + 3]), alpha, b4.w), relu_lo);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                float x = 0.f;
                if (row_live && gn0 + j < p.n) x = fmaxf(fmaf(__uint_as_float(r[j]), alpha, bias_s[cc + j]), relu_lo);
                v[j] = x;
              }
            }
            if (p.mask) {                          // mask box staged in `buf` (coalesced loads, see above)
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const uint4 raw = *reinterpret_cast<const uint4*>(buf + lane * 128 + (((half * 4 + q) ^ (lane & 7)) << 4));
                const uint16_t* mv = reinterpret_cast<const uint16_t*>(&raw);
#pragma unroll
                for (int j = 0; j < 8; ++j)
                  if (!positive16<KIND>(mv[j])) v[q * 8 + j] = 0.f;
              }
            }
            // row `lane` of the box, 16-byte chunk (half*4 + q) XOR-swizzled like TMA's SWIZZLE_128B
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              uint4 o;
              o.x = pack16<KIND>(v[q * 8 + 0], v[q * 8 + 1]);
              o.y = pack16<KIND>(v[q * 8 + 2], v[q * 8 + 3]);
              o.z = pack16<KIND>(v[q * 8 + 4], v[q * 8 + 5]);
              o.w = pack16<KIND>(v[q * 8 + 6], v[q * 8 + 7]);
              *reinterpret_cast<uint4*>(buf + lane * 128 + (((half * 4 + q) ^ (lane & 7)) << 4)) = o;
            }
          }
          fence_async_smem();
          __syncwarp();
          // rows >= m_pad of the tile receive zeros (never read: consumers stop at the padded count); rows >= m_max
          // and columns >= ldc are clipped by the tensor map
          if (elect_one()) {
            tma_store_2d(&p.tc, buf, nb * BN_MAX + c0, mb * BM + quarter * 32);
            tma_store_commit();
          }
          __syncwarp();
          ++boxes_issued;
        }
      } else {
        for (int c0 = parity * 32; c0 < bn_tile; c0 += 64) {
          uint32_t r[32];
          tc_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN_MAX + c0), r);
          const int gn0 = nb * BN_MAX + c0;
          if (row_store) {
            float* crow = (float*)p.c + (int64_t)gm * p.ldc + gn0;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              if (gn0 + q * 4 < p.ldc) {
                float v[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  float x = 0.f;
                  if (row_live && gn0 + q * 4 + j < p.n) {
                    x = fmaf(__uint_as_float(r[q * 4 + j]), alpha, bias_s[c0 + q * 4 + j]);
                    if (p.relu) x = fmaxf(x, 0.f);
                  }
                  v[j] = x;
                }
                reinterpret_cast<float4*>(crow)[q] = make_float4(v[0], v[1], v[2], v[3]);
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {                             // the accumulator is drained: tell the (leader's) MMA issuer
        if (CG == 2) mbar_arrive_on_cta(&s.acc_empty[acc], 0);
        else mbar_arrive(&s.acc_empty[acc]);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (lane == 0) tma_store_wait_all();          // shared memory must stay valid until the last store has read it
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();                // neither CTA leaves (or frees TMEM) while its peer may still touch it
  if (warp == 1) {
    tc_fence_after();
    if (CG == 2) tmem_free_pair<512>(tmem_base);
    else tmem_free<512>(tmem_base);
  }
}

// ------------------------------------------------------------------ TN kernel --------------------
// up to kTnGroup weight-gradient GEMMs that contract over the same rows share ONE launch (e.g. dW_self and dW_neigh of a layer, both
// dpre^T x [h_self | neigh]): every GEMM launch pays ~10 us of prologue / pipeline fill / drain, and one grid over all tiles keeps
// the splits long (tiles * splits <= #SMs)
constexpr int kTnGroup = 4;
struct TnProblem {
  CUtensorMap ta, tb;            // boxes of 64 (inner, n / k index) x 64 (rows m)
  CUtensorMap tout;              // fp32 partials [splits][n][k] (pitch ldo), box 32 x 32 x 1 (TMA store)
  int n, k;                      // output [n, k]
  int k_tiles, tile0;            // tiles of this problem are [tile0, tile0 + n_tiles * k_tiles)
  float* out;                    // partial [splits][n][ldo] (or C itself when splits == 1)
  int ldo;
  int64_t split_stride;
};
struct TnParams {
  TnProblem pr[kTnGroup];
  int n_prob;
  int total_tiles, splits;
  int use_tma_store;
  float alpha_direct;            // output scale of the un-staged single-split store (staged partials are scaled by the reduce)
  const int32_t* m_dev;
  int m_max;
};

// CTA tile = 256 output rows x <= 256 output columns: TWO 128-row accumulators (TMEM columns [0, 256) and [256, 512)) share every B
// stage.  The kernel is bound by what one SM can pull from L2 (~43 B / clock, profiles/r1d_gemm_tn_tc_full.txt: 87 GB/s per SM with
// 128-row tiles); per 128 x 256 x 64 of MMA work a stage now moves 16 KB of A + 16 KB of B instead of 16 + 32.
constexpr int TN_ROWS = 2 * BM;                       // output rows per CTA tile
constexpr int TN_STAGES = 3;
constexpr int TN_A_STAGE_BYTES = 2 * A_STAGE_BYTES;   // two 128-row sub-tiles, each two 64-row chunks of 8 KB
static_assert(TN_STAGES * (TN_A_STAGE_BYTES + B_STAGE_BYTES) == RING_BYTES, "TN ring size mismatch");

template <int KIND>
__global__ void __launch_bounds__(THREADS, 1) k_gemm_tn_tc(const __grid_constant__ TnParams p) {
  constexpr int TF = KIND == 1 ? 1 : 0;
  // a TMA box = CW output-index elements (128 bytes) x BKR contraction rows; bf16: 64 x 64 (8 KB), tf32: 32 x 32 (4 KB).  Stages
  // hold the same bytes either way: 256 output rows of A + up to 256 of B over BKR contraction rows = 32 KB + 32 KB
  constexpr int CW = TF ? 32 : 64;
  constexpr int BKR = TF ? 32 : 64;
  constexpr int CHUNK_BYTES = BKR * 128;
  constexpr int NCH_A = TN_ROWS / CW;
  constexpr int KSTEP = (TF ? 8 : 16) * 128 / 16;           // descriptor address units (16 B) per MMA: its contraction rows x 128 B
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  SmemLayout s = carve(smem_raw, TN_STAGES, B_STAGE_BYTES, RING_BYTES, true);
  s.b0 = smem_raw + TN_STAGES * TN_A_STAGE_BYTES;     // (carve assumes 16 KB A stages)
  const int warp = uniform((int)(threadIdx.x >> 5)), lane = threadIdx.x & 31;

  const int gtile = blockIdx.x % p.total_tiles;
  const int z = blockIdx.x / p.total_tiles;
  int which = 0;
  while (which + 1 < p.n_prob && gtile >= p.pr[which + 1].tile0) ++which;
  const TnProblem& q = p.pr[which];
  const int tile = gtile - q.tile0;
  const int nb = tile / q.k_tiles, kt = tile % q.k_tiles;
  const int row0 = nb * TN_ROWS;
  const int m_dyn = uniform(p.m_dev ? min(*p.m_dev, p.m_max) : p.m_max);
  // contraction range of this split, in 64-row blocks (rows in [m_dyn, round_up(m_dyn, 64)) are zero: zero-tail rule)
  const int blocks_total = (m_dyn + BKR - 1) / BKR;
  const int per = (blocks_total + p.splits - 1) / p.splits;
  const int kb0 = min(z * per, blocks_total), kb1 = min(kb0 + per, blocks_total);
  const int n_sub = (q.n - row0 > BM) ? 2 : 1;                                 // 128-row sub-tiles that hold output rows
  const int n_chunks_a = min(NCH_A, (q.n - row0 + CW - 1) / CW);               // TMA boxes actually needed (sub-tile s = chunks [s, s+1) * NCH_A / 2)
  const int bn_tile = min(BN_MAX, (q.k - kt * BN_MAX + CW - 1) / CW * CW);
  const int n_chunks_b = bn_tile / CW;

  if (threadIdx.x == 64) {
    prefetch_tensormap(&q.ta);
    prefetch_tensormap(&q.tb);
    if (p.use_tma_store) prefetch_tensormap(&q.tout);
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < TN_STAGES; ++i) { mbar_init(&s.full[i], 4); mbar_init(&s.empty[i], 1); }      // (four producers)
    mbar_init(&s.acc_full[0], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc<512>(s.tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = uniform(*s.tmem_slot);
  auto a_stage = [&](int i) { return smem_raw + i * TN_A_STAGE_BYTES; };
  pdl_wait();

  // FOUR TMA producers: warps 0 / 6 load the first / second half of the A chunks of a stage, warps 7 / 8 of the B chunks; each makes
  // its own expect_tx arrival on the full barrier (the split paid under the thread-divergent issue path, see k_gemm_nt_tc; kept)
  auto tma_producer = [&](int which, int part) {    // which: 1 = A chunks, 2 = B chunks; part: 0 / 1 = first / second half of them
    int stage = 0;
    uint32_t phase = 0;
    constexpr int HALF = NCH_A / 2;
    const int n_all = which == 1 ? n_chunks_a : n_chunks_b;
    const int c0 = part * HALF, c1 = min(n_all, c0 + HALF);
    const uint32_t tx = (uint32_t)(max(c1 - c0, 0) * CHUNK_BYTES);
    for (int kb = kb0; kb < kb1; ++kb) {
      mbar_wait(&s.empty[stage], phase ^ 1);
      if (elect_one()) {                             // (all lanes run the loop, see elect_one)
        mbar_expect_tx(&s.full[stage], tx);
        if (which == 1)
          for (int c = c0; c < c1; ++c) tma_load_2d(a_stage(stage) + c * CHUNK_BYTES, &q.ta, &s.full[stage], row0 + c * CW, kb * BKR);
        else
          for (int c = c0; c < c1; ++c) tma_load_2d(s.b(stage) + c * CHUNK_BYTES, &q.tb, &s.full[stage], kt * BN_MAX + c * CW, kb * BKR);
      }
      __syncwarp();
      if (++stage == TN_STAGES) { stage = 0; phase ^= 1; }
    }
  };
  if (warp == 0 || warp >= 6) {
    tma_producer(warp == 0 || warp == 6 ? 1 : 2, warp == 0 || warp == 7 ? 0 : 1);
    __syncwarp();
  } else if (warp == 1) {
    {
      int stage = 0;
      uint32_t phase = 0;
      // M is always issued as 128: when only part of a sub-tile's chunks was loaded its upper accumulator rows hold
      // products with stale shared memory and are never stored (rows >= n)
      const uint32_t idesc = instr_desc(BM, bn_tile, 1, 1, KIND);
      uint32_t accumulate = 0;
      // MN-major descriptors (LBO = distance between 128-byte-wide chunks of the M / N index, SBO = 8 contraction rows): one MMA
      // covers 16 (bf16) / 8 (tf32) contraction rows = 2048 / 1024 bytes = KSTEP in the 14-bit address field; kept branch-free
      const uint64_t a_desc0 = smem_desc(smem_u32(a_stage(0)), CHUNK_BYTES, TF ? 512 : 1024, TF ? 1 : 2),
                     b_desc0 = smem_desc(smem_u32(s.b(0)), CHUNK_BYTES, TF ? 512 : 1024, TF ? 1 : 2);
      const uint32_t acc1 = tmem_base + (uint32_t)BN_MAX;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&s.full[stage], phase);
        tc_fence_after();
        const uint64_t ad = a_desc0 + (uint64_t)(stage * (TN_A_STAGE_BYTES >> 4));
        const uint64_t ad1 = ad + (uint64_t)(A_STAGE_BYTES >> 4);              // second 128-row sub-tile
        const uint64_t bd = b_desc0 + (uint64_t)(stage * (B_STAGE_BYTES >> 4));
        if (elect_one()) {
        if (n_sub == 2) {
          tc_mma<1, TF>(tmem_base, ad, bd, idesc, accumulate);
          tc_mma<1, TF>(acc1, ad1, bd, idesc, accumulate);
          tc_mma<1, TF>(tmem_base, ad + KSTEP, bd + KSTEP, idesc, 1);
          tc_mma<1, TF>(acc1, ad1 + KSTEP, bd + KSTEP, idesc, 1);
          tc_mma<1, TF>(tmem_base, ad + 2 * KSTEP, bd + 2 * KSTEP, idesc, 1);
          tc_mma<1, TF>(acc1, ad1 + 2 * KSTEP, bd + 2 * KSTEP, idesc, 1);
          tc_mma<1, TF>(tmem_base, ad + 3 * KSTEP, bd + 3 * KSTEP, idesc, 1);
          tc_mma<1, TF>(acc1, ad1 + 3 * KSTEP, bd + 3 * KSTEP, idesc, 1);
        } else {
          tc_mma<1, TF>(tmem_base, ad, bd, idesc, accumulate);
          tc_mma<1, TF>(tmem_base, ad + KSTEP, bd + KSTEP, idesc, 1);
          tc_mma<1, TF>(tmem_base, ad + 2 * KSTEP, bd + 2 * KSTEP, idesc, 1);
          tc_mma<1, TF>(tmem_base, ad + 3 * KSTEP, bd + 3 * KSTEP, idesc, 1);
        }
        tc_commit(&s.empty[stage]);
        }
        __syncwarp();
        accumulate = 1;
        if (++stage == TN_STAGES) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) tc_commit(&s.acc_full[0]);
      __syncwarp();
    }
    __syncwarp();
  } else {
    const int quarter = warp & 3;
    const bool have = kb1 > kb0;
    if (have) {
      mbar_wait(&s.acc_full[0], 0);
      tc_fence_after();
    }
    uint8_t* const stage_buf = s.store + (warp - 2) * 2 * STORE_BOX_BYTES;
    uint32_t boxes_issued = 0;
    for (int sub = 0; sub < n_sub; ++sub) {
      const int grow0 = row0 + sub * BM + quarter * 32;      // first output row of this warp's TMEM lane quarter
      const uint32_t tcol0 = (uint32_t)(sub * BN_MAX);
      if (p.use_tma_store) {
        if (grow0 >= q.n) continue;                          // whole boxes clipped
        for (int c0 = 0; c0 < bn_tile; c0 += 32) {
          if (kt * BN_MAX + c0 >= q.k) break;                // whole box clipped
          uint8_t* buf = stage_buf + (boxes_issued & 1) * STORE_BOX_BYTES;
          if (boxes_issued >= 2) {
            if (lane == 0) tma_store_wait_read<1>();
            __syncwarp();
          }
          uint32_t r[32];
          if (have) {
            tc_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + tcol0 + (uint32_t)c0, r);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) r[j] = 0u;
          }
#pragma unroll
          for (int qq = 0; qq < 8; ++qq)
            *reinterpret_cast<uint4*>(buf + lane * 128 + ((qq ^ (lane & 7)) << 4)) = make_uint4(r[qq * 4], r[qq * 4 + 1], r[qq * 4 + 2], r[qq * 4 + 3]);
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_3d(&q.tout, buf, kt * BN_MAX + c0, grow0, z);   // rows >= n / cols >= k clipped
            tma_store_commit();
          }
          ++boxes_issued;
        }
      } else {
        const int gn = grow0 + lane;                         // output row
        float* orow = q.out + (int64_t)z * q.split_stride + (int64_t)gn * q.ldo;
        for (int c0 = 0; c0 < bn_tile; c0 += 32) {
          uint32_t r[32];
          if (have) {
            tc_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + tcol0 + (uint32_t)c0, r);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) r[j] = 0u;
          }
          if (gn < q.n) {
            const int gk0 = kt * BN_MAX + c0;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (gk0 + j < q.k) orow[gk0 + j] = __uint_as_float(r[j]) * p.alpha_direct;
          }
        }
      }
    }
    if (p.use_tma_store) {
      if (lane == 0) tma_store_wait_all();
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_free<512>(tmem_base);
  }
}

// ------------------------------------------------------------------ host side ---------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
int g_tc_state = 0;   // 0 = unknown, 1 = ready, -1 = unavailable

int tc_init() {
  if (g_tc_state != 0) return g_tc_state;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn ||
      q != cudaDriverEntryPointSuccess) {
    cudaGetLastError();
    g_tc_state = -1;
    return -1;
  }
  g_encode = (EncodeTiledFn)fn;
  if (cudaFuncSetAttribute(k_gemm_nt_tc<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_NT1) != cudaSuccess ||
      cudaFuncSetAttribute(k_gemm_nt_tc<2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_NT2) != cudaSuccess ||
      cudaFuncSetAttribute(k_gemm_nt_tc<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_NT1) != cudaSuccess ||
      cudaFuncSetAttribute(k_gemm_nt_tc<2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_NT2) != cudaSuccess ||
      cudaFuncSetAttribute(k_gemm_nt_tc<1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_NT1) != cudaSuccess ||
      cudaFuncSetAttribute(k_gemm_nt_tc<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_NT2) != cudaSuccess ||
      cudaFuncSetAttribute(k_gemm_tn_tc<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_TN) != cudaSuccess ||
      cudaFuncSetAttribute(k_gemm_tn_tc<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_TN) != cudaSuccess ||
      cudaFuncSetAttribute(k_gemm_tn_tc<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_TN) != cudaSuccess) {
    cudaGetLastError();
    g_tc_state = -1;
    return -1;
  }
  g_tc_state = 1;
  return 1;
}

// 2-D bf16 (es = 2) or fp32 (es = 4) tensor [rows, cols] with row pitch ld (elements), box = box_cols x box_rows (box_cols * es
// = 128 bytes), 128-byte swizzle
int make_map(CUtensorMap* map, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows, int es = 2,
             CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B, int f16 = 0) {
  OGL_ARG(((uintptr_t)ptr & 15) == 0 && (ld * es) % 16 == 0, "gemm_tc: operand not 16-byte aligned (ptr %p, ld %lld)", ptr, (long long)ld);
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)(rows > 0 ? rows : 1)};
  cuuint64_t strides[1] = {(cuuint64_t)ld * (cuuint64_t)es};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(map, es == 2 ? (f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                        const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("gemm_tc: cuTensorMapEncodeTiled failed (%d) rows %lld cols %lld ld %lld box %dx%d", (int)r, (long long)rows,
              (long long)cols, (long long)ld, box_cols, box_rows);
    return OGL_ERR_CUDA;
  }
  return OGL_OK;
}

// fp32 [d2][d1][d0] tensor (pitch ld0 elements, plane stride d1*ld0), box 32 x 32 x 1, 128-byte swizzle
int make_map_f32_3d(CUtensorMap* map, const void* ptr, int64_t d0, int64_t d1, int64_t d2, int64_t ld0) {
  OGL_ARG(((uintptr_t)ptr & 15) == 0 && (ld0 * 4) % 16 == 0, "gemm_tc: fp32 output not 16-byte aligned");
  cuuint64_t dims[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
  cuuint64_t strides[2] = {(cuuint64_t)ld0 * 4, (cuuint64_t)ld0 * 4 * (cuuint64_t)d1};
  cuuint32_t box[3] = {32, 32, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("gemm_tc: cuTensorMapEncodeTiled (fp32 3-D) failed (%d)", (int)r);
    return OGL_ERR_CUDA;
  }
  return OGL_OK;
}

}  // namespace

bool gemm_tc_available() { return tc_init() == 1; }

// programmatic dependent launch on every tcgen05 GEMM: the row counts the kernels read before their griddepcontrol.wait are
// written by the sampling kernels of an earlier launch sequence, never by the immediate predecessor
template <typename Kernel, typename Params>
static int launch_gemm(Kernel kernel, int grid, int block, int smem, int cluster, const Params& p, cudaStream_t s) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = (size_t)smem;
  cfg.stream = s;
  cudaLaunchAttribute attrs[2];
  int n = 0;
  if (cluster > 1) {
    attrs[n].id = cudaLaunchAttributeClusterDimension;
    attrs[n].val.clusterDim.x = (unsigned)cluster; attrs[n].val.clusterDim.y = 1; attrs[n].val.clusterDim.z = 1;
    ++n;
  }
  attrs[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attrs[n].val.programmaticStreamSerializationAllowed = 1;
  ++n;
  cfg.attrs = attrs;
  cfg.numAttrs = (unsigned)n;
  OGL_CUDA(cudaLaunchKernelEx(&cfg, kernel, p));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return OGL_OK;
}

int gemm_nt_tc(const GemmNT& g, cudaStream_t s) {
  OGL_ARG(tc_init() == 1, "gemm_nt_tc: tcgen05 path unavailable (driver lacks cuTensorMapEncodeTiled?)");
  OGL_ARG((g.in_bf16 != 0) != (g.tf32 != 0), "gemm_nt_tc: 16-bit or tf32 operands only");
  OGL_ARG(!(g.f16 && g.tf32), "gemm_nt_tc: f16 goes with 16-bit operands");
  OGL_ARG(!(g.tf32 && g.out_bf16), "gemm_nt_tc: tf32 operands give fp32 output");
  OGL_ARG(g.n > 0 && g.m_max > 0 && g.n_seg >= 1 && g.n_seg <= 2, "gemm_nt_tc: bad shape");
  const int tf = g.tf32 ? 1 : 0;
  const int es = tf ? 4 : 2;                 // operand element bytes
  const int bke = 128 / es;                  // contraction elements per 128-byte swizzle row
  NtParams p;
  memset(&p, 0, sizeof(p));
  p.n = g.n;
  p.n_tiles = (g.n + BN_MAX - 1) / BN_MAX;
  p.bn = p.n_tiles > 1 ? BN_MAX : (g.n + 15) / 16 * 16;
  p.n_seg = g.n_seg;
  // CTA pairs (cta_group::2) when there are enough 256-row super tiles to occupy every pair of SMs
  const int64_t super_tiles = ceil_div(ceil_div(g.m_max, BM), 2) * p.n_tiles;
  const int cg = (g.force_cg == 1 || g.force_cg == 2) ? g.force_cg : ((super_tiles >= sm_count() / 2 && p.bn % 32 == 0) ? 2 : 1);
  for (int i = 0; i < g.n_seg; ++i) {
    p.k[i] = g.k[i];
    p.a_rows_dev[i] = g.a_rows_dev[i];
    const int64_t a_rows = g.a_rows_max[i] > 0 ? g.a_rows_max[i] : g.m_max;      // rows that exist in segment i's A buffer
    OGL_TRY(make_map(&p.ta[i], g.a[i], a_rows, g.k[i], g.lda[i], bke, BM, es, CU_TENSOR_MAP_SWIZZLE_128B, g.f16));
    OGL_TRY(make_map(&p.tb[i], g.b[i], g.n, g.k[i], g.ldb[i], bke, cg == 2 ? p.bn / 2 : p.bn, es, CU_TENSOR_MAP_SWIZZLE_128B, g.f16));
  }
  p.m_dev = g.m_dev;
  p.m_max = g.m_max;
  p.bias = g.bias;
  p.bias2 = g.bias2;
  p.relu = g.relu;
  p.alpha = g.alpha;
  p.mask = g.mask;
  p.ldmask = g.ldmask;
  p.c = g.c;
  p.ldc = g.ldc;
  p.out_bf16 = g.out_bf16;
  // tf32 mode: activations leave through 32 x 32 fp32 TMA-store boxes (the logits GEMM -- no rounding, not a later operand -- keeps
  // the direct fp32 stores, its 41 columns are no 16-byte multiple of anything)
  p.out_f32_tma = (tf && (g.out_tf32 || g.mask)) ? 1 : 0;
  p.round_out = g.out_tf32;
  p.zero_tail = g.zero_tail;
  OGL_ARG(!(g.mask && !(g.out_bf16 || p.out_f32_tma)), "gemm_nt_tc: the mask epilogue is implemented for the TMA-store outputs only");
  if (g.out_bf16) OGL_TRY(make_map(&p.tc, g.c, g.m_max, g.ldc, g.ldc, 64, 32, 2, CU_TENSOR_MAP_SWIZZLE_128B, g.f16));
  if (p.out_f32_tma) OGL_TRY(make_map(&p.tc, g.c, g.m_max, g.ldc, g.ldc, 32, 32, 4));
  OGL_ARG(g.ldc % 8 == 0 && ((uintptr_t)g.c & 15) == 0, "gemm_nt_tc: output pitch must be a multiple of 8 elements");
  OGL_ARG(!g.mask || (g.ldmask % 8 == 0 && ((uintptr_t)g.mask & 15) == 0), "gemm_nt_tc: mask pitch must be a multiple of 8 elements");
  if (cg == 2) {
    const int pairs = (int)(super_tiles < sm_count() / 2 ? super_tiles : sm_count() / 2);
    if (tf) OGL_TRY(launch_gemm(k_gemm_nt_tc<2, 1>, 2 * pairs, THREADS_NT, SMEM_NT2, 2, p, s));
    else if (g.f16) OGL_TRY(launch_gemm(k_gemm_nt_tc<2, 2>, 2 * pairs, THREADS_NT, SMEM_NT2, 2, p, s));
    else OGL_TRY(launch_gemm(k_gemm_nt_tc<2, 0>, 2 * pairs, THREADS_NT, SMEM_NT2, 2, p, s));
    return OGL_OK;
  }
  const int64_t tiles = ceil_div(g.m_max, BM) * p.n_tiles;
  const int grid = (int)(tiles < sm_count() ? tiles : sm_count());
  if (tf) return launch_gemm(k_gemm_nt_tc<1, 1>, grid, THREADS_NT, SMEM_NT1, 1, p, s);
  if (g.f16) return launch_gemm(k_gemm_nt_tc<1, 2>, grid, THREADS_NT, SMEM_NT1, 1, p, s);
  return launch_gemm(k_gemm_nt_tc<1, 0>, grid, THREADS_NT, SMEM_NT1, 1, p, s);
}

int gemm_tn_tc_group(const GemmTN* g, int count, cudaStream_t s) {
  OGL_ARG(tc_init() == 1, "gemm_tn_tc: tcgen05 path unavailable");
  OGL_ARG(g && count >= 1 && count <= kTnGroup, "gemm_tn_tc: 1..%d problems per launch", kTnGroup);
  TnParams p;
  memset(&p, 0, sizeof(p));
  p.n_prob = count;
  p.m_dev = g[0].m_dev;
  p.m_max = g[0].m_max;
  const int tf = g[0].tf32 ? 1 : 0;
  const int es = tf ? 4 : 2;
  const int cw = 128 / es;                   // TMA box: cw output-index elements (128 bytes) x cw contraction rows
  int tiles = 0;
  int64_t per_total = 0;
  for (int i = 0; i < count; ++i) {
    OGL_ARG((g[i].in_bf16 || g[i].tf32) && g[i].n > 0 && g[i].k > 0 && g[i].m_max > 0, "gemm_tn_tc: bad arguments");
    OGL_ARG(g[i].m_dev == g[0].m_dev && g[i].m_max == g[0].m_max && g[i].tf32 == g[0].tf32 && g[i].f16 == g[0].f16,
            "gemm_tn_tc: grouped problems must contract over the same rows in the same arithmetic");
    TnProblem& q = p.pr[i];
    // (MN-major tf32 operands: the 32-byte-atom flavour of the 128-byte swizzle, see smem_desc)
    const CUtensorMapSwizzle sw = tf ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B;
    OGL_TRY(make_map(&q.ta, g[i].a, g[i].m_max, g[i].n, g[i].lda, cw, cw, es, sw, g[i].f16));
    OGL_TRY(make_map(&q.tb, g[i].b, g[i].m_max, g[i].k, g[i].ldb, cw, cw, es, sw, g[i].f16));
    q.n = g[i].n;
    q.k = g[i].k;
    q.k_tiles = (g[i].k + BN_MAX - 1) / BN_MAX;
    q.tile0 = tiles;
    tiles += ((g[i].n + TN_ROWS - 1) / TN_ROWS) * q.k_tiles;
    q.ldo = (g[i].k + 3) / 4 * 4;
    per_total += (int64_t)g[i].n * q.ldo;
  }
  p.total_tiles = tiles;
  // one CTA per SM and exactly one wave: tiles * splits <= #SMs (150 CTAs on 148 SMs would run as two waves)
  int splits = sm_count() / tiles;
  const int by_rows = (int)ceil_div(g[0].m_max, 4 * cw);          // at least 4 contraction blocks per split
  if (splits > by_rows) splits = by_rows;
  float* ws = g[0].partial;
  const int64_t ws_elems = ws ? g[0].partial_elems : 0;
  if ((int64_t)splits * per_total > ws_elems) splits = (int)(ws_elems / per_total);
  if (splits < 1) splits = 1;
  p.splits = splits;
  const bool staged = ws != nullptr && per_total <= ws_elems;       // partials (pitch % 4 == 0) take TMA stores
  OGL_ARG(staged || count == 1, "gemm_tn_tc: a grouped launch needs the split workspace");
  ReduceGroup rg;
  memset(&rg, 0, sizeof(rg));
  rg.count = count;
  rg.splits = splits;
  int64_t off = 0;
  for (int i = 0; i < count; ++i) {
    TnProblem& q = p.pr[i];
    if (!staged) {
      OGL_ARG(splits == 1, "gemm_tn_tc: internal: split without workspace");
      q.out = g[i].c;
      q.ldo = g[i].ldc;
      q.split_stride = 0;
    } else {
      const int64_t per = (int64_t)g[i].n * q.ldo;
      q.out = ws + off;
      q.split_stride = per;
      OGL_TRY(make_map_f32_3d(&q.tout, q.out, g[i].k, g[i].n, splits, q.ldo));
      rg.pr[i] = {q.out, g[i].c, g[i].n, g[i].k, q.ldo, g[i].ldc, g[i].alpha};
      off += (int64_t)splits * per;
    }
  }
  p.use_tma_store = staged ? 1 : 0;
  p.alpha_direct = g[0].alpha;
  if (tf) OGL_TRY(launch_gemm(k_gemm_tn_tc<1>, tiles * splits, THREADS, SMEM_TN, 1, p, s));
  else if (g[0].f16) OGL_TRY(launch_gemm(k_gemm_tn_tc<2>, tiles * splits, THREADS, SMEM_TN, 1, p, s));
  else OGL_TRY(launch_gemm(k_gemm_tn_tc<0>, tiles * splits, THREADS, SMEM_TN, 1, p, s));
  if (staged) return reduce_splits_group(rg, s);
  return OGL_OK;
}

int gemm_tn_tc(const GemmTN& g, cudaStream_t s) { return gemm_tn_tc_group(&g, 1, s); }

}  // namespace ogl

using namespace ogl;

extern "C" int ogl_gemm_bf16_nt(const void* a_dev, int lda, const void* b_dev, int ldb, float* c_dev, int ldc, int m, int n, int k,
                                void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(a_dev && b_dev && c_dev && m > 0 && n > 0 && k > 0, "ogl_gemm_bf16_nt: bad arguments");
  GemmNT g;
  g.a[0] = a_dev; g.lda[0] = lda; g.b[0] = b_dev; g.ldb[0] = ldb; g.k[0] = k; g.n_seg = 1;
  g.c = c_dev; g.ldc = ldc; g.m_max = m; g.n = n; g.in_bf16 = 1; g.out_bf16 = 0; g.zero_tail = 0;
  return gemm_nt_tc(g, (cudaStream_t)stream);
}

extern "C" int ogl_gemm_bf16_nt_ex(const void* a_dev, int lda, const void* b_dev, int ldb, void* c_dev, int ldc, int m, int n, int k,
                                   int out_bf16, const float* bias_dev, int relu, int cg, void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(a_dev && b_dev && c_dev && m > 0 && n > 0 && k > 0, "ogl_gemm_bf16_nt_ex: bad arguments");
  GemmNT g;
  g.a[0] = a_dev; g.lda[0] = lda; g.b[0] = b_dev; g.ldb[0] = ldb; g.k[0] = k; g.n_seg = 1;
  g.c = c_dev; g.ldc = ldc; g.m_max = m; g.n = n; g.in_bf16 = 1; g.out_bf16 = out_bf16; g.zero_tail = 0;
  g.bias = bias_dev; g.relu = relu; g.force_cg = cg;
  return gemm_nt_tc(g, (cudaStream_t)stream);
}

extern "C" int ogl_gemm_bf16_tn(const void* a_dev, int lda, const void* b_dev, int ldb, float* c_dev, int ldc, int m, int n, int k,
                                float* workspace_dev, int64_t workspace_elems, void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(a_dev && b_dev && c_dev && m > 0 && n > 0 && k > 0, "ogl_gemm_bf16_tn: bad arguments");
  GemmTN g;
  g.a = a_dev; g.lda = lda; g.b = b_dev; g.ldb = ldb; g.c = c_dev; g.ldc = ldc; g.n = n; g.k = k; g.m_max = m; g.in_bf16 = 1;
  g.partial = workspace_dev; g.partial_elems = workspace_dev ? workspace_elems : 0;
  return gemm_tn_tc(g, (cudaStream_t)stream);
}

// tf32 flavour of the two entry points above (fp32 operands that hold TF32-rounded values; tests / bench)
extern "C" int ogl_gemm_tf32_nt_ex(const float* a_dev, int lda, const float* b_dev, int ldb, float* c_dev, int ldc, int m, int n, int k,
                                   int tma_out, const float* bias_dev, int relu, const float* mask_dev, int ldmask, int cg, void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(a_dev && b_dev && c_dev && m > 0 && n > 0 && k > 0, "ogl_gemm_tf32_nt_ex: bad arguments");
  GemmNT g;
  g.a[0] = a_dev; g.lda[0] = lda; g.b[0] = b_dev; g.ldb[0] = ldb; g.k[0] = k; g.n_seg = 1;
  g.c = c_dev; g.ldc = ldc; g.m_max = m; g.n = n; g.tf32 = 1; g.out_tf32 = tma_out; g.zero_tail = 0;
  g.bias = bias_dev; g.relu = relu; g.force_cg = cg; g.mask = mask_dev; g.ldmask = ldmask;
  return gemm_nt_tc(g, (cudaStream_t)stream);
}

extern "C" int ogl_gemm_tf32_tn(const float* a_dev, int lda, const float* b_dev, int ldb, float* c_dev, int ldc, int m, int n, int k,
                                float* workspace_dev, int64_t workspace_elems, void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(a_dev && b_dev && c_dev && m > 0 && n > 0 && k > 0, "ogl_gemm_tf32_tn: bad arguments");
  GemmTN g;
  g.a = a_dev; g.lda = lda; g.b = b_dev; g.ldb = ldb; g.c = c_dev; g.ldc = ldc; g.n = n; g.k = k; g.m_max = m; g.tf32 = 1;
  g.partial = workspace_dev; g.partial_elems = workspace_dev ? workspace_elems : 0;
  return gemm_tn_tc(g, (cudaStream_t)stream);
}

// fp16 flavour (mode OGL_FP16: tcgen05 kind::f16 with fp16 operands; tests / bench).  mask (fp16, [m, ldmask]): out = mask > 0 ? out : 0;
// alpha scales the weight-gradient output (the plan passes 1 / loss scale there)
extern "C" int ogl_gemm_f16_nt_ex(const void* a_dev, int lda, const void* b_dev, int ldb, void* c_dev, int ldc, int m, int n, int k,
                                  int out_f16, const float* bias_dev, int relu, const void* mask_dev, int ldmask, int cg, void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(a_dev && b_dev && c_dev && m > 0 && n > 0 && k > 0, "ogl_gemm_f16_nt_ex: bad arguments");
  GemmNT g;
  g.a[0] = a_dev; g.lda[0] = lda; g.b[0] = b_dev; g.ldb[0] = ldb; g.k[0] = k; g.n_seg = 1;
  g.c = c_dev; g.ldc = ldc; g.m_max = m; g.n = n; g.in_bf16 = 1; g.f16 = 1; g.out_bf16 = out_f16; g.zero_tail = 0;
  g.bias = bias_dev; g.relu = relu; g.force_cg = cg; g.mask = mask_dev; g.ldmask = ldmask;
  return gemm_nt_tc(g, (cudaStream_t)stream);
}

extern "C" int ogl_gemm_f16_tn(const void* a_dev, int lda, const void* b_dev, int ldb, float* c_dev, int ldc, int m, int n, int k,
                               float alpha, float* workspace_dev, int64_t workspace_elems, void* stream) {
  OGL_TRY(require_device());
  OGL_ARG(a_dev && b_dev && c_dev && m > 0 && n > 0 && k > 0, "ogl_gemm_f16_tn: bad arguments");
  GemmTN g;
  g.a = a_dev; g.lda = lda; g.b = b_dev; g.ldb = ldb; g.c = c_dev; g.ldc = ldc; g.n = n; g.k = k; g.m_max = m; g.in_bf16 = 1; g.f16 = 1;
  g.alpha = alpha;
  g.partial = workspace_dev; g.partial_elems = workspace_dev ? workspace_elems : 0;
  return gemm_tn_tc(g, (cudaStream_t)stream);
}
