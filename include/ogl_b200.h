/*
 * ogl_b200.h -- C ABI of the B200-native streaming GraphSAGE hot path.
 *
 * Drop-in boundary for MassimoPerini/online-gnn-learning's `--backend pytorch --cuda`
 * path.  The reference has no FFI of its own (it is pure Python over DGL + PyTorch), so
 * every entry point below cites the reference call site (file:line under
 * /root/reference) whose DGL / PyTorch / Python work it replaces.  INTEGRATION.md shows
 * the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / C++ types.  `*_dev` pointers are device
 *     memory, `*_host` pointers are host memory (pinned for async copies).
 *   - every call returns 0 on success, <0 on error; ogl_last_error() returns the message
 *     of the last failing call on this thread.  No C++ exception crosses the boundary.
 *   - all work is ordered on the caller's `stream` (a cudaStream_t passed as void*);
 *     one host thread per GPU; the library starts no host threads.
 *   - persistent device memory lives only inside the opaque handles created/destroyed
 *     here.  There is NO CPU fallback: every entry point fails if no sm_100 device is
 *     present.
 */
#ifndef OGL_B200_H_
#define OGL_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#pragma GCC visibility push(default)

typedef struct ogl_graph ogl_graph;       /* streaming in-edge CSR (slack rows + snapshot tails) */
typedef struct ogl_features ogl_features; /* device feature / label store (padded rows) */
typedef struct ogl_plan ogl_plan;         /* sampler + GraphSAGE-pool model + optimiser workspace */
typedef struct ogl_sumtree ogl_sumtree;   /* fp64 sum-tree for PBR */
typedef struct ogl_peer ogl_peer;         /* one rank's end of the NVLink peer-memory gradient exchange */

/* arithmetic mode of the dense path.  OGL_F32: fp32 storage, SIMT FFMA GEMMs (exact; rtol 1e-5 against the fp32 reference path).
 * OGL_BF16: bf16 storage, tcgen05 kind::f16 GEMMs with fp32 accumulation (fastest; ~2^-9 per stored value).
 * OGL_TF32: fp32 storage with every GEMM operand rounded to TF32 where it is produced, tcgen05 kind::tf32 GEMMs with fp32
 *           accumulation -- the tensor-core mode that meets rtol 1e-3 against the reference's fp32 path (utils.py:63-64).
 * OGL_FP16: fp16 storage (the same 10 explicit mantissa bits as TF32 in half the bytes), tcgen05 kind::f16 GEMMs with fp32
 *           accumulation, STATIC LOSS SCALING: activation gradients are stored times a power of two chosen from the loss scale
 *           (so that they sit in fp16's normal range) and every weight / bias gradient is unscaled, exactly, where it is written
 *           in fp32.  TF32's error at bf16's speed; stored values must stay below 65504 (standardised features). */
enum { OGL_F32 = 0, OGL_BF16 = 1, OGL_TF32 = 2, OGL_FP16 = 3 };
enum { OGL_OK = 0, OGL_ERR_CUDA = -1, OGL_ERR_ARG = -2, OGL_ERR_CAPACITY = -3, OGL_ERR_NODEVICE = -4 };

const char* ogl_last_error(void);
int ogl_version(void);
/* number of kernels launched by this library since process start (bench.py: gpu_launches) */
int64_t ogl_kernel_launches(void);

/* ------------------------------------------------------------------ graph ----------
 * Replaces dgl.graph([]) + add_nodes / add_edges / subgraph as driven by
 *   train/graph/dynamic_graph_edge.py:27,61-72 (build), :190-218 (evolve)
 *   train/graph/dynamic_graph_vertex.py:82-94 (build), :132-141 (evolve)
 * Canonical content: in-neighbour list of v = sources of edges with dst == v in
 * ascending edge id (edge id = insertion order).
 */
int ogl_graph_create(ogl_graph** out, int64_t v_cap, int64_t e_cap_directed);
int ogl_graph_destroy(ogl_graph* g);
/* add_nodes(n): ids [V, V+n) become valid rows */
int ogl_graph_insert_vertices(ogl_graph* g, int64_t n, void* stream);
/* add_edges(src,dst) [then add_edges(dst,src) if symmetric]; device or host int64 ids.
 * Edge ids continue the insertion order: forward edges first, then the reverse edges
 * (dynamic_graph_edge.py:214-215). */
int ogl_graph_insert_edges(ogl_graph* g, const int64_t* src_dev, const int64_t* dst_dev, int64_t n,
                           int symmetric, void* stream);
/* a shard of a destination-range-partitioned CSR (SURVEY 8(e), config 5): its rows are local, the source ids stored in them
 * global -- sources are then accepted in [0, n_sources) instead of [0, number of local vertices) (0 restores the default) */
int ogl_graph_set_source_bound(ogl_graph* g, int64_t n_sources);
int ogl_graph_insert_edges_host(ogl_graph* g, const int64_t* src_host, const int64_t* dst_host, int64_t n,
                                int symmetric, void* stream);
/* vertex streams: load the parent graph once (ids already relabelled to arrival rank,
 * in-CSR in parent edge-id order), then activate a prefix; rebuilds the induced CSR the
 * way graph.subgraph(evolving_vertices) does at dynamic_graph_vertex.py:85,140 */
int ogl_graph_load_parent(ogl_graph* g, const int64_t* indptr_dev, const int64_t* indices_dev,
                          const int64_t* eids_dev, int64_t n_vertices, void* stream);
int ogl_graph_set_active_prefix(ogl_graph* g, int64_t n_active, void* stream);
int ogl_graph_num_vertices(ogl_graph* g, int64_t* out);
int ogl_graph_num_edges(ogl_graph* g, int64_t* out);          /* directed */
int ogl_graph_degrees(ogl_graph* g, int64_t* out_dev, void* stream);
/* canonical compact CSR (indptr[V+1], indices[E], eids[E]); eids_dev may be NULL */
int ogl_graph_export_csr(ogl_graph* g, int64_t* indptr_dev, int64_t* indices_dev, int64_t* eids_dev, void* stream);
/* squeeze relocation garbage out of the adjacency pool (also run automatically when full) */
int ogl_graph_compact(ogl_graph* g, void* stream);
/* pool statistics: {pool_used, pool_cap, relocations, compactions} */
int ogl_graph_stats(ogl_graph* g, int64_t out[4]);

/* ------------------------------------------------------------------ features --------
 * Replaces graph.ndata['feat'] / ['target'] storage + the per-batch CPU gather and H2D
 * copy at train/graphsage/pytorch/model.py:88-99; rows are appended by add_nodes
 * (dynamic_graph_edge.py:64-65,206-207).  Rows are stored padded, in the arithmetic mode.
 */
int ogl_features_create(ogl_features** out, int64_t v_cap, int n_feats, int mode);
int ogl_features_destroy(ogl_features* f);
/* rows [row0, row0+n) <- fp32 feats[n, n_feats] and int64 labels[n]; dev or host source */
int ogl_features_write(ogl_features* f, int64_t row0, int64_t n, const float* feats, const int64_t* labels,
                       int src_is_host, void* stream);
/* rows[i] <- fp32 feats[src_rows[i]] (device table gather; vertex-stream relabelling) */
int ogl_features_write_permuted(ogl_features* f, int64_t n, const float* feats_dev, const int64_t* labels_dev,
                                const int64_t* src_rows_dev, void* stream);

/* ------------------------------------------------------------------ plan ------------
 * One plan = the sampler, the L-layer GraphSAGE('pool') model and Adam, with all
 * workspaces sized for max_seeds.  Replaces, per minibatch,
 *   dgl.sampling.MultiLayerNeighborSampler + NodeDataLoader   pytorch/model.py:44-47,128-131
 *   GraphSAGE.forward over DGL SAGEConv('pool')              graphsage_dgl.py:48-59
 *   CrossEntropyLoss / backward / Adam.step                  pytorch/model.py:20-25,103-107
 */
typedef struct {
  int n_layers;          /* = number of hops/blocks (reference: always 2) */
  int dims[8];           /* dims[0]=F, dims[1..L-1]=hidden, dims[L]=classes */
  int fanouts[8];        /* fanouts[0] at the seeds hop, [1] next hop out, ... */
  int max_seeds;
  int64_t v_cap;
  int mode;              /* OGL_F32 | OGL_BF16 | OGL_TF32 | OGL_FP16 */
  int gemm_impl;         /* 0 = default for mode (tcgen05 for bf16 / tf32 / fp16, SIMT for f32), 1 = force SIMT (tests) */
  uint64_t seed;         /* Philox key */
  float lr, beta1, beta2, eps;
  float feat_drop;       /* SAGEConv(feat_drop=dropout), graphsage_dgl.py:41-46: dropout of every layer's input rows in training mode
                            (train steps; ogl_plan_forward after ogl_plan_set_option("train_mode", 1)); 0 = off.  The mask is keyed by
                            the optimiser step in a train step and by the number of earlier training-mode ogl_plan_forward calls in
                            a direct forward (each such call advances it; ogl_plan_reset_optimizer zeroes it) */
} ogl_plan_config;

/* mode OGL_FP16: the power of two the stored activation gradients of a backward pass carry for a given loss scale (1 / global batch):
 * 2^floor(log2(64 / loss_scale)), i.e. the largest |dlogits| element is stored in (32, 64].  Pure host function (no device needed);
 * oracle/sage.py: grad_scale_for is its twin */
float ogl_fp16_grad_scale(float loss_scale);
int ogl_plan_create(ogl_plan** out, const ogl_plan_config* cfg);
int ogl_plan_destroy(ogl_plan* p);
/* flat fp32 parameter / gradient buffers (caller-owned device memory, e.g. a torch
 * tensor): per layer i, in order fc_pool.weight [in,in], fc_pool.bias [in],
 * fc_self.weight [out,in], fc_self.bias [out], fc_neigh.weight [out,in], fc_neigh.bias [out] */
int64_t ogl_plan_param_count(const ogl_plan* p);
int ogl_plan_bind_params(ogl_plan* p, float* params_dev, float* grads_dev, void* stream);
/* call after params were changed outside the library (load_state_dict) */
int ogl_plan_refresh_params(ogl_plan* p, void* stream);
int ogl_plan_set_step(ogl_plan* p, uint32_t step, void* stream);
/* fresh optimiser state (Adam moments and step counter zeroed) and Philox step = philox_step: the reference's build_optimizer()
 * constructs a new torch.optim.Adam (pytorch/model.py:22-25) */
int ogl_plan_reset_optimizer(ogl_plan* p, uint32_t philox_step, void* stream);
/* sticky device-side error flags since the last call (synchronises; clears them).  bit 0: a seed id outside [0, n_vertices) was
 * passed to a sampling / train / eval call -- it was replaced by vertex 0 so that no row metadata is read out of bounds (DGL's
 * NodeDataLoader raises on such ids, pytorch/model.py:128-131).  bit 1: ogl_plan_infer_full_loss / ogl_plan_full_xent met a label
 * outside [0, classes) -- that vertex's loss is NaN (torch's cross_entropy raises on such labels) */
int ogl_plan_error_flags(ogl_plan* p, uint32_t* out);

/* sample the L-hop minibatch for `seeds` (device int64, n_seeds <= max_seeds) */
int ogl_plan_sample(ogl_plan* p, ogl_graph* g, const int64_t* seeds_dev, int n_seeds, void* stream);
/* forward over the sampled minibatch; logits_dev (fp32 [n_seeds, classes]) may be NULL.  In training mode with feat_drop > 0 it
 * advances the direct-forward dropout counter (see ogl_plan_config.feat_drop) */
int ogl_plan_forward(ogl_plan* p, ogl_features* f, float* logits_dev, void* stream);
/* loss + backward; grads land in the bound gradient buffer (overwritten).
 * loss_scale multiplies dlogits (1/global_batch for the 'mean' reduction);
 * per_vertex_loss_dev (fp32 [n_seeds]) may be NULL; loss_sum_dev (fp32 [1], may be NULL; here and in every step entry point
 * below) receives the sum of the per-vertex losses -- any device-ACCESSIBLE address: device memory, or pinned host memory, in
 * which case the loss kernel stores the 4 bytes over PCIe itself and no D2H copy is needed (valid once the stream has passed) */
int ogl_plan_loss_backward(ogl_plan* p, ogl_features* f, float loss_scale, float* per_vertex_loss_dev,
                           float* loss_sum_dev, void* stream);
/* autograd-compat path (GraphSAGE.forward(blocks, x) + loss.backward() driven from Python):
 * supply the input rows x [n_rows, F] fp32 for the outermost level instead of gathering them
 * (then call ogl_plan_forward with f == NULL), and back-propagate a caller-computed
 * dlogits [n_seeds, classes] fp32 into the bound gradient buffer.  dlogits_amax = max |dlogits| (read only in mode OGL_FP16: the
 * activation gradients are stored times ogl_fp16_grad_scale(dlogits_amax), so the largest is in (32, 64] whatever the loss's
 * reduction or scale; 0 or a non-finite value gives scale 1) */
int ogl_plan_set_input(ogl_plan* p, const float* x_dev, int n_rows, void* stream);
int ogl_plan_backward(ogl_plan* p, const float* dlogits_dev, float dlogits_amax, void* stream);
int ogl_plan_adam_step(ogl_plan* p, void* stream);
/* fused: sample + forward + loss + backward (+ Adam if do_step) for host or device seeds */
int ogl_plan_train_step(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_seeds,
                        int seeds_on_host, float loss_scale, int do_step, float* per_vertex_loss_dev,
                        float* loss_sum_dev, void* stream);
/* n_batches consecutive train steps of `batch` seeds each (seeds = [n_batches * batch]) without returning to the host in
 * between -- the batch_timestep minibatches of one snapshot (pytorch/model.py:129-134).  per_vertex_loss_dev
 * [n_batches * batch] and loss_sums_dev [n_batches] may be NULL */
int ogl_plan_train_steps(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_batches, int batch, int seeds_on_host,
                         float loss_scale, int do_step, float* per_vertex_loss_dev, float* loss_sums_dev, void* stream);
/* the same step in two calls, for data-parallel pipelining: step_begin = sample + gather (independent of the weights: it
 * can run while the previous step's gradient all-reduce + Adam are still in flight on another stream); step_finish =
 * forward + loss + backward (+ Adam if do_step) over the minibatch begun last */
int ogl_plan_step_begin(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_seeds, int seeds_on_host,
                        void* stream);
int ogl_plan_step_finish(ogl_plan* p, ogl_features* f, float loss_scale, int do_step, float* per_vertex_loss_dev,
                         float* loss_sum_dev, void* stream);
/* step_finish (without Adam) in two pieces for a bucketed gradient exchange: after _head every gradient except layer 0's
 * fc_pool.weight (the first in*in floats of the flat buffer) is final; _tail computes that last one */
int ogl_plan_step_finish_head(ogl_plan* p, ogl_features* f, float loss_scale, float* per_vertex_loss_dev, float* loss_sum_dev,
                              void* stream);
int ogl_plan_step_finish_tail(ogl_plan* p, ogl_features* f, void* stream);
/* data-parallel finish in ONE launch sequence (one CUDA graph per step): forward .. backward with the gradient exchange over NVLink
 * peer memory and Adam as nodes of the same graph -- all gradients but layer 0's fc_pool.weight are exchanged beside the last
 * weight-gradient GEMM, that one after it.  The plan's gradient buffer must be `peer`'s (ogl_peer_buffer). */
int ogl_plan_step_finish_dp(ogl_plan* p, ogl_peer* peer, ogl_features* f, float loss_scale, float* per_vertex_loss_dev,
                            float* loss_sum_dev, void* stream);
/* software pipeline (the job of NodeDataLoader's worker processes, pytorch/model.py:128-131): sample + gather of a FUTURE minibatch,
 * enqueued on the plan's own stream into the plan's second buffer set, ordered after everything enqueued on `stream` so far.  Up to
 * two minibatches may be pending.  The next ogl_plan_train_step / ogl_plan_step_finish[_head] on the plan consumes the oldest pending
 * minibatch (forward .. Adam only; its `seeds` argument is then ignored, n_seeds must match).  Call order for full overlap:
 *   prefetch(0); for i: { prefetch(i+1); train_step(i); }
 * ogl_plan_train_steps pipelines its minibatches this way internally (option "pipeline", default 1). */
int ogl_plan_prefetch(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_seeds, int seeds_on_host, void* stream);
int ogl_plan_prefetch_pending(const ogl_plan* p);   /* number of prefetched minibatches not yet consumed (0..2) */
/* ---- data-parallel gradient exchange over NVLink peer memory, fused with Adam (SURVEY 8(e); the reference is single-process) ----
 * Every rank owns a gradient buffer inside an allocation its peers map through CUDA IPC.  ogl_plan_peer_adam launches ONE kernel:
 * barrier over peer-memory flags -> gradients [lo, hi) summed over the ranks in rank order with P2P loads (bit-identical replicas) ->
 * Adam on the local fp32 parameters + bf16 weight shadows -> "done reading" flags to the peers.  Replaces
 * all_reduce(flat_grad) + ogl_plan_adam_step.  Protocol per step, identical on every rank:
 *     ogl_peer_wait_readers   (before the backward pass overwrites the gradient buffer)
 *     ... backward ...        (the plan's gradient buffer must be ogl_peer_buffer)
 *     ogl_plan_peer_adam(lo, hi, last) for each bucket, the same buckets in the same order on every rank
 * Setup: create -> exchange the 64-byte ogl_peer_handle of every rank (any transport) -> ogl_peer_connect(all handles, rank order). */
int ogl_peer_create(ogl_peer** out, int rank, int world, int64_t n_floats);
int ogl_peer_destroy(ogl_peer* p);
int ogl_peer_handle(ogl_peer* p, void* handle64);
int ogl_peer_connect(ogl_peer* p, const void* handles /* world x 64 bytes */);
int ogl_peer_connect_local(ogl_peer* p, ogl_peer* const* all /* the world peers of ONE process, rank order */);
int ogl_peer_buffer(ogl_peer* p, float** grads_dev);
int ogl_peer_wait_readers(ogl_peer* p, void* stream);
int ogl_plan_peer_adam(ogl_plan* p, ogl_peer* peer, int64_t lo, int64_t hi, int last, float* reduced_out_dev /* may be NULL */, void* stream);
/* ---- streaming inference with cached per-vertex intermediates (inference_optimized.py:144-301; SURVEY 8(f)-3), fp32 ------------
 * ogl_graph_row_degrees / ogl_graph_gather_rows: g.out_degrees(v) / g.in_edges(v) / g.out_edges(v) on the streaming CSR of the
 *   serving graph (:185, :194-196, :205): degrees of the listed vertices, then their adjacency rows (ascending edge id) written at
 *   offsets_dev[i] (the exclusive prefix sums of the degrees).
 * ogl_infer_rows_linear: out[out_ids[i]] = act(x1[ids1[i]] . w1^T + b1 (+ x2[ids2[i]] . w2^T + b2)): relu(fc_pool(h)) (:258-260) and
 *   fc_self(h) + fc_neigh(neigh) (:273-276) on a row set; weights row-major [n_out, k] as torch.nn.Linear stores them.
 * ogl_infer_induced_mean: out[v] = mean over in-edges (u -> v) with member[u] != 0 of proj[u], 0 if none, for v in nodes: DGL's
 *   subgraph(S).update_all(copy_src, mean) as the handler uses it (:265-268). */
int ogl_graph_row_degrees(ogl_graph* g, const int64_t* v_dev, int64_t n, int64_t* deg_out_dev, void* stream);
int ogl_graph_gather_rows(ogl_graph* g, const int64_t* v_dev, int64_t n, const int64_t* offsets_dev, int64_t* out_src_dev, void* stream);
int ogl_infer_rows_linear(const float* x1_dev, int ld1, const int64_t* ids1_dev, const float* w1_dev, int k1, const float* b1_dev,
                          const float* x2_dev, int ld2, const int64_t* ids2_dev, const float* w2_dev, int k2, const float* b2_dev,
                          int relu, float* out_dev, int ldo, const int64_t* out_ids_dev, int64_t n_rows, int n_out, void* stream);
/* the neighbourhood query of one request in one launch: rows [0, v_off) of g hold in-edge sources, rows [v_off, 2 v_off) out-edge targets.
 * out_dev (int64): [overflow, total_in, total_out, out_deg[n], in_off[n+1], out_off[n+1], in_src[cap_in], out_dst[cap_out], out_deg_of_dst[cap_out]];
 * in / out rows are listed only for vertices whose out-degree is < th */
int ogl_infer_query(ogl_graph* g, const int64_t* v_dev, int n, int64_t v_off, int th, int cap_in, int cap_out, int64_t* out_dev, void* stream);
int ogl_infer_induced_mean(ogl_graph* g, const uint8_t* member_dev, const int64_t* nodes_dev, int64_t n, const float* proj_dev, int ldp,
                           int n_feats, float* out_dev, int ldo, void* stream);
/* options: "cuda_graph" (default 1), "side_stream" (default 1): ogl_plan_train_step replays a captured CUDA graph of its launch sequence
 * (re-captured when the graph pool, the handles, n_seeds or the output pointers change) */
int ogl_plan_set_option(ogl_plan* p, const char* name, int value);
/* out = {graphs captured, graph replays} */
int ogl_plan_graph_stats(ogl_plan* p, int64_t out[2]);
/* eval: sample + forward + per-vertex CE loss (PBR recompute_priorities, pytorch/model.py:210-254) */
int ogl_plan_eval_step(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_seeds,
                       int seeds_on_host, float* logits_dev, float* per_vertex_loss_dev, void* stream);
/* ---- full-neighbourhood inference (DGL's model.inference(g, x)): every in-edge, no sampling -------------------------------
 * ogl_plan_infer_full: logits [n, classes] fp32 of the plan's model for the vertices seeds_dev[0..n) (device int64; seeds_dev == NULL:
 *   n = the number of vertices of g, all of them, in id order).  Layer by layer over every vertex: relu(fc_pool) over all rows, the
 *   segment max over the whole in-edge row of each vertex, fc_self + fc_neigh; with seeds the last layer runs on the seed rows only.
 *   Evaluation semantics (no feat_drop).  Max-pooling is exact, so the result is bit-reproducible and independent of the order in which
 *   the edges were inserted.  Ordered on `stream`; changes no plan state (Philox / Adam counters, minibatch buffers, pending
 *   prefetches, captured step graphs).  The plan keeps the activations of every layer for all vertices ([V, pitch] tables, allocated
 *   on first use, grown with the graph, freed with the plan): a graph whose activations do not fit in device memory fails with
 *   OGL_ERR_CAPACITY.  A seed id outside [0, n_vertices) is replaced by vertex 0 and raises bit 0 of ogl_plan_error_flags.
 *   Destination shards (ogl_graph_set_source_bound) are rejected.  It is a loop of ogl_plan_infer_full_layer over the layers.
 *   With seeds, a hidden layer l runs on S_l only, S_{L-1} = the seeds, S_l = S_{l+1} u N_in(S_{l+1}) (ogl_graph_in_frontier),
 *   from the top down as long as S_l costs sum(in-degree + 1) <= 0.9 (E + V); that layer and every layer below it run over all
 *   rows otherwise.  The result is bit-identical either way.  Each expanded layer synchronises `stream` once: the size of S_l is
 *   copied to the host to size the layer's launches.
 * ogl_plan_infer_full_layer: layer `layer` of ogl_plan_infer_full for the destination rows rows_dev[0..n) (device int64) or, with
 *   rows_dev == NULL, [row0, row0 + n) (within [0, n_vertices)): hp = relu(h Wp^T + bp) over ALL vertices of g (h = f's table for
 *   layer 0, h_dev is then unused; else h_dev [n_vertices, ldh] in the storage type, ldh = round_up(layer's input width, 8), 16-byte
 *   aligned), the segment max over the listed rows, out[0..n) = [h_r | neigh_r] [Ws | Wn]^T + b: ReLU and the storage type with
 *   ldo = round_up(layer's output width, 8) for a hidden layer, fp32 logits with ldo >= classes for the last.  Every row is computed on
 *   its own, so any split of the rows gives the bits of the one call over all of them (data-parallel inference: each rank runs its
 *   rows, then the ranks exchange them).  n == 0 is a no-op.  Same state guarantees, workspace and errors as ogl_plan_infer_full.
 * ogl_graph_segment_max: the segment max on its own: out[r, :cols] = max over the in-edges (u -> v_r) of x[u, :cols], 0 for a vertex
 *   without in-edges, v_r = rows_dev[r] (rows_dev == NULL: v_r = r and n_rows must be the vertex count).  x [*, ld] holds a row for
 *   every vertex of g in the storage type of `mode` (OGL_F32 / OGL_TF32: fp32, OGL_BF16: bf16, OGL_FP16: fp16); x and out 16-byte
 *   aligned, ld and ldo multiples of 16 bytes; columns are written in 16-byte strips up to round_up(cols, 16 bytes) <= ldo.  A listed
 *   id outside [0, n_vertices) gives a zero row.  Synchronises `stream` (it frees its scratch before returning).
 * ogl_graph_in_frontier: the in-neighbourhood frontier of rows_dev[0..n) (device int64; ids outside [0, n_vertices) are ignored):
 *   out_rows_dev (device int32, capacity n_vertices) receives the distinct vertices of S u N_in(S) in ascending order, *out_n their
 *   number and *out_edge_cost the sum over them of (in-degree + 1), the rows and edges a segment max over them reads.  Reads the
 *   streaming CSR in place (vertex-stream prefixes included).  Synchronises `stream` (it frees its scratch before returning).
 * ogl_plan_infer_full_loss: ogl_plan_infer_full followed by the per-vertex cross entropy on its logits (PBR priorities from exact
 *   neighbourhoods, pytorch/model.py:210-254): per_vertex_loss_dev[r] = logsumexp(logits[r, :classes]) - logits[r, y] (fp32 [n]),
 *   y = f's label of seed r (of vertex r without seeds).  logits_dev (fp32 [n, classes]) may be NULL; when given it receives the
 *   logits, bit-identical to ogl_plan_infer_full's.  The loss is the training loss's arithmetic (ogl_plan_loss_backward,
 *   ogl_plan_eval_step): equal logits give bit-equal losses.  Same state guarantees, workspace and rejections as
 *   ogl_plan_infer_full; an out-of-range seed id uses vertex 0 (logits and label) and raises bit 0, a label outside [0, classes)
 *   gives NaN and raises bit 1 of ogl_plan_error_flags.
 * ogl_plan_full_xent: that loss on its own over a caller's fp32 logits block [n, ld] (ld >= classes, the plan's class count): row r
 *   belongs to vertex rows_dev[r] (device int64) or, with rows_dev == NULL, row0 + r (within the feature store's rows).  A listed id
 *   outside [0, the feature store's vertex capacity) uses vertex 0's label and raises bit 0; a label outside [0, classes) gives NaN
 *   and raises bit 1.  n == 0 is a no-op.  Ordered on `stream`, no host synchronisation; changes no plan state but the error flags.
 *   Data-parallel priorities run the last layer on a rank's rows (ogl_plan_infer_full_layer), this loss on them, and exchange
 *   only the losses. */
int ogl_plan_infer_full(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds_dev, int64_t n, float* logits_dev,
                        void* stream);
int ogl_plan_infer_full_layer(ogl_plan* p, ogl_graph* g, ogl_features* f, int layer, const void* h_dev, int ldh,
                              const int64_t* rows_dev, int64_t row0, int64_t n, void* out_dev, int ldo, void* stream);
int ogl_plan_infer_full_loss(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds_dev, int64_t n,
                             float* logits_dev /* may be NULL */, float* per_vertex_loss_dev, void* stream);
int ogl_plan_full_xent(ogl_plan* p, ogl_features* f, const float* logits_dev, int ld, const int64_t* rows_dev, int64_t row0,
                       int64_t n, float* per_vertex_loss_dev, void* stream);
int ogl_graph_segment_max(ogl_graph* g, int mode, const void* x_dev, int ld, int cols, const int64_t* rows_dev, int64_t n_rows,
                          void* out_dev, int ldo, void* stream);
int ogl_graph_in_frontier(ogl_graph* g, const int64_t* rows_dev, int64_t n, int32_t* out_rows_dev, int64_t* out_n,
                          int64_t* out_edge_cost, void* stream);

/* stage profiling for bench.py's roofline: CUDA events recorded around every stage of the plan's calls on the
 * caller's stream (off by default).  enable=1 (re)starts a collection.  _read synchronises the device and returns,
 * per stage, the summed milliseconds and kernel launches, plus the per-level node counts summed over the
 * profiled train steps (level 0 = seeds ... level L = input nodes). names are '\n'-separated. */
int ogl_plan_profile(ogl_plan* p, int enable);
int ogl_plan_profile_read(ogl_plan* p, char* names_buf, int names_len, float* ms_out, int64_t* launches_out, int max_stages,
                          int* n_stages, int64_t* level_count_sums, int* n_steps);

/* introspection for parity tests: device pointers into the plan's workspaces.
 * level 0 = seeds, level l+1 = src nodes of hop l.  block(hop) = dst level hop. */
int ogl_plan_level_nodes(ogl_plan* p, int level, const int32_t** nodes_dev, const int32_t** count_dev, int* max_count);
int ogl_plan_block_edges(ogl_plan* p, int hop, const int32_t** edge_src_local_dev, const int32_t** edge_src_global_dev,
                         const int64_t** edge_eid_dev, int* fanout);
/* named tensors: "hp<l>", "neigh<l>", "arg<l>", "out<l>" for layer l; "full_h0", "full_h1": the two hidden tables of full inference
 * (raw [rows, widest hidden pitch] blocks, after its first call); returns pointer, rows(max), pitch, elem bytes */
int ogl_plan_tensor(ogl_plan* p, const char* name, const void** ptr_dev, int* rows_max, int* pitch, int* elem_bytes);

/* standalone sampler (config 5 sweep + tests): picks into caller buffers.
 * out_src_dev int32 [n*fanout] (-1 for empty rows), out_eid_dev int64 or NULL */
int ogl_sample_neighbors(ogl_graph* g, const int64_t* dst_dev, int64_t n, int fanout, uint64_t seed,
                         uint32_t step, uint32_t hop, int32_t* out_src_dev, int64_t* out_eid_dev, void* stream);

/* ------------------------------------------------------------------ replay ----------
 * RBR: uniform n-subset of a population of size n_pop (train/graph/train_test_graph.py:210-216;
 * counter-RNG replacement of the in-place random.shuffle).  out_idx_dev int64 [n].
 * PBR: fp64 sum-tree (train/prioritized_replay/segment_tree.py:69-79,94-125) and the
 * stratified proportional draw (replay_buffer.py:164-203).
 */
int ogl_draw_uniform(int64_t n_pop, int64_t n, uint64_t seed, uint32_t counter, int64_t* out_idx_dev, void* stream);

int ogl_sumtree_create(ogl_sumtree** out, int64_t capacity_pow2);
int ogl_sumtree_destroy(ogl_sumtree* t);
int ogl_sumtree_set(ogl_sumtree* t, const int64_t* idx_dev, const double* val_dev, int64_t n, void* stream);
/* leaf[idx] = transform(loss): clip -> log -> running min/max normalise -> +eps -> pow(alpha)
 * (replay_buffer.py:110-130,219-244).  minmax_io_dev = {min_val,max_val,min_log,max_log} running state */
int ogl_sumtree_set_from_loss(ogl_sumtree* t, const int64_t* idx_dev, const float* loss_dev, int64_t n,
                              double clip_lo, double clip_hi, double eps, double alpha, double* minmax_io_dev, void* stream);
/* sum over leaves [lo, hi) with the reference's association order */
int ogl_sumtree_sum(ogl_sumtree* t, int64_t lo, int64_t hi, double* out_dev, void* stream);
/* out_idx[i] = find_prefixsum_idx(mass[i]) */
int ogl_sumtree_find(ogl_sumtree* t, const double* mass_dev, int64_t n, int64_t* out_idx_dev, void* stream);
/* stratified draw: mass_i = u[i]*(p_total/n) + i*(p_total/n), p_total = sum(0, n_items-1) */
int ogl_sumtree_sample_stratified(ogl_sumtree* t, const double* uniforms_dev, int64_t n, int64_t n_items,
                                  int64_t* out_idx_dev, void* stream);
int ogl_sumtree_values(ogl_sumtree* t, const double** value_dev, int64_t* capacity);

/* ------------------------------------------------------------------ evaluation metrics
 * Replaces `output.argmax(axis=1)` + sklearn.metrics.confusion_matrix on the host (train/graphsage/model.py:83-86): the logits stay
 * on the device, cm_dev[y * n_classes + argmax] is incremented per vertex (int64 [n_classes * n_classes + 1], caller-zeroed; the
 * last slot counts labels outside [0, n_classes)).  The macro-F1 of :86 follows from the matrix. */
int ogl_eval_confusion(const float* logits_dev, int ld, int64_t n, int n_classes, const int64_t* labels_dev, int64_t* cm_dev,
                       void* stream);

/* ------------------------------------------------------------------ dense GEMM (tests / bench) */
/* C[M,N] (fp32, ldc) = A[M,K] (bf16, lda) * B[N,K]^T (bf16, ldb), tcgen05 path */
int ogl_gemm_bf16_nt(const void* a_dev, int lda, const void* b_dev, int ldb, float* c_dev, int ldc,
                     int m, int n, int k, void* stream);
/* same with the fused epilogue options of the plan's GEMMs: bf16 or fp32 output, bias[n], ReLU; cg = 0 auto, 1 one CTA
 * per 128-row tile, 2 CTA pairs (tcgen05 cta_group::2) */
int ogl_gemm_bf16_nt_ex(const void* a_dev, int lda, const void* b_dev, int ldb, void* c_dev, int ldc, int m, int n, int k,
                        int out_bf16, const float* bias_dev, int relu, int cg, void* stream);
/* C[N,K] (fp32, ldc) = A[M,N]^T (bf16, lda) * B[M,K] (bf16, ldb): the weight-gradient shape (contraction over
 * rows), tcgen05 path with MN-major operands; workspace holds the split partials (may be NULL: no split) */
int ogl_gemm_bf16_tn(const void* a_dev, int lda, const void* b_dev, int ldb, float* c_dev, int ldc,
                     int m, int n, int k, float* workspace_dev, int64_t workspace_elems, void* stream);
/* the tcgen05 kind::tf32 flavour of the two calls above (mode OGL_TF32: fp32 operands holding TF32-rounded values, fp32
 * accumulation; the arithmetic that replaces the reference's fp32 cuBLAS GEMMs, train/utils.py:63-64).  tma_out != 0: the
 * activation epilogue (TF32-rounded fp32 output through TMA stores, optional mask: out = mask > 0 ? out : 0) */
int ogl_gemm_tf32_nt_ex(const float* a_dev, int lda, const float* b_dev, int ldb, float* c_dev, int ldc, int m, int n, int k,
                        int tma_out, const float* bias_dev, int relu, const float* mask_dev, int ldmask, int cg, void* stream);
int ogl_gemm_tf32_tn(const float* a_dev, int lda, const float* b_dev, int ldb, float* c_dev, int ldc,
                     int m, int n, int k, float* workspace_dev, int64_t workspace_elems, void* stream);
/* the fp16 flavour (mode OGL_FP16: tcgen05 kind::f16 on fp16 operands -- TF32's 10 mantissa bits in half the bytes).  out_f16: fp16
 * output through TMA stores, optional fp16 mask (out = mask > 0 ? out : 0); alpha scales the weight-gradient output (the plan
 * passes 1 / loss scale: activation gradients are stored times a power of two) */
int ogl_gemm_f16_nt_ex(const void* a_dev, int lda, const void* b_dev, int ldb, void* c_dev, int ldc, int m, int n, int k,
                       int out_f16, const float* bias_dev, int relu, const void* mask_dev, int ldmask, int cg, void* stream);
int ogl_gemm_f16_tn(const void* a_dev, int lda, const void* b_dev, int ldb, float* c_dev, int ldc,
                    int m, int n, int k, float alpha, float* workspace_dev, int64_t workspace_elems, void* stream);

#pragma GCC visibility pop
#ifdef __cplusplus
}
#endif
#endif /* OGL_B200_H_ */
