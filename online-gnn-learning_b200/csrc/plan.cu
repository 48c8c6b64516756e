// Feature store + training plan: sampler -> L x SAGEConv('pool') -> CE loss -> backward -> Adam.
//
// One plan owns every workspace, sized once for max_seeds, and every kernel reads its row
// counts from device memory, so a whole train step is a fixed launch sequence with no host
// synchronisation (CUDA-graph capturable).  Replaces the per-minibatch body of
// train/graphsage/pytorch/model.py:77-107 (train_step) and :39-71 (_run_custom_eval).
#include "graph.cuh"
#include "sample.cuh"
#include "gemm.cuh"
#include "sage_kernels.cuh"
#include "peer.cuh"
#include "full_infer.cuh"
#include <cmath>
#include <vector>
#include <string>

using namespace ogl;

static inline int pitch_of(int d) { return round_up(d, 8); }

// ------------------------------------------------------------------ feature store ----------------
struct ogl_features {
  int64_t v_cap = 0;
  int F = 0, pitch = 0, mode = 0;
  void* table = nullptr;      // [v_cap, pitch] in the mode's storage type (fp32 | bf16 | fp16)
  int32_t* labels = nullptr;  // [v_cap]
  float* stage_f = nullptr;   // host-source staging
  int64_t* stage_l = nullptr;
  int64_t stage_rows = 0;
};

extern "C" int ogl_features_create(ogl_features** out, int64_t v_cap, int n_feats, int mode) {
  OGL_TRY(require_device());
  OGL_ARG(out && v_cap > 0 && n_feats > 0 && mode_valid(mode), "ogl_features_create: bad arguments");
  ogl_features* f = new ogl_features();
  f->v_cap = v_cap; f->F = n_feats; f->pitch = pitch_of(n_feats); f->mode = mode;
  const size_t es = mode_bytes(mode);
  OGL_CUDA(cudaMalloc(&f->table, es * (size_t)v_cap * f->pitch));
  OGL_CUDA(cudaMemset(f->table, 0, es * (size_t)v_cap * f->pitch));
  OGL_CUDA(cudaMalloc(&f->labels, sizeof(int32_t) * v_cap));
  OGL_CUDA(cudaMemset(f->labels, 0, sizeof(int32_t) * v_cap));
  *out = f;
  return OGL_OK;
}

extern "C" int ogl_features_destroy(ogl_features* f) {
  if (!f) return OGL_OK;
  cudaFree(f->table); cudaFree(f->labels); cudaFree(f->stage_f); cudaFree(f->stage_l);
  delete f;
  return OGL_OK;
}

extern "C" int ogl_features_write(ogl_features* f, int64_t row0, int64_t n, const float* feats, const int64_t* labels, int src_is_host,
                                  void* stream) {
  OGL_ARG(f && row0 >= 0 && n >= 0 && row0 + n <= f->v_cap, "ogl_features_write: rows [%lld, %lld) out of range", (long long)row0, (long long)(row0 + n));
  if (n == 0) return OGL_OK;
  cudaStream_t s = (cudaStream_t)stream;
  OGL_TRY(readers_wait(f, s));                 // a prefetched minibatch may still be gathering rows on its plan's stream
  if (src_is_host) {
    // chunked H2D through a device staging buffer (fp32 rows are converted/padded on the GPU)
    const int64_t chunk = 1 << 16;
    if (f->stage_rows < chunk) {
      OGL_CUDA(cudaMalloc(&f->stage_f, sizeof(float) * chunk * f->F));
      OGL_CUDA(cudaMalloc(&f->stage_l, sizeof(int64_t) * chunk));
      f->stage_rows = chunk;
    }
    for (int64_t o = 0; o < n; o += chunk) {
      const int64_t m = n - o < chunk ? n - o : chunk;
      if (feats) {
        OGL_CUDA(cudaMemcpyAsync(f->stage_f, feats + o * f->F, sizeof(float) * m * f->F, cudaMemcpyHostToDevice, s));
        OGL_TRY(feat_write(f->mode, f->stage_f, nullptr, m, f->F, f->table, f->pitch, row0 + o, s));
      }
      if (labels) {
        OGL_CUDA(cudaMemcpyAsync(f->stage_l, labels + o, sizeof(int64_t) * m, cudaMemcpyHostToDevice, s));
        OGL_TRY(label_write(f->stage_l, nullptr, m, f->labels, row0 + o, s));
      }
    }
    return OGL_OK;
  }
  if (feats) OGL_TRY(feat_write(f->mode, feats, nullptr, n, f->F, f->table, f->pitch, row0, s));
  if (labels) OGL_TRY(label_write(labels, nullptr, n, f->labels, row0, s));
  return OGL_OK;
}

extern "C" int ogl_features_write_permuted(ogl_features* f, int64_t n, const float* feats_dev, const int64_t* labels_dev,
                                           const int64_t* src_rows_dev, void* stream) {
  OGL_ARG(f && n >= 0 && n <= f->v_cap && src_rows_dev, "ogl_features_write_permuted: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  OGL_TRY(readers_wait(f, s));
  if (feats_dev) OGL_TRY(feat_write(f->mode, feats_dev, src_rows_dev, n, f->F, f->table, f->pitch, 0, s));
  if (labels_dev) OGL_TRY(label_write(labels_dev, src_rows_dev, n, f->labels, 0, s));
  return OGL_OK;
}

// ------------------------------------------------------------------ plan --------------------------
struct LayerBuf {
  int in = 0, out = 0, pin = 0, pout = 0;
  // offsets into the flat fp32 parameter / gradient buffers
  int64_t o_wp = 0, o_bp = 0, o_ws = 0, o_bs = 0, o_wn = 0, o_bn = 0;
  // shadows in the arithmetic type
  void *wp = nullptr, *wpT = nullptr, *ws = nullptr, *wsT = nullptr, *wn = nullptr, *wnT = nullptr;
  // activations
  void* hp = nullptr;       // [nmax[src], pin]
  void* neigh = nullptr;    // [nmax[dst], pin]
  uint8_t* arg = nullptr;   // [nmax[dst], pin]
  void* dpre = nullptr;     // [nmax[dst], pout]   gradient wrt this layer's pre-activation output
  void* dng = nullptr;      // [nmax[dst], pin]    gradient wrt neigh (per layer: its column sums run on the side stream)
  void* dhp = nullptr;      // [nmax[src], pin]    gradient wrt hp (per layer: the fc_pool weight gradient of layer l is computed
                            //                     later, grouped with layer l-1's fc_self / fc_neigh weight gradients)
};

struct ogl_plan {
  ogl_plan_config cfg;
  int L = 0;
  int mode = 0;                          // = cfg.mode
  size_t es = 4;                         // its storage type's element bytes
  std::vector<int> nmax;                 // [L+1]
  std::vector<int32_t*> nodes;           // [L+1]
  int32_t* counts = nullptr;             // [L+1] device
  std::vector<int32_t*> edge_lid, edge_gsrc;   // [L]
  std::vector<int32_t*> rev_ptr, rev_edge;     // [L] reverse edge lists per hop (source row -> picking slots)
  std::vector<int64_t*> edge_eid;
  std::vector<void*> act;                // [L+1]; act[0] = logits (fp32)
  std::vector<LayerBuf> layer;
  ToBlockWs tb;
  int64_t* seeds_stage = nullptr;
  // software pipeline: everything one sampled minibatch owns (node lists, counts, ELL / reverse edge lists, the gathered input rows,
  // the staged seeds) exists twice, so that sample + gather of minibatch i+1 runs on the `pre` stream while forward / backward /
  // Adam of minibatch i runs on the caller's stream.  The members above / below are the CURRENT set; `alt` is the other one.
  struct SampleBufs {
    std::vector<int32_t*> nodes, edge_lid, edge_gsrc, rev_ptr, rev_edge;
    int32_t* counts = nullptr;
    void* x = nullptr;
    int64_t* seeds_stage = nullptr;
  } alt;
  int have_alt = 0, parity = 0;
  int use_pipeline = 1;
  cudaStream_t pre = nullptr;
  cudaEvent_t ev_tail = nullptr, ev_ready[2] = {nullptr, nullptr};
  int pend[2] = {0, 0};                  // [0]: the current set holds a prefetched minibatch; [1]: `alt` holds the one after it
  int pend_n[2] = {0, 0};
  static constexpr int kSeedRing = 4;
  int64_t* seed_ring = nullptr;          // pinned [kSeedRing][max_seeds]: private copies of host seeds handed to ogl_plan_prefetch
  cudaEvent_t ev_ring[kSeedRing] = {nullptr, nullptr, nullptr, nullptr};
  int ring_next = 0;
  int cur_open = 0;                      // ogl_plan_step_begin filled the current set and its finish has not been enqueued yet
  uint32_t* ctl = nullptr;               // [0]=philox step, [1]=adam t, [2]=error flags, [3]=direct training-mode forwards
  int n_seeds = 0;
  // backward scratch
  float* tn_partial = nullptr;
  int64_t tn_partial_elems = 0;
  float* colsum_partial = nullptr;
  float* per_loss = nullptr;
  float* loss_sum = nullptr;
  // parameters
  int64_t n_params = 0;
  float *params = nullptr, *grads = nullptr, *adam_m = nullptr, *adam_v = nullptr;
  ShadowSeg* shadow_segs = nullptr;      // device table for the fused Adam + shadow refresh
  int n_shadow_segs = 0;
  // independent work of a step runs on a side stream (forked / joined with events, also inside graph capture):
  // the weight / bias gradients of fc_self and fc_neigh overlap the dneigh -> pool_bwd -> dW_pool -> dx chain
  int use_side = 1;
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  float head_loss_scale = 0.f;           // loss scale of the last ogl_plan_step_finish_head (its tail must unscale by the same)
  float grad_scale = 1.f;                // mode OGL_FP16: the loss scale the stored activation gradients of the current backward pass carry
  int skip_gather = 0;                   // step_finish: the input rows were already gathered by step_begin
  int train_mode = 0;                    // feat_drop is applied by ogl_plan_forward (train steps set it; eval steps never)
  int adam_in_backward = 0;              // fused step with do_step: the backward pass runs Adam on all but the last gradient itself
  int64_t adam_done_from = 0;            // ... and leaves [0, adam_done_from) to ogl_plan_adam_step
  ogl_peer* dp_peer = nullptr;           // step kind 5: the peer group of the data-parallel finish being enqueued / captured
  int tail_mode = 0;                     // backward: 0 = all, 1 = everything but the last weight-gradient GEMM (layer 0 fc_pool),
                                         // 2 = only that GEMM (data-parallel: its predecessors' gradients are already on the wire)
  int in_train_step = 0;                 // set by the fused train step: sampling may defer the reverse edge lists to the side stream
  int side_pending = 0;                  // side-stream work not yet joined into the main stream
  float* tn_partial2 = nullptr;          // split workspace of the side-stream TN GEMMs
  float* colsum_partial2 = nullptr;
  // CUDA-graph replay of the train step (fixed launch sequence, all sizes read from device memory)
  int use_graph = 1;
  struct StepKey {
    const void *g, *f, *per, *loss;
    uint64_t g_gen;
    int n_seeds, do_step;
    float loss_scale;
    int kind;            // 0 = whole step, 1 = step_begin (sample + gather), 2 = step_finish (forward .. Adam),
                         // 3 = step_finish minus the last weight-gradient GEMM, 4 = that GEMM, 5 = data-parallel finish
    int parity;          // which of the two minibatch buffer sets the captured pointers belong to
    bool operator==(const StepKey& o) const {
      return g == o.g && f == o.f && per == o.per && loss == o.loss && g_gen == o.g_gen && n_seeds == o.n_seeds && do_step == o.do_step &&
             loss_scale == o.loss_scale && kind == o.kind && parity == o.parity;
    }
  };
  struct StepGraph { StepKey key; cudaGraphExec_t exec; uint64_t last_use; };
  std::vector<StepGraph> step_graphs;    // small LRU
  uint64_t graph_clock = 0;
  cudaStream_t cap_stream = nullptr;
  long long graph_replays = 0, graph_captures = 0;
  // stage profiling (bench.py roofline): CUDA events around every stage, on the caller's stream
  int prof_on = 0;
  std::vector<std::string> prof_names;
  struct ProfRec { int stage; cudaEvent_t e0, e1; long long launches; };
  std::vector<ProfRec> prof_recs;
  size_t prof_used = 0;
  int32_t* prof_counts_host = nullptr;   // pinned [kProfSteps][8]
  int prof_steps = 0;
  // full-neighbourhood inference (ogl_plan_infer_full): its own activations over every vertex, allocated on first use and grown
  // geometrically with the graph; nothing of the train / eval state above is read or written by it except the weights
  struct FullWs {
    int64_t rows = 0;                    // row capacity (a multiple of 128)
    void *hp = nullptr, *neigh = nullptr, *hs = nullptr, *h[2] = {nullptr, nullptr};
    void* hc = nullptr;                  // a frontier layer's output rows, compact, before the scatter into h[]
    float* logits = nullptr;
    int32_t* seeds = nullptr;
    int32_t* front = nullptr;            // [L - 1][rows]: the rows hidden layer l needs when it runs on a frontier
    SegmaxWs sm;
    FrontierWs fr;
    FrontierOut* fr_host = nullptr;      // pinned
  } full;
};
constexpr int kProfSteps = 4096;

static void prof_begin(ogl_plan* p, const char* name, cudaStream_t s) {
  if (!p->prof_on) return;
  int stage = -1;
  for (size_t i = 0; i < p->prof_names.size(); ++i)
    if (p->prof_names[i] == name) { stage = (int)i; break; }
  if (stage < 0) { p->prof_names.push_back(name); stage = (int)p->prof_names.size() - 1; }
  if (p->prof_used == p->prof_recs.size()) {
    ogl_plan::ProfRec r;
    cudaEventCreate(&r.e0);
    cudaEventCreate(&r.e1);
    p->prof_recs.push_back(r);
  }
  ogl_plan::ProfRec& r = p->prof_recs[p->prof_used];
  r.stage = stage;
  r.launches = g_launches.load();
  cudaEventRecord(r.e0, s);
}
static void prof_end(ogl_plan* p, cudaStream_t s) {
  if (!p->prof_on) return;
  ogl_plan::ProfRec& r = p->prof_recs[p->prof_used++];
  r.launches = g_launches.load() - r.launches;
  cudaEventRecord(r.e1, s);
}
// stage profiling: the level row counts of the step just enqueued, for the per-step averages of ogl_plan_profile_read
static int record_level_counts(ogl_plan* p, cudaStream_t s) {
  if (p->prof_on && p->prof_steps < kProfSteps) {
    OGL_CUDA(cudaMemcpyAsync(p->prof_counts_host + 8 * p->prof_steps, p->counts, sizeof(int32_t) * (p->L + 1), cudaMemcpyDeviceToHost, s));
    p->prof_steps++;
  }
  return OGL_OK;
}
#define STAGE(name, call)            \
  do {                               \
    prof_begin(p, name, s);          \
    int _sr = (call);                \
    prof_end(p, s);                  \
    if (_sr != OGL_OK) return _sr;   \
  } while (0)
#define STAGE_ON(st, name, call)     \
  do {                               \
    prof_begin(p, name, st);         \
    int _sr = (call);                \
    prof_end(p, st);                 \
    if (_sr != OGL_OK) return _sr;   \
  } while (0)
static std::string nm(const char* fmt, int i) {
  char b[64];
  snprintf(b, sizeof(b), fmt, i);
  return b;
}

static int dmalloc0(void** ptr, size_t bytes) {
  OGL_CUDA(cudaMalloc(ptr, bytes ? bytes : 16));
  OGL_CUDA(cudaMemset(*ptr, 0, bytes ? bytes : 16));
  return OGL_OK;
}
#define DM0(ptr, bytes) OGL_TRY(dmalloc0((void**)&(ptr), (size_t)(bytes)))

extern "C" int64_t ogl_plan_param_count(const ogl_plan* p) { return p ? p->n_params : 0; }

extern "C" int ogl_plan_create(ogl_plan** out, const ogl_plan_config* cfg) {
  OGL_TRY(require_device());
  OGL_ARG(out && cfg, "ogl_plan_create: null");
  OGL_ARG(cfg->n_layers >= 1 && cfg->n_layers <= 7, "ogl_plan_create: n_layers must be in [1,7]");
  OGL_ARG(cfg->max_seeds > 0 && cfg->v_cap > 0, "ogl_plan_create: max_seeds / v_cap must be positive");
  OGL_ARG(mode_valid(cfg->mode), "ogl_plan_create: bad mode");
  OGL_ARG(cfg->feat_drop >= 0.f && cfg->feat_drop < 1.f, "ogl_plan_create: feat_drop must be in [0, 1)");
  for (int i = 0; i <= cfg->n_layers; ++i) OGL_ARG(cfg->dims[i] > 0, "ogl_plan_create: dims[%d] must be positive", i);
  for (int i = 0; i < cfg->n_layers; ++i) OGL_ARG(cfg->fanouts[i] > 0 && cfg->fanouts[i] < 255, "ogl_plan_create: fanouts[%d] must be in [1,254]", i);
  ogl_plan* p = new ogl_plan();
  p->cfg = *cfg;
  const int L = p->L = cfg->n_layers;
  p->mode = cfg->mode;
  p->es = mode_bytes(cfg->mode);
  p->nmax.resize(L + 1);
  p->nmax[0] = cfg->max_seeds;
  for (int h = 0; h < L; ++h) {
    // a frontier = the destination rows themselves (seed lists may hold duplicates, DGL allows them) + the distinct new sources
    int64_t n = (int64_t)p->nmax[h] * (1 + cfg->fanouts[h]);
    if (n > cfg->v_cap + p->nmax[h]) n = cfg->v_cap + p->nmax[h];
    p->nmax[h + 1] = (int)n;
  }
  for (int h = 0; h < L; ++h)
    if (p->nmax[h] >= (1 << 23)) {
      set_error("ogl_plan_create: level %d may hold %d destination rows; the packed reverse edge entries allow < 2^23", h, p->nmax[h]);
      delete p;
      return OGL_ERR_ARG;
    }
  p->nodes.resize(L + 1); p->act.resize(L + 1);
  p->edge_lid.resize(L); p->edge_gsrc.resize(L); p->edge_eid.resize(L); p->layer.resize(L);
  p->rev_ptr.resize(L); p->rev_edge.resize(L);
  DM0(p->counts, sizeof(int32_t) * (L + 1));
  DM0(p->ctl, sizeof(uint32_t) * 4);
  DM0(p->seeds_stage, sizeof(int64_t) * cfg->max_seeds);
  int64_t ne_max = 0;
  for (int lv = 0; lv <= L; ++lv) DM0(p->nodes[lv], sizeof(int32_t) * p->nmax[lv]);
  for (int h = 0; h < L; ++h) {
    const int64_t ne = (int64_t)p->nmax[h] * cfg->fanouts[h];
    if (ne > ne_max) ne_max = ne;
    DM0(p->edge_lid[h], sizeof(int32_t) * ne);
    DM0(p->edge_gsrc[h], sizeof(int32_t) * ne);
    DM0(p->edge_eid[h], sizeof(int64_t) * ne);
    DM0(p->rev_ptr[h], sizeof(int32_t) * ((size_t)p->nmax[h + 1] + 2));
    DM0(p->rev_edge[h], sizeof(int32_t) * ne);
  }
  OGL_TRY(to_block_init(&p->tb, cfg->v_cap, ne_max, p->nmax[L]));
  // activations (row counts padded to 128 for the zero-tail rule)
  auto rows = [](int n) { return (size_t)round_up(n, 128); };
  DM0(p->act[L], p->es * rows(p->nmax[L]) * pitch_of(cfg->dims[0]));
  int64_t off = 0, max_nk = 0, max_colsum = 0;
  for (int l = 0; l < L; ++l) {
    LayerBuf& lb = p->layer[l];
    const int h = L - 1 - l, s = h + 1, d = h;
    lb.in = cfg->dims[l]; lb.out = cfg->dims[l + 1]; lb.pin = pitch_of(lb.in); lb.pout = pitch_of(lb.out);
    lb.o_wp = off; off += (int64_t)lb.in * lb.in;
    lb.o_bp = off; off += lb.in;
    lb.o_ws = off; off += (int64_t)lb.out * lb.in;
    lb.o_bs = off; off += lb.out;
    lb.o_wn = off; off += (int64_t)lb.out * lb.in;
    lb.o_bn = off; off += lb.out;
    DM0(lb.wp, p->es * (size_t)lb.in * lb.pin);
    DM0(lb.wpT, p->es * (size_t)lb.in * lb.pin);
    DM0(lb.ws, p->es * (size_t)lb.out * lb.pin);
    DM0(lb.wsT, p->es * (size_t)lb.in * lb.pout);
    DM0(lb.wn, p->es * (size_t)lb.out * lb.pin);
    DM0(lb.wnT, p->es * (size_t)lb.in * lb.pout);
    DM0(lb.hp, p->es * rows(p->nmax[s]) * lb.pin);
    DM0(lb.neigh, p->es * rows(p->nmax[d]) * lb.pin);
    DM0(lb.arg, rows(p->nmax[d]) * lb.pin);
    DM0(lb.dpre, p->es * rows(p->nmax[d]) * lb.pout);
    DM0(lb.dhp, p->es * rows(p->nmax[s]) * lb.pin);
    DM0(lb.dng, p->es * rows(p->nmax[d]) * lb.pin);
    // layer output: logits are always fp32
    const size_t oes = (l == L - 1) ? 4 : p->es;
    DM0(p->act[d], oes * rows(p->nmax[d]) * lb.pout);
    max_nk = std::max<int64_t>(max_nk, (int64_t)std::max(lb.in, lb.out) * lb.in);
    max_colsum = std::max<int64_t>(max_colsum, colsum_partial_elems(p->nmax[d], lb.pin));
    max_colsum = std::max<int64_t>(max_colsum, colsum_partial_elems(p->nmax[d], lb.pout));
  }
  p->n_params = off;
  {
    std::vector<ShadowSeg> segs;
    for (auto& lb : p->layer) {
      segs.push_back({lb.o_wp, lb.o_wp + (int64_t)lb.in * lb.in, lb.in, lb.in, lb.pin, lb.pin, lb.wp, lb.wpT});
      segs.push_back({lb.o_ws, lb.o_ws + (int64_t)lb.out * lb.in, lb.out, lb.in, lb.pin, lb.pout, lb.ws, lb.wsT});
      segs.push_back({lb.o_wn, lb.o_wn + (int64_t)lb.out * lb.in, lb.out, lb.in, lb.pin, lb.pout, lb.wn, lb.wnT});
    }
    p->n_shadow_segs = (int)segs.size();
    DM0(p->shadow_segs, sizeof(ShadowSeg) * segs.size());
    OGL_CUDA(cudaMemcpy(p->shadow_segs, segs.data(), sizeof(ShadowSeg) * segs.size(), cudaMemcpyHostToDevice));
  }
  p->tn_partial_elems = max_nk * 32;
  DM0(p->tn_partial, sizeof(float) * p->tn_partial_elems);
  DM0(p->colsum_partial, sizeof(float) * max_colsum);
  DM0(p->tn_partial2, sizeof(float) * p->tn_partial_elems);
  DM0(p->colsum_partial2, sizeof(float) * max_colsum);
  OGL_CUDA(cudaStreamCreateWithFlags(&p->side, cudaStreamNonBlocking));
  OGL_CUDA(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
  OGL_CUDA(cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming));
  DM0(p->per_loss, sizeof(float) * cfg->max_seeds);
  DM0(p->loss_sum, sizeof(float) * 4);
  DM0(p->adam_m, sizeof(float) * p->n_params);
  DM0(p->adam_v, sizeof(float) * p->n_params);
  *out = p;
  return OGL_OK;
}

extern "C" int ogl_plan_destroy(ogl_plan* p) {
  if (!p) return OGL_OK;
  readers_remove_owner(p);
  for (auto x : p->nodes) cudaFree(x);
  for (auto x : p->edge_lid) cudaFree(x);
  for (auto x : p->edge_gsrc) cudaFree(x);
  for (auto x : p->edge_eid) cudaFree(x);
  for (auto x : p->rev_ptr) cudaFree(x);
  for (auto x : p->rev_edge) cudaFree(x);
  for (auto x : p->act) cudaFree(x);
  for (auto& lb : p->layer) {
    void* ptrs[] = {lb.wp, lb.wpT, lb.ws, lb.wsT, lb.wn, lb.wnT, lb.hp, lb.neigh, lb.arg, lb.dpre, lb.dhp, lb.dng};
    for (void* q : ptrs) cudaFree(q);
  }
  to_block_free(&p->tb);
  for (auto* v : {&p->alt.nodes, &p->alt.edge_lid, &p->alt.edge_gsrc, &p->alt.rev_ptr, &p->alt.rev_edge})
    for (auto x : *v) cudaFree(x);
  cudaFree(p->alt.counts); cudaFree(p->alt.x); cudaFree(p->alt.seeds_stage);
  void* ptrs[] = {p->counts, p->ctl, p->seeds_stage, p->tn_partial, p->colsum_partial, p->per_loss,
                  p->loss_sum, p->adam_m, p->adam_v, p->shadow_segs};
  for (void* q : ptrs) cudaFree(q);
  for (auto& r : p->prof_recs) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
  cudaDeviceSynchronize();
  if (p->side) cudaStreamDestroy(p->side);
  if (p->pre) cudaStreamDestroy(p->pre);
  for (cudaEvent_t e : {p->ev_tail, p->ev_ready[0], p->ev_ready[1], p->ev_ring[0], p->ev_ring[1], p->ev_ring[2], p->ev_ring[3]})
    if (e) cudaEventDestroy(e);
  if (p->seed_ring) cudaFreeHost(p->seed_ring);
  if (p->ev_fork) cudaEventDestroy(p->ev_fork);
  if (p->ev_join) cudaEventDestroy(p->ev_join);
  cudaFree(p->tn_partial2); cudaFree(p->colsum_partial2);
  for (auto& sg : p->step_graphs) cudaGraphExecDestroy(sg.exec);
  if (p->cap_stream) cudaStreamDestroy(p->cap_stream);
  if (p->prof_counts_host) cudaFreeHost(p->prof_counts_host);
  for (void* q : {p->full.hp, p->full.neigh, p->full.hs, p->full.h[0], p->full.h[1], p->full.hc, (void*)p->full.logits, (void*)p->full.seeds,
                  (void*)p->full.front})
    cudaFree(q);
  segmax_ws_free(&p->full.sm);
  frontier_ws_free(&p->full.fr);
  if (p->full.fr_host) cudaFreeHost(p->full.fr_host);
  delete p;
  return OGL_OK;
}

extern "C" int ogl_plan_refresh_params(ogl_plan* p, void* stream) {
  OGL_ARG(p && p->params, "ogl_plan_refresh_params: parameters not bound");
  cudaStream_t s = (cudaStream_t)stream;
  for (auto& lb : p->layer) {
    OGL_TRY(weight_shadow(p->mode, p->params + lb.o_wp, lb.in, lb.in, lb.wp, lb.pin, lb.wpT, lb.pin, s));
    OGL_TRY(weight_shadow(p->mode, p->params + lb.o_ws, lb.out, lb.in, lb.ws, lb.pin, lb.wsT, lb.pout, s));
    OGL_TRY(weight_shadow(p->mode, p->params + lb.o_wn, lb.out, lb.in, lb.wn, lb.pin, lb.wnT, lb.pout, s));
  }
  return OGL_OK;
}

extern "C" int ogl_plan_bind_params(ogl_plan* p, float* params_dev, float* grads_dev, void* stream) {
  OGL_ARG(p && params_dev && grads_dev, "ogl_plan_bind_params: null");
  OGL_ARG(!p->pend[0] && !p->pend[1], "ogl_plan_bind_params: a prefetched minibatch is pending");
  if (params_dev != p->params || grads_dev != p->grads) {          // captured step graphs hold the old pointers
    OGL_CUDA(cudaDeviceSynchronize());
    for (auto& sg : p->step_graphs) cudaGraphExecDestroy(sg.exec);
    p->step_graphs.clear();
  }
  p->params = params_dev;
  p->grads = grads_dev;
  return ogl_plan_refresh_params(p, stream);
}

extern "C" int ogl_plan_set_step(ogl_plan* p, uint32_t step, void* stream) {
  OGL_ARG(p, "null");
  OGL_CUDA(cudaMemcpyAsync(p->ctl, &step, sizeof(uint32_t), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  OGL_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return OGL_OK;
}

// a fresh optimiser: Adam moments and step counter zeroed, Philox step set (build_optimizer() of the reference constructs a new
// torch.optim.Adam, pytorch/model.py:22-25); also what a replica needs to replay a run from its start
extern "C" int ogl_plan_reset_optimizer(ogl_plan* p, uint32_t philox_step, void* stream) {
  OGL_ARG(p, "ogl_plan_reset_optimizer: null");
  OGL_ARG(!p->pend[0] && !p->pend[1], "ogl_plan_reset_optimizer: a prefetched minibatch is pending");
  cudaStream_t s = (cudaStream_t)stream;
  OGL_CUDA(cudaMemsetAsync(p->adam_m, 0, sizeof(float) * p->n_params, s));
  OGL_CUDA(cudaMemsetAsync(p->adam_v, 0, sizeof(float) * p->n_params, s));
  const uint32_t ctl[2] = {philox_step, 0u};
  OGL_CUDA(cudaMemcpyAsync(p->ctl, ctl, sizeof(ctl), cudaMemcpyHostToDevice, s));
  OGL_CUDA(cudaMemsetAsync(p->ctl + 3, 0, sizeof(uint32_t), s));
  OGL_CUDA(cudaStreamSynchronize(s));
  return OGL_OK;
}

__global__ void k_set_i32(int32_t* p, int32_t v) { *p = v; }

extern "C" int ogl_plan_sample(ogl_plan* p, ogl_graph* g, const int64_t* seeds_dev, int n_seeds, void* stream) {
  OGL_ARG(p && g && seeds_dev, "ogl_plan_sample: null");
  OGL_ARG(n_seeds > 0 && n_seeds <= p->cfg.max_seeds, "ogl_plan_sample: n_seeds %d not in [1, %d]", n_seeds, p->cfg.max_seeds);
  OGL_ARG(p->in_train_step || !p->pend[0], "ogl_plan_sample: a prefetched minibatch is pending (run its train step first)");
  cudaStream_t s = (cudaStream_t)stream;
  const GraphView gv = graph_view(g);
  OGL_ARG(gv.n_vertices <= p->cfg.v_cap, "ogl_plan_sample: graph has more vertices than the plan's v_cap");
  p->n_seeds = n_seeds;
  OGL_TRY(cast_nodes(seeds_dev, p->nodes[0], n_seeds, gv.n_vertices, p->ctl + 2, s));
  OGL_LAUNCH(k_set_i32, 1, 1, 0, s, p->counts, n_seeds);
  for (int h = 0; h < p->L; ++h) {
    STAGE(nm("sample.h%d", h).c_str(), sample_hop(gv, p->nodes[h], p->counts + h, p->nmax[h], p->cfg.fanouts[h], p->cfg.seed, p->ctl, 0,
                                                  (uint32_t)h, p->edge_gsrc[h],
                                                  p->in_train_step ? nullptr : p->edge_eid[h],   // edge ids: only the DGL-style block API reads them
                                                  s));
    STAGE(nm("to_block.h%d", h).c_str(), to_block(&p->tb, p->nodes[h], p->counts + h, p->nmax[h], p->cfg.fanouts[h], p->edge_gsrc[h],
                                                  p->nodes[h + 1], p->counts + h + 1, p->nmax[h + 1], p->edge_lid[h], s));
    // reverse edge lists (only the backward pass reads them): inside the fused train step they are built on the side
    // stream, overlapping the next hop's sampling and the forward pass; joined at the start of the backward pass
    if (p->in_train_step && p->use_side && !p->prof_on) {
      OGL_CUDA(cudaEventRecord(p->ev_fork, s));
      OGL_CUDA(cudaStreamWaitEvent(p->side, p->ev_fork, 0));
      OGL_TRY(reverse_edges(&p->tb, p->edge_lid[h], p->counts + h, p->nmax[h], p->cfg.fanouts[h], p->nmax[h + 1], p->rev_ptr[h],
                            p->rev_edge[h], p->side));
      p->side_pending = 1;
    } else {
      STAGE(nm("rev_edges.h%d", h).c_str(), reverse_edges(&p->tb, p->edge_lid[h], p->counts + h, p->nmax[h], p->cfg.fanouts[h],
                                                          p->nmax[h + 1], p->rev_ptr[h], p->rev_edge[h], s));
    }
  }
  return OGL_OK;
}

// the forward GEMMs of layer l, shared by the sampled forward and full-neighbourhood inference (m_dev: the dynamic row count, or
// nullptr for m_max rows).  The pool GEMM: hp = relu(x Wp^T + bp)
static int pool_gemm(const ogl_plan* p, int l, const void* x, int ldx, void* hp, int ldhp, int m_max, const int32_t* m_dev, cudaStream_t s) {
  const LayerBuf& lb = p->layer[l];
  GemmNT g;
  g.a[0] = x; g.lda[0] = ldx; g.b[0] = lb.wp; g.ldb[0] = lb.pin; g.k[0] = lb.in; g.n_seg = 1;
  g.bias = p->params + lb.o_bp; g.relu = 1;
  g.c = hp; g.ldc = ldhp; g.m_max = m_max; g.m_dev = m_dev; g.n = lb.in; g.mode = p->mode;
  return gemm_nt(g, p->cfg.gemm_impl, s);
}
// the output GEMM: [h_self | neigh] [Ws | Wn]^T + bs + bn, with ReLU and in the storage type for a hidden layer, fp32 logits for the last
static int out_gemm(const ogl_plan* p, int l, const void* self, int ld_self, const void* neigh, int ld_neigh, void* out, int ldo, int m_max,
                    const int32_t* m_dev, cudaStream_t s) {
  const LayerBuf& lb = p->layer[l];
  const bool last = l == p->L - 1;
  GemmNT g;
  g.a[0] = self; g.lda[0] = ld_self; g.b[0] = lb.ws; g.ldb[0] = lb.pin; g.k[0] = lb.in;
  g.a[1] = neigh; g.lda[1] = ld_neigh; g.b[1] = lb.wn; g.ldb[1] = lb.pin; g.k[1] = lb.in; g.n_seg = 2;
  g.bias = p->params + lb.o_bs; g.bias2 = p->params + lb.o_bn; g.relu = !last;
  g.c = out; g.ldc = ldo; g.m_max = m_max; g.m_dev = m_dev; g.n = lb.out; g.mode = p->mode; g.out_f32 = last;
  return gemm_nt(g, p->cfg.gemm_impl, s);
}

// drop_step: the device word that keys feat_drop's mask (the last Philox counter word).  A fused step passes its optimiser step
// ctl[1]; a direct ogl_plan_forward passes ctl[3], see there.
static int plan_forward(ogl_plan* p, ogl_features* f, float* logits_dev, const uint32_t* drop_step, cudaStream_t s) {
  OGL_ARG(p && p->params, "ogl_plan_forward: null / parameters not bound");
  OGL_ARG(!f || (f->mode == p->cfg.mode && f->F == p->cfg.dims[0]), "ogl_plan_forward: feature store does not match the plan (mode/F)");
  OGL_ARG(p->n_seeds > 0, "ogl_plan_forward: no minibatch sampled");
  const int L = p->L;
  // f == NULL: the input rows were supplied by ogl_plan_set_input
  if (f && !p->skip_gather)
    STAGE("gather", gather_rows(p->mode, f->table, f->pitch, p->nodes[L], p->counts + L, p->nmax[L], p->act[L], s));
  const bool drop = p->train_mode && p->cfg.feat_drop > 0.f;
  for (int l = 0; l < L; ++l) {
    LayerBuf& lb = p->layer[l];
    const int h = L - 1 - l, sl = h + 1, dl = h;
    // feat_drop: the layer's input rows are dropped out once, in place (they feed fc_pool, h_self and the weight gradients alike)
    if (drop)
      STAGE(nm("l%d.feat_drop", l).c_str(), feat_drop(p->mode, p->act[sl], lb.pin, lb.in, p->counts + sl, p->nmax[sl], p->cfg.feat_drop,
                                                      p->cfg.seed, drop_step, l, s));
    STAGE(nm("l%d.pool_gemm", l).c_str(), pool_gemm(p, l, p->act[sl], lb.pin, lb.hp, lb.pin, p->nmax[sl], p->counts + sl, s));
    STAGE(nm("l%d.segmax", l).c_str(),
          segmax_fwd(p->mode, lb.hp, lb.pin, p->edge_lid[h], p->cfg.fanouts[h], p->counts + dl, p->nmax[dl], lb.neigh, lb.arg, s));
    // (the destination rows are the first rows of the source level)
    STAGE(nm("l%d.out_gemm", l).c_str(),
          out_gemm(p, l, p->act[sl], lb.pin, lb.neigh, lb.pin, p->act[dl], lb.pout, p->nmax[dl], p->counts + dl, s));
  }
  if (logits_dev)
    OGL_TRY(unpad_copy((const float*)p->act[0], p->layer[L - 1].pout, p->nmax[0], p->counts, p->cfg.dims[L], logits_dev, s));
  return OGL_OK;
}

// A direct forward in training mode keys its dropout mask by its own counter ctl[3] and advances it.  A caller that drives the
// forward / backward itself and updates the weights with its own optimiser (the autograd bridge + torch.optim) never runs the
// plan's Adam, so the optimiser step ctl[1] that keys the fused steps' masks would stay put and every forward would reuse one mask.
extern "C" int ogl_plan_forward(ogl_plan* p, ogl_features* f, float* logits_dev, void* stream) {
  OGL_ARG(p, "ogl_plan_forward: null");
  cudaStream_t s = (cudaStream_t)stream;
  OGL_TRY(plan_forward(p, f, logits_dev, p->ctl + 3, s));
  if (p->train_mode && p->cfg.feat_drop > 0.f) OGL_TRY(bump(p->ctl + 3, nullptr, s));
  return OGL_OK;
}

// Static loss scaling of mode OGL_FP16.  The activation gradients (dlogits and everything the backward pass derives from it) are
// STORED times gs = 2^k, k chosen from the caller's loss scale (1 / global batch) so that the largest |dlogits| element is in
// [32, 64): values down to 1e-6 of it stay in fp16's normal range, and there are ten binades of headroom to 65504.  Every fp32
// result that leaves the backward pass -- the weight gradients (the TN GEMMs' reduce) and the bias gradients (column sums) -- is
// multiplied by 1 / gs where it is written; a power of two, so the unscaling is exact and Adam, the peer exchange and the
// gradient readers see true gradients.
extern "C" float ogl_fp16_grad_scale(float loss_scale) {
  const float a = fabsf(loss_scale);
  if (!(a > 0.f) || !std::isfinite(a)) return 1.f;
  int e = 0;
  frexpf(64.f / a, &e);                 // 64 / a = m * 2^e, m in [0.5, 1)
  return ldexpf(1.f, e - 1);            // 2^floor(log2(64 / a)):  a * gs in (32, 64]
}
static float grad_scale_for(const ogl_plan* p, float loss_scale) { return p->mode == OGL_FP16 ? ogl_fp16_grad_scale(loss_scale) : 1.f; }

static int plan_loss(ogl_plan* p, ogl_features* f, float scale, int want_grad, float* per_vertex_loss_dev, float* loss_sum_dev, cudaStream_t s) {
  const int L = p->L;
  LayerBuf& last = p->layer[L - 1];
  p->grad_scale = want_grad ? grad_scale_for(p, scale) : 1.f;
  scale *= p->grad_scale;
  float* per = per_vertex_loss_dev ? per_vertex_loss_dev : p->per_loss;
  STAGE("xent", xent(p->mode, (const float*)p->act[0], last.pout, p->cfg.dims[L], f->labels, p->nodes[0], p->counts, p->nmax[0],
                     round_up(p->nmax[0], 128), scale, per, last.dpre, last.pout, want_grad, s));
  if (loss_sum_dev) STAGE("loss_sum", sum_f32(per, p->counts, p->nmax[0], loss_sum_dev, s));
  return OGL_OK;
}

static int plan_backward_layers(ogl_plan* p, cudaStream_t s);
static int join_side(ogl_plan* p, cudaStream_t s);
static int adam_range(ogl_plan* p, int64_t lo, int64_t hi, cudaStream_t s) {
  return adam_shadow(p->mode, p->params, p->grads, p->adam_m, p->adam_v, lo, hi, p->cfg.lr, p->cfg.beta1, p->cfg.beta2, p->cfg.eps, p->ctl + 1,
                     p->shadow_segs, p->n_shadow_segs, s);
}

extern "C" int ogl_plan_loss_backward(ogl_plan* p, ogl_features* f, float loss_scale, float* per_vertex_loss_dev, float* loss_sum_dev,
                                      void* stream) {
  OGL_ARG(p && f && p->params && p->n_seeds > 0, "ogl_plan_loss_backward: plan not ready");
  cudaStream_t s = (cudaStream_t)stream;
  OGL_TRY(plan_loss(p, f, loss_scale, 1, per_vertex_loss_dev, loss_sum_dev, s));
  return plan_backward_layers(p, s);
}

static int plan_backward_layers(ogl_plan* p, cudaStream_t s) {
  const int L = p->L;
  auto dw_pool = [&](int l) {                     // dWp = dhp^T act[src] of layer l
    LayerBuf& lb = p->layer[l];
    const int sl = L - l;
    GemmTN tp;
    tp.a = lb.dhp; tp.lda = lb.pin; tp.n = lb.in; tp.b = p->act[sl]; tp.ldb = lb.pin; tp.k = lb.in;
    tp.c = p->grads + lb.o_wp; tp.ldc = lb.in; tp.m_max = p->nmax[sl]; tp.m_dev = p->counts + sl; tp.mode = p->mode;
    tp.alpha = 1.f / p->grad_scale;
    tp.partial = p->tn_partial; tp.partial_elems = p->tn_partial_elems;
    return tp;
  };
  if (p->tail_mode == 2) {                        // only dWp of layer 0 (its dhp was left in place by the tail_mode 1 pass)
    STAGE("l0.dW_pool", gemm_tn(dw_pool(0), p->cfg.gemm_impl, s));
    return OGL_OK;
  }
  OGL_TRY(join_side(p, s));                      // reverse edge lists built on the side stream during sampling
  for (int l = L - 1; l >= 0; --l) {
    LayerBuf& lb = p->layer[l];
    const int h = L - 1 - l, sl = h + 1, dl = h;
    float* G = p->grads;
    // dWs = dpre^T act[src][:n_d] ; dWn = dpre^T neigh ; db = colsum(dpre): independent of the chain below -> side stream.
    // They contract over the rows of level dl -- and so does the fc_pool weight gradient of the layer ABOVE (dhp[l+1]^T act[dl]),
    // which was held back for this: the three GEMMs go out as ONE grouped launch.
    const bool ov = p->use_side && !p->prof_on;
    cudaStream_t ss = ov ? p->side : s;
    if (ov) {
      OGL_CUDA(cudaEventRecord(p->ev_fork, s));                 // dpre of this layer (and dhp of the layer above) are complete on s
      OGL_CUDA(cudaStreamWaitEvent(p->side, p->ev_fork, 0));
    }
    GemmTN grp[3];
    int ng = 0;
    if (l + 1 < L) grp[ng++] = dw_pool(l + 1);
    GemmTN t;
    t.a = lb.dpre; t.lda = lb.pout; t.n = lb.out; t.b = p->act[sl]; t.ldb = lb.pin; t.k = lb.in;
    t.c = G + lb.o_ws; t.ldc = lb.in; t.m_max = p->nmax[dl]; t.m_dev = p->counts + dl; t.mode = p->mode;
    t.alpha = 1.f / p->grad_scale;
    grp[ng++] = t;
    t.b = lb.neigh; t.c = G + lb.o_wn;
    grp[ng++] = t;
    for (int i = 0; i < ng; ++i) { grp[i].partial = ov ? p->tn_partial2 : p->tn_partial; grp[i].partial_elems = p->tn_partial_elems; }
    STAGE_ON(ss, nm("l%d.dW_group", l).c_str(), gemm_tn_group(grp, ng, p->cfg.gemm_impl, ss));
    STAGE_ON(ss, nm("l%d.db_out", l).c_str(), colsum(p->mode, lb.dpre, lb.pout, lb.out, p->counts + dl, p->nmax[dl],
                                                     ov ? p->colsum_partial2 : p->colsum_partial, G + lb.o_bs, G + lb.o_bn, ss,
                                                     1.f / p->grad_scale));
    // dneigh = dpre Wn
    GemmNT n1;
    n1.a[0] = lb.dpre; n1.lda[0] = lb.pout; n1.b[0] = lb.wnT; n1.ldb[0] = lb.pout; n1.k[0] = lb.out; n1.n_seg = 1;
    n1.c = lb.dng; n1.ldc = lb.pin; n1.m_max = p->nmax[dl]; n1.m_dev = p->counts + dl; n1.n = lb.in;
    n1.mode = p->mode; n1.zero_tail = 0;
    n1.mask = lb.neigh; n1.ldmask = lb.pin;        // relu'(hp) at the argmax: neigh[d, f] == hp[src(arg), f]
    STAGE(nm("l%d.dneigh_gemm", l).c_str(), gemm_nt(n1, p->cfg.gemm_impl, s));
    // fc_pool bias gradient: every dng[d, f] lands in exactly one source row, so colsum(dhp) == colsum(dng).  Side stream too (behind the
    // weight-gradient group): only Adam reads it
    if (ov) {
      OGL_CUDA(cudaEventRecord(p->ev_fork, s));
      OGL_CUDA(cudaStreamWaitEvent(p->side, p->ev_fork, 0));
    }
    STAGE_ON(ss, nm("l%d.db_pool", l).c_str(), colsum(p->mode, lb.dng, lb.pin, lb.in, p->counts + dl, p->nmax[dl],
                                                      ov ? p->colsum_partial2 : p->colsum_partial, G + lb.o_bp, nullptr, ss,
                                                      1.f / p->grad_scale));
    // max-pool backward as a gather over the reverse edge lists
    STAGE(nm("l%d.pool_bwd", l).c_str(), pool_bwd(p->mode, lb.dng, lb.pin, lb.arg, p->rev_ptr[h], p->rev_edge[h], p->cfg.fanouts[h],
                                                  p->counts + sl, p->nmax[sl], lb.dhp, s));
    // dWp = dhp^T act[src]: layer 0 computes it here (the step's last and largest weight gradient; data-parallel runs peel it off
    // as the second gradient bucket); the layers above hold it back for the next grouped launch
    if (l == 0 && p->tail_mode != 1) STAGE("l0.dW_pool", gemm_tn(dw_pool(0), p->cfg.gemm_impl, s));
    if (l > 0) {
      // dpre[l-1] = relu'(act[src]) * ( dhp Wp + [dpre Ws on the first n_d rows] )
      LayerBuf& prev = p->layer[l - 1];
      GemmNT d;
      d.a[0] = lb.dhp; d.lda[0] = lb.pin; d.b[0] = lb.wpT; d.ldb[0] = lb.pin; d.k[0] = lb.in;
      d.a[1] = lb.dpre; d.lda[1] = lb.pout; d.b[1] = lb.wsT; d.ldb[1] = lb.pout; d.k[1] = lb.out; d.a_rows_dev[1] = p->counts + dl;
      d.a_rows_max[1] = round_up(p->nmax[dl], 128);
      d.n_seg = 2;
      d.mask = p->act[sl]; d.ldmask = lb.pin;      // (after feat_drop a dropped element is 0 as well: relu' and the keep mask in one)
      if (p->train_mode && p->cfg.feat_drop > 0.f) d.alpha = 1.f / (1.f - p->cfg.feat_drop);
      d.c = prev.dpre; d.ldc = prev.pout; d.m_max = p->nmax[sl]; d.m_dev = p->counts + sl; d.n = lb.in;
      d.mode = p->mode;
      STAGE(nm("l%d.dx_gemm", l).c_str(), gemm_nt(d, p->cfg.gemm_impl, s));
    }
  }
  if (p->use_side && !p->prof_on) {                                   // join: the side-stream gradients precede Adam / the caller
    // fused step with Adam: every gradient except layer 0's fc_pool.weight (the first in*in floats) is final on the side stream
    // while the main stream still computes that last, largest one: their Adam update runs there, beside it
    if (p->adam_in_backward && p->n_params > p->layer[0].o_bp) {
      OGL_TRY(adam_range(p, p->layer[0].o_bp, p->n_params, p->side));
      p->adam_done_from = p->layer[0].o_bp;
    }
    OGL_CUDA(cudaEventRecord(p->ev_join, p->side));
    OGL_CUDA(cudaStreamWaitEvent(s, p->ev_join, 0));
  }
  return OGL_OK;
}

extern "C" int ogl_plan_set_input(ogl_plan* p, const float* x_dev, int n_rows, void* stream) {
  OGL_ARG(p && x_dev && n_rows > 0 && n_rows <= p->nmax[p->L], "ogl_plan_set_input: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  const int L = p->L, F = p->cfg.dims[0], pt = pitch_of(F);
  OGL_TRY(feat_write(p->mode, x_dev, nullptr, n_rows, F, p->act[L], pt, 0, s));
  const int np = std::min(round_up(n_rows, 128), round_up(p->nmax[L], 128));
  if (np > n_rows) OGL_CUDA(cudaMemsetAsync((char*)p->act[L] + p->es * (size_t)n_rows * pt, 0, p->es * (size_t)(np - n_rows) * pt, s));
  return OGL_OK;
}

extern "C" int ogl_plan_backward(ogl_plan* p, const float* dlogits_dev, float dlogits_amax, void* stream) {
  OGL_ARG(p && dlogits_dev && p->params && p->n_seeds > 0, "ogl_plan_backward: plan not ready");
  cudaStream_t s = (cudaStream_t)stream;
  LayerBuf& last = p->layer[p->L - 1];
  const int n = p->n_seeds;
  // mode OGL_FP16: the caller's dlogits may have any magnitude (reduction "sum", a scaled loss, a batch of one), so the scale is
  // the fused loss's rule applied to their largest |element|: it is stored in (32, 64], whatever the loss.  0 or a non-finite
  // maximum gives scale 1 (zeros stay zeros, inf / NaN propagate).
  p->grad_scale = grad_scale_for(p, dlogits_amax);
  OGL_TRY(feat_write(p->mode, dlogits_dev, nullptr, n, last.out, last.dpre, last.pout, 0, s, p->grad_scale));
  const int np = round_up(n, 128);
  if (np > n) OGL_CUDA(cudaMemsetAsync((char*)last.dpre + p->es * (size_t)n * last.pout, 0, p->es * (size_t)(np - n) * last.pout, s));
  return plan_backward_layers(p, s);
}

extern "C" int ogl_plan_adam_step(ogl_plan* p, void* stream) {
  OGL_ARG(p && p->params, "ogl_plan_adam_step: parameters not bound");
  cudaStream_t s = (cudaStream_t)stream;
  // (a fused step has already updated [adam_done_from, n_params) on the side stream, see plan_backward_layers)
  const int64_t hi = p->adam_done_from > 0 ? p->adam_done_from : p->n_params;
  p->adam_done_from = 0;
  STAGE("adam", adam_range(p, 0, hi, s));
  OGL_TRY(bump(nullptr, p->ctl + 1, s));
  return OGL_OK;
}

// data-parallel twin of ogl_plan_adam_step: gradients [lo, hi) are summed over the ranks of `peer` through NVLink peer memory inside
// the Adam kernel (peer.cu).  `last` != 0 on the final bucket of a step: the Adam step counter advances after it.
static int peer_adam_range(ogl_plan* p, ogl_peer* peer, int64_t lo, int64_t hi, float* reduced_out_dev, cudaStream_t s) {
  PeerAdamArgs a;
  a.mode = p->mode; a.params = p->params; a.grads = p->grads; a.m = p->adam_m; a.v = p->adam_v;
  a.lr = p->cfg.lr; a.b1 = p->cfg.beta1; a.b2 = p->cfg.beta2; a.eps = p->cfg.eps;
  a.t_dev = p->ctl + 1; a.segs = p->shadow_segs; a.n_segs = p->n_shadow_segs; a.reduced_out = reduced_out_dev;
  return peer_sum_adam(peer, a, lo, hi, s);
}

extern "C" int ogl_plan_peer_adam(ogl_plan* p, ogl_peer* peer, int64_t lo, int64_t hi, int last, float* reduced_out_dev, void* stream) {
  OGL_ARG(p && p->params && peer, "ogl_plan_peer_adam: parameters not bound / null peer group");
  OGL_ARG(lo >= 0 && hi <= p->n_params, "ogl_plan_peer_adam: range outside the %lld parameters", (long long)p->n_params);
  cudaStream_t s = (cudaStream_t)stream;
  PeerAdamArgs a;
  a.mode = p->mode; a.params = p->params; a.grads = p->grads; a.m = p->adam_m; a.v = p->adam_v;
  a.lr = p->cfg.lr; a.b1 = p->cfg.beta1; a.b2 = p->cfg.beta2; a.eps = p->cfg.eps;
  a.t_dev = p->ctl + 1; a.segs = p->shadow_segs; a.n_segs = p->n_shadow_segs; a.reduced_out = reduced_out_dev;
  OGL_TRY(peer_sum_adam(peer, a, lo, hi, s));
  if (last) OGL_TRY(bump(nullptr, p->ctl + 1, s));
  return OGL_OK;
}

static int stage_seeds(ogl_plan* p, const int64_t* seeds, int n_seeds, int on_host, const int64_t** out, cudaStream_t s) {
  OGL_ARG(n_seeds > 0 && n_seeds <= p->cfg.max_seeds, "n_seeds %d not in [1, %d]", n_seeds, p->cfg.max_seeds);
  if (on_host) {
    OGL_CUDA(cudaMemcpyAsync(p->seeds_stage, seeds, sizeof(int64_t) * n_seeds, cudaMemcpyHostToDevice, s));
    *out = p->seeds_stage;
  } else {
    *out = seeds;
  }
  return OGL_OK;
}

// ---- the fixed launch sequences of a train step over the seeds already staged in p->seeds_stage ----------------
// kind 0: everything; kind 1: sample + gather (needs no weights: in data-parallel runs it overlaps the gradient
// all-reduce + Adam of the previous step); kind 2: forward .. backward (.. Adam)
static int join_side(ogl_plan* p, cudaStream_t s) {
  if (p->side_pending) {
    OGL_CUDA(cudaEventRecord(p->ev_join, p->side));
    OGL_CUDA(cudaStreamWaitEvent(s, p->ev_join, 0));
    p->side_pending = 0;
  }
  return OGL_OK;
}

static int step_body(ogl_plan* p, int kind, ogl_graph* g, ogl_features* f, int n_seeds, float loss_scale, int do_step,
                     float* per_vertex_loss_dev, float* loss_sum_dev, cudaStream_t s) {
  if (kind == 0 || kind == 1) {
    p->in_train_step = 1;
    const int rs = ogl_plan_sample(p, g, p->seeds_stage, n_seeds, s);
    p->in_train_step = 0;
    OGL_TRY(rs);
  }
  if (kind == 1) {
    OGL_ARG(f->mode == p->cfg.mode && f->F == p->cfg.dims[0], "ogl_plan_step_begin: feature store does not match the plan (mode/F)");
    STAGE("gather", gather_rows(p->mode, f->table, f->pitch, p->nodes[p->L], p->counts + p->L, p->nmax[p->L], p->act[p->L], s));
    OGL_TRY(bump(p->ctl, nullptr, s));            // the Philox step advances with the sampling, not with the (possibly later) finish
    return join_side(p, s);                       // a captured graph must rejoin its forked stream
  }
  if (kind == 4) {
    p->grad_scale = grad_scale_for(p, loss_scale);
    p->tail_mode = 2;
    const int rb = plan_backward_layers(p, s);
    p->tail_mode = 0;
    return rb;
  }
  if (kind == 5) {
    // the whole data-parallel finish as ONE launch sequence (one CUDA graph per step): the split form (head graph | exchange kernel
    // | tail graph | exchange kernel on a communication stream, with events between them) costs ~80 us of launch / dependency latency
    // per step even on a single rank; here the exchanges are nodes of the same graph as the GEMMs they overlap.
    //   forward -> peers have read my previous gradients -> loss -> backward without the last weight-gradient GEMM
    //   -> [side: exchange + Adam of everything but layer 0's fc_pool.weight]  ||  [main: that GEMM]
    //   -> exchange + Adam of fc_pool.weight -> optimiser step counter
    ogl_peer* peer = p->dp_peer;
    OGL_ARG(peer && p->use_side, "ogl_plan_step_finish_dp: needs a peer group and the side stream");
    p->skip_gather = 1;
    const int keep_mode = p->train_mode;
    p->train_mode = 1;
    int r = plan_forward(p, f, nullptr, p->ctl + 1, s);
    p->skip_gather = 0;
    // the peers must have finished reading my previous gradients before this step's backward pass overwrites them: checked HERE,
    // after the forward pass (a quarter of a millisecond after they started reading), not at the start of the step where it is a
    // third box-wide synchronisation on the critical path
    if (r == OGL_OK) r = peer_wait_readers(peer, s);
    if (r == OGL_OK) {
      p->tail_mode = 1;
      r = ogl_plan_loss_backward(p, f, loss_scale, per_vertex_loss_dev, loss_sum_dev, s);
      p->tail_mode = 0;
    }
    p->train_mode = keep_mode;
    OGL_TRY(r);
    const int64_t n0 = p->layer[0].o_bp;            // = in * in: layer 0's fc_pool.weight leads the flat buffers
    OGL_CUDA(cudaEventRecord(p->ev_fork, s));
    OGL_CUDA(cudaStreamWaitEvent(p->side, p->ev_fork, 0));
    if (p->n_params > n0) OGL_TRY(peer_adam_range(p, peer, n0, p->n_params, nullptr, p->side));
    OGL_CUDA(cudaEventRecord(p->ev_join, p->side));
    p->tail_mode = 2;
    r = plan_backward_layers(p, s);
    p->tail_mode = 0;
    OGL_CUDA(cudaStreamWaitEvent(s, p->ev_join, 0));
    OGL_TRY(r);
    OGL_TRY(peer_adam_range(p, peer, 0, n0, nullptr, s));
    return bump(nullptr, p->ctl + 1, s);
  }
  p->skip_gather = (kind == 2 || kind == 3);
  const int keep_mode = p->train_mode;
  p->train_mode = 1;                             // a train step: feat_drop on (the reference calls model.train() first, pytorch/model.py:120)
  const int rf = plan_forward(p, f, nullptr, p->ctl + 1, s);
  p->skip_gather = 0;
  if (rf != OGL_OK) { p->train_mode = keep_mode; return rf; }
  p->tail_mode = (kind == 3) ? 1 : 0;
  p->adam_in_backward = (do_step && kind != 3) ? 1 : 0;
  const int rl = ogl_plan_loss_backward(p, f, loss_scale, per_vertex_loss_dev, loss_sum_dev, s);
  p->train_mode = keep_mode;
  p->tail_mode = 0;
  p->adam_in_backward = 0;
  OGL_TRY(rl);
  if (do_step) OGL_TRY(ogl_plan_adam_step(p, s));
  if (kind == 0) OGL_TRY(bump(p->ctl, nullptr, s));
  return OGL_OK;
}

// run step_body directly, or capture it once per key and replay the graph
static int run_step(ogl_plan* p, int kind, ogl_graph* g, ogl_features* f, int n_seeds, float loss_scale, int do_step,
                    float* per_vertex_loss_dev, float* loss_sum_dev, cudaStream_t s) {
  if (!p->use_graph || p->prof_on) return step_body(p, kind, g, f, n_seeds, loss_scale, do_step, per_vertex_loss_dev, loss_sum_dev, s);
  const ogl_plan::StepKey key{kind == 5 ? (const void*)p->dp_peer : (const void*)g, f, per_vertex_loss_dev, loss_sum_dev, g ? graph_generation(g) : 0, n_seeds, do_step, loss_scale, kind, p->parity};
  ogl_plan::StepGraph* hit = nullptr;
  for (auto& sg : p->step_graphs)
    if (sg.key == key) { hit = &sg; break; }
  if (!hit) {
    if (!p->cap_stream) OGL_CUDA(cudaStreamCreateWithFlags(&p->cap_stream, cudaStreamNonBlocking));
    OGL_CUDA(cudaStreamBeginCapture(p->cap_stream, cudaStreamCaptureModeThreadLocal));
    const int r = step_body(p, kind, g, f, n_seeds, loss_scale, do_step, per_vertex_loss_dev, loss_sum_dev, p->cap_stream);
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(p->cap_stream, &graph);
    if (r != OGL_OK) { if (graph) cudaGraphDestroy(graph); return r; }
    OGL_CUDA(e);
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ei = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    OGL_CUDA(ei);
    if (p->step_graphs.size() >= 24) {          // evict the least recently used
      size_t lru = 0;
      for (size_t i = 1; i < p->step_graphs.size(); ++i)
        if (p->step_graphs[i].last_use < p->step_graphs[lru].last_use) lru = i;
      cudaGraphExecDestroy(p->step_graphs[lru].exec);
      p->step_graphs.erase(p->step_graphs.begin() + lru);
    }
    p->step_graphs.push_back({key, exec, 0});
    hit = &p->step_graphs.back();
    p->graph_captures++;
  }
  hit->last_use = ++p->graph_clock;
  OGL_CUDA(cudaGraphLaunch(hit->exec, s));
  p->graph_replays++;
  if (kind < 2) p->n_seeds = n_seeds;
  return OGL_OK;
}

static int stage_step_seeds(ogl_plan* p, const int64_t* seeds, int n_seeds, int seeds_on_host, cudaStream_t s) {
  OGL_ARG(n_seeds > 0 && n_seeds <= p->cfg.max_seeds, "n_seeds %d not in [1, %d]", n_seeds, p->cfg.max_seeds);
  // seeds always go through the plan's staging buffer so that a captured graph is independent of the caller's pointer
  OGL_CUDA(cudaMemcpyAsync(p->seeds_stage, seeds, sizeof(int64_t) * n_seeds, seeds_on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s));
  return OGL_OK;
}


// ------------------------------------------------------------------ software pipeline ---------------
// sample + gather of a minibatch need the graph, the feature table and the seeds, but no weights: they run ahead, on the plan's
// `pre` stream and into the other buffer set, while the previous minibatch's forward / backward / Adam occupies the caller's stream
// (the reference gets the same effect from NodeDataLoader worker processes, pytorch/model.py:128-131).
static int ensure_pipeline(ogl_plan* p) {
  if (p->have_alt) return OGL_OK;
  const int L = p->L;
  ogl_plan::SampleBufs& a = p->alt;
  a.nodes.assign(L + 1, nullptr); a.edge_lid.assign(L, nullptr); a.edge_gsrc.assign(L, nullptr);
  a.rev_ptr.assign(L, nullptr); a.rev_edge.assign(L, nullptr);
  DM0(a.counts, sizeof(int32_t) * (L + 1));
  DM0(a.seeds_stage, sizeof(int64_t) * p->cfg.max_seeds);
  for (int lv = 0; lv <= L; ++lv) DM0(a.nodes[lv], sizeof(int32_t) * p->nmax[lv]);
  for (int h = 0; h < L; ++h) {
    const int64_t ne = (int64_t)p->nmax[h] * p->cfg.fanouts[h];
    DM0(a.edge_lid[h], sizeof(int32_t) * ne);
    DM0(a.edge_gsrc[h], sizeof(int32_t) * ne);
    DM0(a.rev_ptr[h], sizeof(int32_t) * ((size_t)p->nmax[h + 1] + 2));
    DM0(a.rev_edge[h], sizeof(int32_t) * ne);
  }
  DM0(a.x, p->es * (size_t)round_up(p->nmax[L], 128) * pitch_of(p->cfg.dims[0]));
  OGL_CUDA(cudaStreamCreateWithFlags(&p->pre, cudaStreamNonBlocking));
  OGL_CUDA(cudaEventCreateWithFlags(&p->ev_tail, cudaEventDisableTiming));
  for (int i = 0; i < 2; ++i) OGL_CUDA(cudaEventCreateWithFlags(&p->ev_ready[i], cudaEventDisableTiming));
  OGL_CUDA(cudaMallocHost(&p->seed_ring, sizeof(int64_t) * ogl_plan::kSeedRing * p->cfg.max_seeds));
  for (int i = 0; i < ogl_plan::kSeedRing; ++i) OGL_CUDA(cudaEventCreateWithFlags(&p->ev_ring[i], cudaEventDisableTiming));
  p->have_alt = 1;
  return OGL_OK;
}

static void swap_bufs(ogl_plan* p) {
  ogl_plan::SampleBufs& a = p->alt;
  std::swap(p->nodes, a.nodes); std::swap(p->edge_lid, a.edge_lid); std::swap(p->edge_gsrc, a.edge_gsrc);
  std::swap(p->rev_ptr, a.rev_ptr); std::swap(p->rev_edge, a.rev_edge);
  std::swap(p->counts, a.counts); std::swap(p->act[p->L], a.x); std::swap(p->seeds_stage, a.seeds_stage);
  p->parity ^= 1;
}

// enqueue sample + gather of one minibatch on the `pre` stream, ordered after everything enqueued on `s` so far (graph inserts,
// feature writes, the producer of device-resident seeds, and the step that last read the target buffer set)
static int prefetch_impl(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_seeds, int seeds_on_host, cudaStream_t s) {
  OGL_ARG(n_seeds > 0 && n_seeds <= p->cfg.max_seeds, "ogl_plan_prefetch: n_seeds %d not in [1, %d]", n_seeds, p->cfg.max_seeds);
  OGL_TRY(ensure_pipeline(p));
  OGL_ARG(!(p->pend[0] && p->pend[1]), "ogl_plan_prefetch: two minibatches are already pending");
  const int slot = (p->pend[0] || p->cur_open) ? 1 : 0;
  OGL_ARG(!(slot && p->pend[1]), "ogl_plan_prefetch: the other buffer set already holds a prefetched minibatch");
  // host seeds are copied into a pinned ring slot at once (the caller's buffer is free when this returns; pageable memory costs no
  // stream synchronisation); device seeds may still be in production on the caller's stream and must stay valid until consumed
  const int64_t* src = seeds;
  if (seeds_on_host) {
    const int k = p->ring_next;
    p->ring_next = (k + 1) % ogl_plan::kSeedRing;
    OGL_CUDA(cudaEventSynchronize(p->ev_ring[k]));           // the H2D copy that last used this slot has run (normally long ago)
    memcpy(p->seed_ring + (size_t)k * p->cfg.max_seeds, seeds, sizeof(int64_t) * n_seeds);
    src = p->seed_ring + (size_t)k * p->cfg.max_seeds;
  }
  OGL_CUDA(cudaEventRecord(p->ev_tail, s));
  OGL_CUDA(cudaStreamWaitEvent(p->pre, p->ev_tail, 0));
  if (slot) swap_bufs(p);
  int r = OGL_OK;
  if (cudaMemcpyAsync(p->seeds_stage, src, sizeof(int64_t) * n_seeds, seeds_on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice,
                      p->pre) != cudaSuccess) {
    set_error("ogl_plan_prefetch: seed copy failed: %s", cudaGetErrorString(cudaGetLastError()));
    r = OGL_ERR_CUDA;
  }
  if (seeds_on_host && r == OGL_OK && cudaEventRecord(p->ev_ring[(p->ring_next + ogl_plan::kSeedRing - 1) % ogl_plan::kSeedRing], p->pre) != cudaSuccess)
    r = OGL_ERR_CUDA;
  const int n_keep = p->n_seeds;
  if (r == OGL_OK) r = run_step(p, 1, g, f, n_seeds, 0.f, 0, nullptr, nullptr, p->pre);
  p->n_seeds = n_keep;                                       // n_seeds describes the minibatch the caller's stream works on
  if (r == OGL_OK && cudaEventRecord(p->ev_ready[p->parity], p->pre) != cudaSuccess) r = OGL_ERR_CUDA;
  // writers of the graph / feature store order themselves after this prefetch from now on (common.cu: readers_wait)
  if (r == OGL_OK) readers_add(g, f, p->ev_ready[p->parity], p);
  // stage profiling wants every stage alone on the device: the caller's stream waits for the prefetch at once (no overlap)
  if (r == OGL_OK && p->prof_on && cudaStreamWaitEvent(s, p->ev_ready[p->parity], 0) != cudaSuccess) r = OGL_ERR_CUDA;
  if (slot) swap_bufs(p);
  OGL_TRY(r);
  p->pend[slot] = 1;
  p->pend_n[slot] = n_seeds;
  return OGL_OK;
}

// the caller's stream takes over the prefetched minibatch held by the current buffer set
static int consume_prefetched(ogl_plan* p, int n_seeds, cudaStream_t s) {
  OGL_ARG(p->pend[0], "internal: no prefetched minibatch");
  OGL_ARG(n_seeds == p->pend_n[0], "train step of %d seeds, but the prefetched minibatch has %d", n_seeds, p->pend_n[0]);
  OGL_CUDA(cudaStreamWaitEvent(s, p->ev_ready[p->parity], 0));
  p->n_seeds = n_seeds;
  return OGL_OK;
}
static void advance_prefetched(ogl_plan* p) {                // after the finish of the current minibatch has been enqueued
  p->pend[0] = 0;
  p->cur_open = 0;
  if (p->pend[1]) {
    swap_bufs(p);
    p->pend[0] = 1; p->pend_n[0] = p->pend_n[1];
    p->pend[1] = 0;
  }
}

extern "C" int ogl_plan_prefetch(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_seeds, int seeds_on_host,
                                 void* stream) {
  OGL_ARG(p && g && f && seeds, "ogl_plan_prefetch: null");
  OGL_ARG(f->mode == p->cfg.mode && f->F == p->cfg.dims[0], "ogl_plan_prefetch: feature store does not match the plan (mode/F)");
  return prefetch_impl(p, g, f, seeds, n_seeds, seeds_on_host, (cudaStream_t)stream);
}

extern "C" int ogl_plan_prefetch_pending(const ogl_plan* p) { return p ? p->pend[0] + p->pend[1] : 0; }

extern "C" int ogl_plan_train_step(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_seeds, int seeds_on_host,
                                   float loss_scale, int do_step, float* per_vertex_loss_dev, float* loss_sum_dev, void* stream) {
  OGL_ARG(p && g && f && seeds, "ogl_plan_train_step: null");
  OGL_ARG(p->params, "ogl_plan_train_step: parameters not bound");
  cudaStream_t s = (cudaStream_t)stream;
  if (p->pend[0]) {
    // the minibatch was sampled + gathered ahead by ogl_plan_prefetch (same seeds, by contract): only forward .. Adam remain
    OGL_TRY(consume_prefetched(p, n_seeds, s));
    const int r = run_step(p, 2, nullptr, f, n_seeds, loss_scale, do_step, per_vertex_loss_dev, loss_sum_dev, s);
    advance_prefetched(p);
    OGL_TRY(r);
  } else {
    OGL_ARG(!p->pend[1], "ogl_plan_train_step: a prefetched minibatch is pending behind an unfinished ogl_plan_step_begin");
    OGL_TRY(stage_step_seeds(p, seeds, n_seeds, seeds_on_host, s));
    OGL_TRY(run_step(p, 0, g, f, n_seeds, loss_scale, do_step, per_vertex_loss_dev, loss_sum_dev, s));
    p->cur_open = 0;
  }
  return record_level_counts(p, s);
}

// `n_batches` consecutive train steps of `batch` seeds each in ONE call (the reference runs batch_timestep minibatches per
// snapshot, pytorch/model.py:129-134): no per-step host round trip; per-vertex losses / loss sums of step i land at
// per_vertex_loss_dev[i * batch ...] / loss_sums_dev[i]
extern "C" int ogl_plan_train_steps(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_batches, int batch,
                                    int seeds_on_host, float loss_scale, int do_step, float* per_vertex_loss_dev, float* loss_sums_dev,
                                    void* stream) {
  OGL_ARG(p && g && f && seeds && n_batches >= 0, "ogl_plan_train_steps: bad arguments");
  OGL_ARG(p->params, "ogl_plan_train_steps: parameters not bound");
  cudaStream_t s = (cudaStream_t)stream;
  OGL_ARG(!p->pend[0], "ogl_plan_train_steps: a prefetched minibatch is pending");
  if (n_batches >= 2 && p->use_pipeline && p->use_graph && !p->prof_on) {
    // software-pipelined: sample + gather of minibatch i+1 (pre stream, other buffer set) overlap forward .. Adam of minibatch i
    OGL_ARG(f->mode == p->cfg.mode && f->F == p->cfg.dims[0], "ogl_plan_train_steps: feature store does not match the plan (mode/F)");
    OGL_TRY(prefetch_impl(p, g, f, seeds, batch, seeds_on_host, s));
    for (int i = 0; i < n_batches; ++i) {
      if (i + 1 < n_batches) OGL_TRY(prefetch_impl(p, g, f, seeds + (int64_t)(i + 1) * batch, batch, seeds_on_host, s));
      OGL_TRY(consume_prefetched(p, batch, s));
      const int r = run_step(p, 2, nullptr, f, batch, loss_scale, do_step, per_vertex_loss_dev ? p->per_loss : nullptr,
                             loss_sums_dev ? p->loss_sum : nullptr, s);
      advance_prefetched(p);
      OGL_TRY(r);
      if (per_vertex_loss_dev)
        OGL_CUDA(cudaMemcpyAsync(per_vertex_loss_dev + (int64_t)i * batch, p->per_loss, sizeof(float) * batch, cudaMemcpyDeviceToDevice, s));
      if (loss_sums_dev) OGL_CUDA(cudaMemcpyAsync(loss_sums_dev + i, p->loss_sum, sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    return OGL_OK;
  }
  for (int i = 0; i < n_batches; ++i) {
    OGL_TRY(stage_step_seeds(p, seeds + (int64_t)i * batch, batch, seeds_on_host, s));
    // fixed internal outputs keep one captured graph valid for every step; results are copied out per step
    OGL_TRY(run_step(p, 0, g, f, batch, loss_scale, do_step, per_vertex_loss_dev ? p->per_loss : nullptr,
                     loss_sums_dev ? p->loss_sum : nullptr, s));
    if (per_vertex_loss_dev)
      OGL_CUDA(cudaMemcpyAsync(per_vertex_loss_dev + (int64_t)i * batch, p->per_loss, sizeof(float) * batch, cudaMemcpyDeviceToDevice, s));
    if (loss_sums_dev) OGL_CUDA(cudaMemcpyAsync(loss_sums_dev + i, p->loss_sum, sizeof(float), cudaMemcpyDeviceToDevice, s));
  }
  return OGL_OK;
}

extern "C" int ogl_plan_step_begin(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_seeds, int seeds_on_host,
                                   void* stream) {
  OGL_ARG(p && g && f && seeds, "ogl_plan_step_begin: null");
  cudaStream_t s = (cudaStream_t)stream;
  OGL_ARG(!p->pend[0] && !p->pend[1], "ogl_plan_step_begin: a prefetched minibatch is pending");
  OGL_TRY(stage_step_seeds(p, seeds, n_seeds, seeds_on_host, s));
  OGL_TRY(run_step(p, 1, g, f, n_seeds, 0.f, 0, nullptr, nullptr, s));
  p->cur_open = 1;
  return OGL_OK;
}

// step_finish in two pieces for bucketed gradient exchange: `head` leaves only the last weight-gradient GEMM (layer 0's
// fc_pool.weight, the first parameter of the flat buffer) undone, `tail` runs it.  Every other gradient is final after
// `head`, so its all-reduce can overlap `tail`.
extern "C" int ogl_plan_step_finish_head(ogl_plan* p, ogl_features* f, float loss_scale, float* per_vertex_loss_dev, float* loss_sum_dev,
                                         void* stream) {
  OGL_ARG(p && f && p->params && (p->n_seeds > 0 || p->pend[0]), "ogl_plan_step_finish_head: no step begun / parameters not bound");
  if (p->pend[0]) OGL_TRY(consume_prefetched(p, p->pend_n[0], (cudaStream_t)stream));   // (released by _tail)
  p->head_loss_scale = loss_scale;               // the tail (step kind 4) unscales its weight gradient by the same loss scale
  return run_step(p, 3, nullptr, f, p->n_seeds, loss_scale, 0, per_vertex_loss_dev, loss_sum_dev, (cudaStream_t)stream);
}

extern "C" int ogl_plan_step_finish_tail(ogl_plan* p, ogl_features* f, void* stream) {
  OGL_ARG(p && f && p->params && p->n_seeds > 0, "ogl_plan_step_finish_tail: no step begun / parameters not bound");
  cudaStream_t s = (cudaStream_t)stream;
  const int r4 = run_step(p, 4, nullptr, f, p->n_seeds, p->head_loss_scale, 0, nullptr, nullptr, s);
  advance_prefetched(p);
  OGL_TRY(r4);
  return record_level_counts(p, s);
}

// data-parallel finish: forward .. backward with the gradient exchange over NVLink peer memory and Adam inside the same launch
// sequence (step kind 5).  The plan's gradient buffer must be the peer group's (ogl_peer_buffer).
extern "C" int ogl_plan_step_finish_dp(ogl_plan* p, ogl_peer* peer, ogl_features* f, float loss_scale, float* per_vertex_loss_dev,
                                       float* loss_sum_dev, void* stream) {
  OGL_ARG(p && peer && f && p->params && (p->n_seeds > 0 || p->pend[0]), "ogl_plan_step_finish_dp: no step begun / parameters not bound");
  cudaStream_t s = (cudaStream_t)stream;
  if (p->pend[0]) OGL_TRY(consume_prefetched(p, p->pend_n[0], s));
  p->dp_peer = peer;
  const int r5 = run_step(p, 5, nullptr, f, p->n_seeds, loss_scale, 1, per_vertex_loss_dev, loss_sum_dev, s);
  p->dp_peer = nullptr;
  advance_prefetched(p);
  OGL_TRY(r5);
  return record_level_counts(p, s);
}

extern "C" int ogl_plan_step_finish(ogl_plan* p, ogl_features* f, float loss_scale, int do_step, float* per_vertex_loss_dev,
                                    float* loss_sum_dev, void* stream) {
  OGL_ARG(p && f && p->params && (p->n_seeds > 0 || p->pend[0]), "ogl_plan_step_finish: no step begun / parameters not bound");
  cudaStream_t s = (cudaStream_t)stream;
  const int was_pending = p->pend[0];
  if (was_pending) OGL_TRY(consume_prefetched(p, p->pend_n[0], s));
  const int r2 = run_step(p, 2, nullptr, f, p->n_seeds, loss_scale, do_step, per_vertex_loss_dev, loss_sum_dev, s);
  advance_prefetched(p);
  OGL_TRY(r2);
  return record_level_counts(p, s);
}

extern "C" int ogl_plan_set_option(ogl_plan* p, const char* name, int value) {
  OGL_ARG(p && name, "ogl_plan_set_option: null");
  if (strcmp(name, "cuda_graph") == 0) { p->use_graph = value ? 1 : 0; return OGL_OK; }
  if (strcmp(name, "side_stream") == 0) { p->use_side = value ? 1 : 0; return OGL_OK; }
  if (strcmp(name, "pipeline") == 0) { p->use_pipeline = value ? 1 : 0; return OGL_OK; }
  if (strcmp(name, "train_mode") == 0) { p->train_mode = value ? 1 : 0; return OGL_OK; }
  set_error("ogl_plan_set_option: unknown option '%s'", name);
  return OGL_ERR_ARG;
}

// bit 0: a seed id outside [0, n_vertices) was handed to a sampling call since the last read (it was replaced by vertex 0);
// bit 1: a full-inference loss met a label outside [0, classes) (its loss is NaN); synchronises the device, clears the flags
extern "C" int ogl_plan_error_flags(ogl_plan* p, uint32_t* out) {
  OGL_ARG(p && out, "ogl_plan_error_flags: null");
  OGL_CUDA(cudaDeviceSynchronize());
  OGL_CUDA(cudaMemcpy(out, p->ctl + 2, sizeof(uint32_t), cudaMemcpyDeviceToHost));
  OGL_CUDA(cudaMemset(p->ctl + 2, 0, sizeof(uint32_t)));
  return OGL_OK;
}

extern "C" int ogl_plan_graph_stats(ogl_plan* p, int64_t out[2]) {
  OGL_ARG(p && out, "ogl_plan_graph_stats: null");
  out[0] = p->graph_captures;
  out[1] = p->graph_replays;
  return OGL_OK;
}

extern "C" int ogl_plan_eval_step(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds, int n_seeds, int seeds_on_host,
                                  float* logits_dev, float* per_vertex_loss_dev, void* stream) {
  OGL_ARG(p && g && f && seeds, "ogl_plan_eval_step: null");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t* sd = nullptr;
  OGL_TRY(stage_seeds(p, seeds, n_seeds, seeds_on_host, &sd, s));
  OGL_TRY(ogl_plan_sample(p, g, sd, n_seeds, stream));
  const int keep_mode = p->train_mode;
  p->train_mode = 0;                             // evaluation: no dropout (model.eval(), pytorch/model.py:41)
  const int rfw = ogl_plan_forward(p, f, logits_dev, stream);
  p->train_mode = keep_mode;
  OGL_TRY(rfw);
  if (per_vertex_loss_dev) OGL_TRY(plan_loss(p, f, 1.f, 0, per_vertex_loss_dev, nullptr, s));
  OGL_TRY(bump(p->ctl, nullptr, s));
  return OGL_OK;
}

// ------------------------------------------------------------------ full-neighbourhood inference ----
// DGL's model.inference(g, x): layer by layer over EVERY vertex and EVERY in-edge, no sampling.  Per layer: hp = relu(h Wp^T + bp) over
// all rows (layer 0 reads the feature table itself), the CSR segment max, then [h | neigh] [Ws | Wn]^T + b (ReLU except on the
// last layer).  With seeds, the last layer's segment max and output GEMM run on the seed rows only.  Reads the weights and shadows;
// leaves the Philox / Adam counters, the minibatch buffers, pending prefetches and captured step graphs alone.
static int full_ws_reserve(ogl_plan* p, int64_t rows_needed) {
  ogl_plan::FullWs& w = p->full;
  if (rows_needed <= w.rows) return OGL_OK;
  const int64_t rows = round_up((int)std::max<int64_t>(rows_needed, w.rows + w.rows / 2), 128);
  int max_pin = 0, max_hid = 8;
  for (int l = 0; l < p->L; ++l) {
    max_pin = std::max(max_pin, p->layer[l].pin);
    if (l < p->L - 1) max_hid = std::max(max_hid, p->layer[l].pout);
  }
  for (void* q : {w.hp, w.neigh, w.hs, w.h[0], w.h[1], w.hc, (void*)w.logits, (void*)w.seeds, (void*)w.front}) cudaFree(q);
  w.hp = w.neigh = w.hs = w.h[0] = w.h[1] = w.hc = nullptr;
  w.logits = nullptr;
  w.seeds = w.front = nullptr;
  w.rows = 0;
  const size_t r = (size_t)rows;
  const size_t bytes[9] = {p->es * r * max_pin, p->es * r * max_pin, p->es * r * max_pin, p->es * r * max_hid, p->es * r * max_hid,
                           p->es * r * max_hid, sizeof(float) * r * p->layer[p->L - 1].pout, sizeof(int32_t) * r,
                           sizeof(int32_t) * r * std::max(p->L - 1, 1)};
  void** ptrs[9] = {&w.hp, &w.neigh, &w.hs, &w.h[0], &w.h[1], &w.hc, (void**)&w.logits, (void**)&w.seeds, (void**)&w.front};
  for (int i = 0; i < 9; ++i)
    if (dmalloc0(ptrs[i], bytes[i]) != OGL_OK) {
      cudaGetLastError();
      for (int j = 0; j < 9; ++j) { cudaFree(*ptrs[j]); *ptrs[j] = nullptr; }
      set_error("ogl_plan_infer_full: cannot allocate the activations of %lld rows (full-graph inference keeps every layer's [V, pitch] "
                "tables in device memory; graphs that do not fit are not supported)", (long long)rows);
      return OGL_ERR_CAPACITY;
    }
  w.rows = rows;
  return OGL_OK;
}

// the argument checks both entry points share; *V = the graph's vertex count
static int full_check(const ogl_plan* p, ogl_graph* g, const ogl_features* f, const char* who, int64_t* V) {
  OGL_ARG(p && g && f, "%s: null", who);
  OGL_ARG(p->params, "%s: parameters not bound", who);
  OGL_ARG(f->mode == p->cfg.mode && f->F == p->cfg.dims[0], "%s: feature store does not match the plan (mode/F)", who);
  OGL_ARG(graph_source_bound(g) == 0, "%s: the graph is a destination shard (ogl_graph_set_source_bound); full inference needs every "
          "source row", who);
  *V = graph_view(g).n_vertices;
  OGL_ARG(*V <= f->v_cap, "%s: graph has more vertices than the feature store", who);
  OGL_ARG(*V < (1LL << 31), "%s: too many vertices", who);
  return OGL_OK;
}

// layer l for the destination rows rows32[0..n) (device, ids already in [0, V)) or, with rows32 == nullptr, [row0, row0 + n):
// hp = relu(h Wp^T + bp) over every vertex (layer 0 reads the feature table itself), the segment max over the n rows, then
// [h_r | neigh_r] [Ws | Wn]^T + b into out [n, ldo]: ReLU and the storage type for a hidden layer, fp32 logits for the last.
// The GEMMs compute every row on its own, so any split of the rows gives the same bits.
static int full_layer(ogl_plan* p, const GraphView& gv, int64_t E, const ogl_features* f, int l, const void* h, int ldh,
                      const int32_t* rows32, int64_t row0, int64_t n, void* out, int ldo, cudaStream_t s) {
  ogl_plan::FullWs& w = p->full;
  LayerBuf& lb = p->layer[l];
  const bool last = l == p->L - 1;
  const int m = (int)n;
  if (l == 0) {
    h = f->table;
    ldh = f->pitch;
  }
  STAGE(nm("full.l%d.pool_gemm", l).c_str(), pool_gemm(p, l, h, ldh, w.hp, lb.pin, (int)gv.n_vertices, nullptr, s));
  STAGE(nm("full.l%d.segmax", l).c_str(), csr_segmax(p->mode, gv, E, w.hp, lb.pin, lb.in, rows32, nullptr, row0, m, w.neigh, lb.pin,
                                                     &w.sm, s));
  const int mp = round_up(m, 128);
  if (mp > m) OGL_CUDA(cudaMemsetAsync((char*)w.neigh + p->es * (size_t)m * lb.pin, 0, p->es * (size_t)(mp - m) * lb.pin, s));
  // the self term: the listed rows gathered, or the range read in place (the TMA base of the GEMM must be 16-byte aligned)
  const void* self = (const char*)h + p->es * (size_t)row0 * ldh;
  if (rows32) {
    OGL_TRY(gather_rows(p->mode, h, ldh, rows32, nullptr, m, w.hs, s));
    self = w.hs;
  }
  OGL_ARG(((uintptr_t)self & 15) == 0, "full inference: the self rows of layer %d start off the 16-byte grid", l);
  // (the logits go through the plan's padded buffer: the GEMM writes rows of a multiple of 8 columns)
  STAGE(nm("full.l%d.out_gemm", l).c_str(), out_gemm(p, l, self, ldh, w.neigh, lb.pin, last ? (void*)w.logits : out, last ? lb.pout : ldo, m,
                                                    nullptr, s));
  if (last && out != (void*)w.logits)
    OGL_CUDA(cudaMemcpy2DAsync(out, sizeof(float) * ldo, w.logits, sizeof(float) * lb.pout, sizeof(float) * lb.out, n,
                               cudaMemcpyDeviceToDevice, s));
  return OGL_OK;
}

// A hidden layer runs on the frontier of the rows above it when those rows cost sum(deg + 1) <= kFrontierTheta * (E + V): the
// segment max then reads their in-edges only.  Above that share the frontier kernels and the row scatter cost more than the edges
// they save, and the layer (with every layer below it) runs over all rows.  DESIGN.md 3d has the measured crossover.
constexpr double kFrontierTheta = 0.9;

// the layer loop of ogl_plan_infer_full[_loss] (arguments checked, n > 0, V > 0): logits [n, ldo] of the seeds (w.seeds after the
// cast) or of every vertex; logits == w.logits (ldo = the last layer's pitch) leaves them in the plan's buffer.  With seeds, the
// hidden layers run from the top down on S_{L-1} = the seeds, S_l = S_{l+1} u N_in(S_{l+1}) while S_l is cheap enough (above); each
// such S_l is read back to the host (one small copy and a stream synchronisation per expanded layer) to size the layer's launches.
// A frontier layer scatters its rows into the [V, pitch] table; rows outside S_l keep stale contents, which no needed row reads:
// layer l + 1 reads h at S_{l+1} and N_in(S_{l+1}), both inside S_l, and its pool GEMM computes every row on its own.
static int full_forward(ogl_plan* p, ogl_graph* g, const ogl_features* f, const int64_t* seeds_dev, int64_t n, int64_t V, float* logits,
                        int ldo, cudaStream_t s) {
  OGL_TRY(full_ws_reserve(p, std::max(V, n)));
  ogl_plan::FullWs& w = p->full;
  const int L = p->L;
  const GraphView gv = graph_view(g);
  const int64_t E = graph_num_edges(g);
  // out-of-range seed ids are replaced by vertex 0 and raise error bit 0, as in ogl_plan_eval_step
  if (seeds_dev) OGL_TRY(cast_nodes(seeds_dev, w.seeds, n, V, p->ctl + 2, s));
  int lo = L - 1;                        // hidden layers [lo, L - 1) run on their frontier rows w.front + l * w.rows
  std::vector<int64_t> rows_of(L, 0);
  if (seeds_dev && L > 1) {
    if (!w.fr_host) OGL_CUDA(cudaMallocHost(&w.fr_host, sizeof(FrontierOut)));
    const double budget = kFrontierTheta * (double)(E + V);
    for (int l = L - 2; l >= 0; --l) {
      const int32_t* above = l == L - 2 ? w.seeds : w.front + (size_t)(l + 1) * w.rows;
      const int64_t n_above = l == L - 2 ? n : rows_of[l + 1];
      STAGE(nm("full.l%d.frontier", l).c_str(), in_frontier(gv, E, above, nullptr, n_above, w.front + (size_t)l * w.rows, &w.fr, s));
      OGL_CUDA(cudaMemcpyAsync(w.fr_host, w.fr.out, sizeof(FrontierOut), cudaMemcpyDeviceToHost, s));
      OGL_CUDA(cudaStreamSynchronize(s));
      if ((double)w.fr_host->cost > budget) break;
      rows_of[l] = w.fr_host->n;
      lo = l;
    }
  }
  const void* h = nullptr;
  for (int l = 0; l < L; ++l) {
    const bool last = l == L - 1, on_seeds = last && seeds_dev;
    const LayerBuf& lb = p->layer[l];
    void* out = last ? (void*)logits : w.h[l & 1];
    if (!last && l >= lo) {
      const int32_t* rows = w.front + (size_t)l * w.rows;
      OGL_TRY(full_layer(p, gv, E, f, l, h, lb.pin, rows, 0, rows_of[l], w.hc, lb.pout, s));
      STAGE(nm("full.l%d.scatter", l).c_str(), scatter_rows(p->mode, w.hc, lb.pout, rows, (int)rows_of[l], out, s));
    } else {
      OGL_TRY(full_layer(p, gv, E, f, l, h, lb.pin, on_seeds ? w.seeds : nullptr, 0, on_seeds ? n : V, out, last ? ldo : lb.pout, s));
    }
    h = out;
  }
  return OGL_OK;
}

extern "C" int ogl_plan_infer_full(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds_dev, int64_t n, float* logits_dev,
                                   void* stream) {
  int64_t V = 0;
  OGL_TRY(full_check(p, g, f, "ogl_plan_infer_full", &V));
  if (!seeds_dev) n = V;
  OGL_ARG(n >= 0 && n < (1LL << 31), "ogl_plan_infer_full: n out of range");
  if (n == 0) return OGL_OK;
  OGL_ARG(logits_dev, "ogl_plan_infer_full: null logits");
  OGL_ARG(V > 0, "ogl_plan_infer_full: the graph has no vertices");
  return full_forward(p, g, f, seeds_dev, n, V, logits_dev, p->cfg.dims[p->L], (cudaStream_t)stream);
}

extern "C" int ogl_plan_infer_full_loss(ogl_plan* p, ogl_graph* g, ogl_features* f, const int64_t* seeds_dev, int64_t n, float* logits_dev,
                                        float* per_vertex_loss_dev, void* stream) {
  int64_t V = 0;
  OGL_TRY(full_check(p, g, f, "ogl_plan_infer_full_loss", &V));
  if (!seeds_dev) n = V;
  OGL_ARG(n >= 0 && n < (1LL << 31), "ogl_plan_infer_full_loss: n out of range");
  if (n == 0) return OGL_OK;
  OGL_ARG(per_vertex_loss_dev, "ogl_plan_infer_full_loss: null loss");
  OGL_ARG(V > 0, "ogl_plan_infer_full_loss: the graph has no vertices");
  cudaStream_t s = (cudaStream_t)stream;
  const int C = p->cfg.dims[p->L];
  // without a logits buffer of the caller's the loss reads the plan's padded one
  float* logits = logits_dev;
  int ld = C;
  if (!logits_dev) {
    OGL_TRY(full_ws_reserve(p, std::max(V, n)));
    logits = p->full.logits;
    ld = p->layer[p->L - 1].pout;
  }
  OGL_TRY(full_forward(p, g, f, seeds_dev, n, V, logits, ld, s));
  // (the seed ids were cast and range-checked into w.seeds by full_forward)
  return full_xent(logits, ld, C, f->labels, seeds_dev ? p->full.seeds : nullptr, nullptr, 0, n, V, per_vertex_loss_dev, p->ctl + 2, s);
}

extern "C" int ogl_plan_full_xent(ogl_plan* p, ogl_features* f, const float* logits_dev, int ld, const int64_t* rows_dev, int64_t row0,
                                  int64_t n, float* per_vertex_loss_dev, void* stream) {
  OGL_ARG(p && f, "ogl_plan_full_xent: null");
  OGL_ARG(n >= 0, "ogl_plan_full_xent: n < 0");
  if (n == 0) return OGL_OK;
  const int C = p->cfg.dims[p->L];
  OGL_ARG(logits_dev && per_vertex_loss_dev && ld >= C && ((uintptr_t)logits_dev & 3) == 0 && ((uintptr_t)per_vertex_loss_dev & 3) == 0,
          "ogl_plan_full_xent: logits must be fp32 [n, ld] with ld >= %d classes, loss fp32 [n]", C);
  OGL_ARG(rows_dev || (row0 >= 0 && row0 + n <= f->v_cap), "ogl_plan_full_xent: rows [%lld, %lld) are not rows of the feature store (%lld)",
          (long long)row0, (long long)(row0 + n), (long long)f->v_cap);
  return full_xent(logits_dev, ld, C, f->labels, nullptr, rows_dev, row0, n, f->v_cap, per_vertex_loss_dev, p->ctl + 2, (cudaStream_t)stream);
}

extern "C" int ogl_plan_infer_full_layer(ogl_plan* p, ogl_graph* g, ogl_features* f, int layer, const void* h_dev, int ldh,
                                         const int64_t* rows_dev, int64_t row0, int64_t n, void* out_dev, int ldo, void* stream) {
  int64_t V = 0;
  OGL_TRY(full_check(p, g, f, "ogl_plan_infer_full_layer", &V));
  OGL_ARG(layer >= 0 && layer < p->L, "ogl_plan_infer_full_layer: layer %d out of range [0, %d)", layer, p->L);
  OGL_ARG(n >= 0 && n < (1LL << 31), "ogl_plan_infer_full_layer: n out of range");
  OGL_ARG(rows_dev || (row0 >= 0 && row0 + n <= V), "ogl_plan_infer_full_layer: rows [%lld, %lld) are not vertices of the graph (%lld)",
          (long long)row0, (long long)(row0 + n), (long long)V);
  if (n == 0) return OGL_OK;
  OGL_ARG(V > 0, "ogl_plan_infer_full_layer: the graph has no vertices");
  const LayerBuf& lb = p->layer[layer];
  const bool last = layer == p->L - 1;
  OGL_ARG(layer == 0 || (h_dev && ldh == lb.pin && ((uintptr_t)h_dev & 15) == 0),
          "ogl_plan_infer_full_layer: h must be a 16-byte aligned [n_vertices, %d] table of layer %d's input", lb.pin, layer);
  if (last)
    OGL_ARG(out_dev && ldo >= lb.out && ((uintptr_t)out_dev & 3) == 0, "ogl_plan_infer_full_layer: the logits need ldo >= %d", lb.out);
  else
    OGL_ARG(out_dev && ldo == lb.pout && ((uintptr_t)out_dev & 15) == 0,
            "ogl_plan_infer_full_layer: out must be a 16-byte aligned [n, %d] table of layer %d's output", lb.pout, layer);
  cudaStream_t s = (cudaStream_t)stream;
  OGL_TRY(full_ws_reserve(p, std::max(V, n)));
  if (rows_dev) OGL_TRY(cast_nodes(rows_dev, p->full.seeds, n, V, p->ctl + 2, s));
  return full_layer(p, graph_view(g), graph_num_edges(g), f, layer, h_dev, ldh, rows_dev ? p->full.seeds : nullptr, rows_dev ? 0 : row0, n,
                    out_dev, ldo, s);
}

// ------------------------------------------------------------------ incremental inference ----------
// The pieces StreamingInference (inference.py) keeps its own per-vertex tables current with, for a row list or a row range at a time:
// the pool GEMM of listed rows scattered into the caller's hp table, and a layer's segment max (whole rows, or the suffix of edges
// appended since the last refresh, or rows already in the caller's neigh table) + output GEMM scattered into its hidden or logits
// table.  p->full's tables only serve as compact scratch within one call, so full-inference calls between refreshes do no harm.
// The GEMMs compute every row on its own and the segment max is exact: a row computed here has the bits of full_forward's.

// a row list: its ids cast into w.seeds (out-of-range ids become vertex 0 and raise error bit 0); a range: nullptr
static int stream_list(ogl_plan* p, const int64_t* rows_dev, int64_t n, int64_t V, const int32_t** rows32, cudaStream_t s) {
  *rows32 = nullptr;
  if (!rows_dev) return OGL_OK;
  OGL_TRY(cast_nodes(rows_dev, p->full.seeds, n, V, p->ctl + 2, s));
  *rows32 = p->full.seeds;
  return OGL_OK;
}

// compact rows [n, pitch] into the caller's table [*, pitch]: by vertex id, or [row0, row0 + n) in one copy
static int put_rows(int mode, size_t es, const void* rows, int pitch, const int32_t* rows32, int64_t row0, int64_t n, void* table,
                    cudaStream_t s) {
  if (rows32) return scatter_rows(mode, rows, pitch, rows32, (int)n, table, s);
  OGL_CUDA(cudaMemcpyAsync((char*)table + es * (size_t)row0 * pitch, rows, es * (size_t)n * pitch, cudaMemcpyDeviceToDevice, s));
  return OGL_OK;
}

// the listed rows of a table gathered into compact scratch (zero rows up to the next multiple of 128), or the range read in place
static int rows_of(const ogl_plan* p, const void* table, int pitch, const int32_t* rows32, int64_t row0, int64_t n, void* scratch,
                   const void** out, cudaStream_t s) {
  if (!rows32) {
    *out = (const char*)table + p->es * (size_t)row0 * pitch;
    return OGL_OK;
  }
  OGL_TRY(gather_rows(p->mode, table, pitch, rows32, nullptr, (int)n, scratch, s));
  const int64_t np = round_up((int)n, 128);
  if (np > n) OGL_CUDA(cudaMemsetAsync((char*)scratch + p->es * (size_t)n * pitch, 0, p->es * (size_t)(np - n) * pitch, s));
  *out = scratch;
  return OGL_OK;
}

static int stream_check(const ogl_plan* p, ogl_graph* g, const ogl_features* f, int layer, const void* h_dev, int ldh, const int64_t* rows_dev,
                        int64_t row0, int64_t n, const char* who, int64_t* V) {
  OGL_TRY(full_check(p, g, f, who, V));
  OGL_ARG(layer >= 0 && layer < p->L, "%s: layer %d out of range [0, %d)", who, layer, p->L);
  OGL_ARG(n >= 0 && n < (1LL << 31), "%s: n out of range", who);
  OGL_ARG(rows_dev || (row0 >= 0 && row0 + n <= *V), "%s: rows [%lld, %lld) are not vertices of the graph (%lld)", who, (long long)row0,
          (long long)(row0 + n), (long long)*V);
  const LayerBuf& lb = p->layer[layer];
  OGL_ARG(layer == 0 || (h_dev && ldh == lb.pin && ((uintptr_t)h_dev & 15) == 0),
          "%s: h must be a 16-byte aligned [n_vertices, %d] table of layer %d's input", who, lb.pin, layer);
  return OGL_OK;
}

extern "C" int ogl_plan_pool_rows(ogl_plan* p, ogl_graph* g, ogl_features* f, int layer, const void* h_dev, int ldh, const int64_t* rows_dev,
                                  int64_t row0, int64_t n, void* hp_dev, int ldhp, void* stream) {
  int64_t V = 0;
  OGL_TRY(stream_check(p, g, f, layer, h_dev, ldh, rows_dev, row0, n, "ogl_plan_pool_rows", &V));
  if (n == 0) return OGL_OK;
  const LayerBuf& lb = p->layer[layer];
  OGL_ARG(hp_dev && ldhp == lb.pin && ((uintptr_t)hp_dev & 15) == 0, "ogl_plan_pool_rows: hp must be a 16-byte aligned [*, %d] table", lb.pin);
  cudaStream_t s = (cudaStream_t)stream;
  OGL_TRY(full_ws_reserve(p, std::max(V, n)));
  ogl_plan::FullWs& w = p->full;
  const int32_t* rows32 = nullptr;
  OGL_TRY(stream_list(p, rows_dev, n, V, &rows32, s));
  if (layer == 0) {
    h_dev = f->table;
    ldh = f->pitch;
  }
  const void* a = nullptr;
  prof_begin(p, nm("stream.l%d.pool_rows", layer).c_str(), s);
  int r = rows_of(p, h_dev, ldh, rows32, row0, n, w.hs, &a, s);
  if (r == OGL_OK) r = pool_gemm(p, layer, a, ldh, w.hp, lb.pin, (int)n, nullptr, s);
  prof_end(p, s);
  OGL_TRY(r);
  STAGE(nm("stream.l%d.scatter", layer).c_str(), put_rows(p->mode, p->es, w.hp, lb.pin, rows32, row0, n, hp_dev, s));
  return OGL_OK;
}

extern "C" int ogl_plan_stream_rows(ogl_plan* p, ogl_graph* g, ogl_features* f, int layer, const void* h_dev, int ldh, const void* hp_dev,
                                    int ldhp, const int64_t* rows_dev, int64_t row0, int64_t n, void* neigh_dev, int ldn, int neigh_mode,
                                    const int64_t* deg_prev_dev, void* out_dev, int ldo, void* stream) {
  int64_t V = 0;
  OGL_TRY(stream_check(p, g, f, layer, h_dev, ldh, rows_dev, row0, n, "ogl_plan_stream_rows", &V));
  if (n == 0) return OGL_OK;
  const LayerBuf& lb = p->layer[layer];
  const bool last = layer == p->L - 1;
  OGL_ARG(neigh_mode >= 0 && neigh_mode <= 2, "ogl_plan_stream_rows: neigh_mode %d is not 0 (segment max), 1 (suffix) or 2 (table)", neigh_mode);
  OGL_ARG(neigh_mode == 2 || (hp_dev && ldhp == lb.pin && ((uintptr_t)hp_dev & 15) == 0),
          "ogl_plan_stream_rows: hp must be a 16-byte aligned [n_vertices, %d] table", lb.pin);
  OGL_ARG((neigh_mode == 0 && !neigh_dev) || (neigh_dev && ldn == lb.pin && ((uintptr_t)neigh_dev & 15) == 0),
          "ogl_plan_stream_rows: neigh must be a 16-byte aligned [*, %d] table%s", lb.pin, neigh_mode ? "" : " (or NULL)");
  OGL_ARG(neigh_mode != 1 || deg_prev_dev, "ogl_plan_stream_rows: the suffix max needs deg_prev");
  OGL_ARG(out_dev && ldo == lb.pout && ((uintptr_t)out_dev & 15) == 0,
          "ogl_plan_stream_rows: out must be a 16-byte aligned [*, %d] table (%s)", lb.pout, last ? "fp32 logits" : "the storage type");
  cudaStream_t s = (cudaStream_t)stream;
  OGL_TRY(full_ws_reserve(p, std::max(V, n)));
  ogl_plan::FullWs& w = p->full;
  const GraphView gv = graph_view(g);
  const int64_t E = graph_num_edges(g);
  const int32_t* rows32 = nullptr;
  OGL_TRY(stream_list(p, rows_dev, n, V, &rows32, s));
  if (layer == 0) {
    h_dev = f->table;
    ldh = f->pitch;
  }
  const void* neigh = w.neigh;
  if (neigh_mode == 0) {
    STAGE(nm("stream.l%d.segmax", layer).c_str(), csr_segmax(p->mode, gv, E, hp_dev, ldhp, lb.in, rows32, nullptr, row0, n, w.neigh, lb.pin,
                                                             &w.sm, s));
    const int64_t np = round_up((int)n, 128);
    if (np > n) OGL_CUDA(cudaMemsetAsync((char*)w.neigh + p->es * (size_t)n * lb.pin, 0, p->es * (size_t)(np - n) * lb.pin, s));
    if (neigh_dev)
      STAGE(nm("stream.l%d.scatter", layer).c_str(), put_rows(p->mode, p->es, w.neigh, lb.pin, rows32, row0, n, neigh_dev, s));
  } else {
    if (neigh_mode == 1)
      STAGE(nm("stream.l%d.segmax_suffix", layer).c_str(), csr_segmax_suffix(p->mode, gv, E, hp_dev, ldhp, lb.in, rows32, nullptr, row0, n,
                                                                             deg_prev_dev, neigh_dev, ldn, &w.sm, s));
    OGL_TRY(rows_of(p, neigh_dev, ldn, rows32, row0, n, w.neigh, &neigh, s));
  }
  const void* self = nullptr;
  OGL_TRY(rows_of(p, h_dev, ldh, rows32, row0, n, w.hs, &self, s));
  void* res = last ? (void*)w.logits : w.hc;
  STAGE(nm("stream.l%d.out_gemm", layer).c_str(), out_gemm(p, layer, self, ldh, neigh, lb.pin, res, lb.pout, (int)n, nullptr, s));
  STAGE(nm("stream.l%d.scatter", layer).c_str(), put_rows(last ? OGL_F32 : p->mode, last ? sizeof(float) : p->es, res, lb.pout, rows32, row0, n,
                                                          out_dev, s));
  return OGL_OK;
}

extern "C" int ogl_plan_out_frontier(ogl_plan* p, ogl_graph* g, int layer, const int64_t* rows_dev, int64_t n, int64_t* out_rows_dev,
                                     int64_t* out_n, int64_t* out_edge_cost, void* stream) {
  OGL_ARG(p && g && out_n && out_edge_cost && n >= 0 && (rows_dev || n == 0), "ogl_plan_out_frontier: bad arguments");
  OGL_ARG(graph_source_bound(g) == 0, "ogl_plan_out_frontier: the graph is a destination shard (ogl_graph_set_source_bound)");
  const GraphView gv = graph_view(g);
  OGL_ARG(out_rows_dev || gv.n_vertices == 0, "ogl_plan_out_frontier: null out_rows");
  cudaStream_t s = (cudaStream_t)stream;
  ogl_plan::FullWs& w = p->full;
  if (!w.fr_host) OGL_CUDA(cudaMallocHost(&w.fr_host, sizeof(FrontierOut)));
  STAGE(nm("stream.l%d.frontier", layer).c_str(), out_frontier(gv, graph_num_edges(g), rows_dev, n, nullptr, out_rows_dev, &w.fr, s));
  OGL_CUDA(cudaMemcpyAsync(w.fr_host, w.fr.out, sizeof(FrontierOut), cudaMemcpyDeviceToHost, s));
  OGL_CUDA(cudaStreamSynchronize(s));
  *out_n = w.fr_host->n;
  *out_edge_cost = (int64_t)w.fr_host->cost;
  return OGL_OK;
}

// ------------------------------------------------------------------ stage profiling -----------------
extern "C" int ogl_plan_profile(ogl_plan* p, int enable) {
  OGL_ARG(p, "ogl_plan_profile: null");
  if (enable && !p->prof_counts_host) OGL_CUDA(cudaMallocHost(&p->prof_counts_host, sizeof(int32_t) * 8 * kProfSteps));
  p->prof_on = enable ? 1 : 0;
  p->prof_used = 0;          // (re)start: event pairs are reused
  p->prof_steps = 0;
  return OGL_OK;
}

extern "C" int ogl_plan_profile_read(ogl_plan* p, char* names_buf, int names_len, float* ms_out, int64_t* launches_out, int max_stages,
                                     int* n_stages, int64_t* level_count_sums /*[8]*/, int* n_steps) {
  OGL_ARG(p && names_buf && ms_out && launches_out && n_stages, "ogl_plan_profile_read: null");
  OGL_CUDA(cudaDeviceSynchronize());
  const int ns = (int)p->prof_names.size();
  OGL_ARG(ns <= max_stages, "ogl_plan_profile_read: %d stages, room for %d", ns, max_stages);
  std::string joined;
  for (int i = 0; i < ns; ++i) { ms_out[i] = 0.f; launches_out[i] = 0; joined += p->prof_names[i]; joined += '\n'; }
  OGL_ARG((int)joined.size() < names_len, "ogl_plan_profile_read: name buffer too small");
  memcpy(names_buf, joined.c_str(), joined.size() + 1);
  for (size_t i = 0; i < p->prof_used; ++i) {
    float ms = 0.f;
    OGL_CUDA(cudaEventElapsedTime(&ms, p->prof_recs[i].e0, p->prof_recs[i].e1));
    ms_out[p->prof_recs[i].stage] += ms;
    launches_out[p->prof_recs[i].stage] += p->prof_recs[i].launches;
  }
  *n_stages = ns;
  if (level_count_sums) {
    for (int l = 0; l < 8; ++l) level_count_sums[l] = 0;
    for (int st = 0; st < p->prof_steps; ++st)
      for (int l = 0; l <= p->L; ++l) level_count_sums[l] += p->prof_counts_host[8 * st + l];
  }
  if (n_steps) *n_steps = p->prof_steps;
  return OGL_OK;
}

// ------------------------------------------------------------------ introspection ------------------
extern "C" int ogl_plan_level_nodes(ogl_plan* p, int level, const int32_t** nodes_dev, const int32_t** count_dev, int* max_count) {
  OGL_ARG(p && level >= 0 && level <= p->L, "ogl_plan_level_nodes: bad level");
  if (nodes_dev) *nodes_dev = p->nodes[level];
  if (count_dev) *count_dev = p->counts + level;
  if (max_count) *max_count = p->nmax[level];
  return OGL_OK;
}

extern "C" int ogl_plan_block_edges(ogl_plan* p, int hop, const int32_t** edge_src_local_dev, const int32_t** edge_src_global_dev,
                                    const int64_t** edge_eid_dev, int* fanout) {
  OGL_ARG(p && hop >= 0 && hop < p->L, "ogl_plan_block_edges: bad hop");
  if (edge_src_local_dev) *edge_src_local_dev = p->edge_lid[hop];
  if (edge_src_global_dev) *edge_src_global_dev = p->edge_gsrc[hop];
  if (edge_eid_dev) *edge_eid_dev = p->edge_eid[hop];
  if (fanout) *fanout = p->cfg.fanouts[hop];
  return OGL_OK;
}

extern "C" int ogl_plan_tensor(ogl_plan* p, const char* name, const void** ptr_dev, int* rows_max, int* pitch, int* elem_bytes) {
  OGL_ARG(p && name && ptr_dev, "ogl_plan_tensor: null");
  const std::string n(name);
  const int L = p->L;
  auto ret = [&](const void* ptr, int r, int pt, int eb) {
    *ptr_dev = ptr;
    if (rows_max) *rows_max = r;
    if (pitch) *pitch = pt;
    if (elem_bytes) *elem_bytes = eb;
    return OGL_OK;
  };
  if (n == "x") return ret(p->act[L], p->nmax[L], pitch_of(p->cfg.dims[0]), (int)p->es);
  if (n == "full_h0" || n == "full_h1") {       // full inference's hidden tables (as raw [rows, widest hidden pitch] blocks)
    OGL_ARG(p->full.h[0], "ogl_plan_tensor: '%s' is allocated by the first full-inference call", name);
    int max_hid = 8;
    for (int l = 0; l + 1 < L; ++l) max_hid = std::max(max_hid, p->layer[l].pout);
    return ret(p->full.h[n.back() - '0'], (int)p->full.rows, max_hid, (int)p->es);
  }
  if (n.size() >= 2) {
    const int l = n.back() - '0';
    const std::string base = n.substr(0, n.size() - 1);
    if (l >= 0 && l < L) {
      LayerBuf& lb = p->layer[l];
      const int h = L - 1 - l;
      if (base == "hp") return ret(lb.hp, p->nmax[h + 1], lb.pin, (int)p->es);
      if (base == "neigh") return ret(lb.neigh, p->nmax[h], lb.pin, (int)p->es);
      if (base == "arg") return ret(lb.arg, p->nmax[h], lb.pin, 1);
      if (base == "out") return ret(p->act[h], p->nmax[h], lb.pout, l == L - 1 ? 4 : (int)p->es);
      if (base == "dpre") return ret(lb.dpre, p->nmax[h], lb.pout, (int)p->es);
      if (base == "dng") return ret(lb.dng, p->nmax[h], lb.pin, (int)p->es);
      if (base == "dhp") return ret(lb.dhp, p->nmax[h + 1], lb.pin, (int)p->es);
    }
    // reverse edge lists of hop h (the current buffer set): offsets [nmax[h+1] + 1], entries (dst << 8) | slot [nmax[h] * fanout]
    if (l >= 0 && l < L && base == "rev_ptr") return ret(p->rev_ptr[l], p->nmax[l + 1] + 1, 1, 4);
    if (l >= 0 && l < L && base == "rev_edge") return ret(p->rev_edge[l], p->nmax[l] * p->cfg.fanouts[l], 1, 4);
  }
  set_error("ogl_plan_tensor: unknown tensor '%s'", name);
  return OGL_ERR_ARG;
}
