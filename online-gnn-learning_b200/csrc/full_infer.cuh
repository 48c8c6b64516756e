// Segment max over the in-edge rows of the streaming CSR and the in-neighbourhood frontier of a row list (full-neighbourhood
// inference, see full_infer.cu).
#pragma once
#include "graph.cuh"

namespace ogl {

// a row with more in-edges than this is a hub: its edges are cut into chunks of this many, one warp per chunk
constexpr int kSegmaxChunk = 2048;

struct SegmaxHub {
  int64_t r;       // output row
  int32_t v;       // vertex
  int32_t base;    // first chunk slot
  int32_t n;       // chunk slots (0: the row was reduced in place by the row pass)
  int32_t pad;
};

// device scratch of csr_segmax, sized from the graph's edge count and the row width in bytes
struct SegmaxWs {
  unsigned long long* ctl = nullptr;   // [0] row cursor, [1] hubs, [2] chunk slots, [3] chunk cursor
  SegmaxHub* hubs = nullptr;
  int32_t* chunk_hub = nullptr;
  void* partial = nullptr;             // [chunk_cap, row bytes]
  int64_t hub_cap = 0, chunk_cap = 0, row_bytes = 0;
};
int segmax_ws_reserve(SegmaxWs* ws, int64_t n_edges, int64_t row_bytes);
void segmax_ws_free(SegmaxWs* ws);

// out[r, :cols] = max over the in-edges (u -> v_r) of x[u, :cols], 0 for a row without in-edges; v_r = rows32[r] | rows64[r] |
// row0 + r (at most one list; row0 is ignored with a list).  A listed id outside [0, n_vertices) gives a zero row.  Columns are
// processed in 16-byte strips, so out columns up to round_up(cols, 16 / element bytes) are written.  Exact: the result does not depend on edge order or on the split.
int csr_segmax(int mode, const GraphView& gv, int64_t n_edges, const void* x, int ld, int cols, const int32_t* rows32,
               const int64_t* rows64, int64_t row0, int64_t n_rows, void* out, int ldo, SegmaxWs* ws, cudaStream_t s);

// device scratch of in_frontier, sized from the vertex and edge capacity
struct FrontierOut {
  unsigned long long cost;             // sum over the result of (in-degree + 1)
  int32_t n;                           // rows in the result
  int32_t pad;
};
struct FrontierWs {
  uint32_t* bits = nullptr;            // [words] membership bitmap
  uint32_t* bits_in = nullptr;         // [words] out_frontier: the input set S (bits is the result)
  int32_t *uniq = nullptr, *counts = nullptr, *offs = nullptr, *scan = nullptr;
  int2* chunks = nullptr;              // (vertex, first edge) of a hub's chunk
  unsigned long long* ctl = nullptr;   // [0] distinct input rows, [1] row cursor, [2] chunk slots, [3] chunk cursor
  FrontierOut* out = nullptr;
  int64_t v_cap = 0, chunk_cap = 0;
};
int frontier_ws_reserve(FrontierWs* ws, int64_t n_vertices, int64_t n_edges);
void frontier_ws_free(FrontierWs* ws);

// the in-neighbourhood frontier S u N_in(S) of S = {v_r}, v_r = rows32[r] | rows64[r] (exactly one list, r < n): out_rows[0..m)
// = its vertices in ascending order (capacity n_vertices), ws->out = {m, sum over them of (in-degree + 1)} on the device.  A listed
// id outside [0, n_vertices) is ignored.  Reads the streaming CSR in place; ordered on s, no host synchronisation.
int in_frontier(const GraphView& gv, int64_t n_edges, const int32_t* rows32, const int64_t* rows64, int64_t n, int32_t* out_rows,
                FrontierWs* ws, cudaStream_t s);

// the out-neighbourhood frontier S u N_out(S) of S = {v_r} (the same lists and result as in_frontier, out_rows32 | out_rows64 exactly
// one): a vertex joins when a source of one of its in-edges is in S.  The CSR stores in-edges only, so this is one pass over every
// row's adjacency, read in place (hub rows cut into kSegmaxChunk chunks), against a bitmap of S; the result is a second bitmap
// seeded with S, so one call expands by one hop.  O(E) work whatever |S|.  Ordered on s, no host synchronisation.
int out_frontier(const GraphView& gv, int64_t n_edges, const int64_t* rows64, int64_t n, int32_t* out_rows32, int64_t* out_rows64,
                 FrontierWs* ws, cudaStream_t s);

// suffix segment max, in place: for v_r = rows32[r] | rows64[r] | row0 + r (r < n; a listed id outside [0, n_vertices) is skipped), acc[v_r, :cols] = max(acc[v_r],
// max over the in-edges of v_r at row positions [deg_prev[v_r], deg[v_r]) of x[src]) -- the edges appended since a refresh at which
// the row had deg_prev[v_r] edges.  deg_prev[v_r] == 0 (or larger than the degree) replaces the row instead (zeros for a row without
// in-edges).  The arithmetic of csr_segmax, so the result is the bits of a whole-row max.  A suffix longer than kSegmaxChunk is cut
// into chunks like a hub row.  acc [*, ldacc] in the storage type, indexed by vertex id; listed ids must be distinct.
int csr_segmax_suffix(int mode, const GraphView& gv, int64_t n_edges, const void* x, int ld, int cols, const int32_t* rows32,
                      const int64_t* rows64, int64_t row0, int64_t n, const int64_t* deg_prev, void* acc, int ldacc, SegmaxWs* ws, cudaStream_t s);

// loss[r] = logsumexp(logits[r, :C]) - logits[r, labels[v_r]] for r < n (fp32 logits [n, ld]), v_r = rows32[r] | rows64[r] | row0 + r
// (at most one list).  The arithmetic of the training loss (warp_logsumexp): equal logits give bit-equal losses.  A v_r outside
// [0, n_vertices) uses vertex 0's label and ORs 1 into *err; a label outside [0, C) gives NaN and ORs 2 into *err.
int full_xent(const float* logits, int ld, int C, const int32_t* labels, const int32_t* rows32, const int64_t* rows64, int64_t row0,
              int64_t n, int64_t n_vertices, float* loss, uint32_t* err, cudaStream_t s);

}  // namespace ogl
