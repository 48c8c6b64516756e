// Device-side view of the streaming CSR shared by graph.cu / sample.cu / plan.cu.
#pragma once
#include "common.cuh"

namespace ogl {

struct GraphCtl {
  unsigned long long pool_top;      // persistent: next free adjacency slot
  unsigned long long relocations;   // persistent: rows moved to the pool top so far
  unsigned int bar_count, bar_gen;  // persistent: grid barrier of the fused streaming insert (count returns to 0, generation grows)
  // ---- per-batch (zeroed before every chunk) ----
  int n_touched;
  int bad_id;
  int n_large;                      // rows whose tail is ordered by a whole CTA
  int n_med;                        // rows whose tail is ordered by one warp in shared memory
  int n_small;                      // rows whose tail (2..32 edges) is ordered by one warp in registers
  int overflow;                     // fused insert: the batch needs more pool than is left; nothing was changed
  unsigned long long need;          // slots this batch takes from the pool top
  unsigned long long scratch_top;   // bump pointer into the tail-ordering scratch
};

struct GraphView {
  const int64_t* row_start;
  const int32_t* deg;
  const unsigned long long* adj;   // (edge id << 32) | source vertex
  int64_t n_vertices;
};

}  // namespace ogl

struct ogl_graph;
namespace ogl {
GraphView graph_view(const ogl_graph* g);
// changes whenever a device pointer of the view changes (pool rebuild): invalidates captured CUDA graphs
uint64_t graph_generation(const ogl_graph* g);
// directed edges stored (the sum of the row degrees)
int64_t graph_num_edges(const ogl_graph* g);
// 0, or the source id bound of a destination shard (ogl_graph_set_source_bound)
int64_t graph_source_bound(const ogl_graph* g);
}
