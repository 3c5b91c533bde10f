// Library-level C ABI: version, error strings, tuning knobs, launch counter.
#include "common.cuh"
#include <string.h>
#include <mutex>
#include <map>
#include <string>

namespace gnn {

static thread_local char t_err[512] = "";
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_err, sizeof(t_err), fmt, ap);
  va_end(ap);
}

int num_sms() {
  // immutable per-device cache (SURVEY.md §8b: "no global mutable state beyond an
  // immutable per-device properties cache")
  static int cache[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cache[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cache[dev] = n;
  }
  return cache[dev];
}

static std::mutex g_tune_mu;
static std::map<std::string, int>& tune_map() {
  static std::map<std::string, int> m = {
      {"sage.smem_kb", 48},      // shared-memory ring per CTA of the TMA gather (4 CTAs/SM)
      {"sage.chunk_bytes", 12288},  // bytes per ring stage
      {"sage.force_ldg", 0},     // 1: never take the TMA path
      {"sage.ctas_per_sm", 4},
      {"sage.packed_add", -1},   // FADD2 in the consumers: -1 = bf16 only, 0 never, 1 always
      {"spmm.long_row", 2048},   // rows above this nnz go to the CTA-per-chunk path (planned call)
      {"spmm.chunk", 8192},      // edges per long-row chunk
      {"spmm.unroll", 0},        // 0 = heuristic
      {"spmm.ctas3", 1},          // 1: multi-vector rows (CHUNKS 2..5) use the 3-CTAs/SM instantiation (0: 2 CTAs/SM)
      {"spmm.rows_per_team", 0},  // >0 overrides the caller's rows_per_team (tuning sweeps)
      {"spmm.team_edges", 512},   // host plan: edges one team should hold (graph.py rows_per_team)
      {"gat.stage_edges", 128},  // logits staged per warp pass
      {"gat.bwd_stage_edges", 64},  // edges staged per warp pass of the backward kernels
      {"gat.coop_min_avg_deg", 256},  // nnz/n at which every row gets a whole CTA
      {"gat.long_row", 1024},        // rows above this get a CTA in the otherwise warp-per-row schedule
      {"metapath.small_max", 256},   // product rows with at most this many products: one warp sorts them (cap 256)
      {"metapath.medium_max", 8192}, // ... at most this many: one CTA sorts them (cap 8192); longer rows: bitmap
      {"metapath.tile_cols", 0},     // columns per bitmap tile of the hub-row path (0 = as many as shared memory holds)
      {"spgemm.warp_slots", 1024},   // masked value products: rows with at most this many output entries ...
      {"spgemm.warp_list", 1024},    // ... and a left row of at most this many keys take a warp; the rest a whole CTA
  };
  return m;
}
int tuning(const char* key, int dflt) {
  std::lock_guard<std::mutex> g(g_tune_mu);
  auto& m = tune_map();
  auto it = m.find(key);
  return it == m.end() ? dflt : it->second;
}

}  // namespace gnn

extern "C" {

int gnn_version(void) { return 100; /* 0.1.0 */ }

const char* gnn_last_error_string(void) { return gnn::t_err; }

const char* gnn_status_string(int s) {
  switch (s) {
    case GNN_OK: return "ok";
    case GNN_ERR_BAD_ARG: return "bad argument";
    case GNN_ERR_MISALIGNED: return "misaligned pointer or leading dimension";
    case GNN_ERR_UNSUPPORTED: return "unsupported shape";
    case GNN_ERR_CUDA: return "CUDA error";
    case GNN_ERR_WORKSPACE: return "workspace too small";
    default: return "unknown status";
  }
}

int64_t gnn_launch_count(void) { return gnn::g_launches.load(); }

int gnn_set_tuning(const char* key, int value) {
  if (!key) return GNN_ERR_BAD_ARG;
  std::lock_guard<std::mutex> g(gnn::g_tune_mu);
  auto& m = gnn::tune_map();
  auto it = m.find(key);
  if (it == m.end()) {
    gnn::set_error("unknown tuning key '%s'", key);
    return GNN_ERR_BAD_ARG;
  }
  it->second = value;
  return GNN_OK;
}

int gnn_get_tuning(const char* key, int* value) {
  if (!key || !value) return GNN_ERR_BAD_ARG;
  std::lock_guard<std::mutex> g(gnn::g_tune_mu);
  auto& m = gnn::tune_map();
  auto it = m.find(key);
  if (it == m.end()) {
    gnn::set_error("unknown tuning key '%s'", key);
    return GNN_ERR_BAD_ARG;
  }
  *value = it->second;
  return GNN_OK;
}

}  // extern "C"
