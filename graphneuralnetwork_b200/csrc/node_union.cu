// Deterministic node-set union with remap: the device half of the de-duplicating GraphSAGE collate
// (GraphSAGE/data_utils.py:100-116, `set(nodes) | set(samples)` followed by the id -> position maps).
// The set is ascending global id (the reference iterates a CPython set, i.e. hash order; no per-row arithmetic
// depends on that order, only where rows sit, and the maps carry it).
//
// Method, O(n_a + n_b) and independent of the number of graph nodes:
//   1. key every slot s of [ids_a | ids_b] by its id, a negative id by the largest key (sorts last, excluded);
//   2. one CUB radix sort of (key, slot) pairs;
//   3. head flag per sorted position (a valid key that differs from its predecessor) and an inclusive scan of the
//      flags: the scan value minus one is the rank of the run, i.e. the position of its id in the union;
//   4. scatter: a head writes its id to out_ids[rank], every position writes its rank to its slot's map, positions
//      at or past the count write -1 into out_ids so that the padded set can feed the sampler and the next union.
// Integer work only, no atomics: the same input gives the same bits.
#include "common.cuh"
#include <cub/cub.cuh>

using namespace gnn;

namespace {

inline int grid_for(int64_t n, int block = 256) {
  int64_t g = (n + block - 1) / block;
  const int64_t cap = (int64_t)num_sms() * 32;
  g = g < 1 ? 1 : g;
  return (int)(g > cap ? cap : g);
}

template <typename I, typename K>
__global__ void union_keys_kernel(const I* __restrict__ ids_a, int64_t n_a, const I* __restrict__ ids_b, int64_t n,
                                  K* __restrict__ keys, int32_t* __restrict__ slots) {
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x) {
    const I id = s < n_a ? ids_a[s] : ids_b[s - n_a];
    keys[s] = id < 0 ? ~(K)0 : (K)id;
    slots[s] = (int32_t)s;
  }
}

template <typename K>
__global__ void union_heads_kernel(const K* __restrict__ keys, int64_t n, int32_t* __restrict__ heads) {
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
    const K k = keys[p];
    heads[p] = (k != ~(K)0 && (p == 0 || keys[p - 1] != k)) ? 1 : 0;
  }
}

template <typename I, typename K>
__global__ void union_scatter_kernel(const K* __restrict__ keys, const int32_t* __restrict__ slots,
                                     const int32_t* __restrict__ heads, const int32_t* __restrict__ rank1, int64_t n,
                                     int64_t n_a, I* __restrict__ out_ids, int64_t* __restrict__ out_count,
                                     int64_t* __restrict__ map_a, int64_t* __restrict__ map_b) {
  const int64_t count = rank1[n - 1];
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
    const K k = keys[p];
    const int64_t r = (k == ~(K)0) ? -1 : (int64_t)rank1[p] - 1;
    if (heads[p]) out_ids[r] = (I)k;
    if (p >= count) out_ids[p] = (I)-1;
    const int64_t s = slots[p];
    if (s < n_a) map_a[s] = r;
    else map_b[s - n_a] = r;
    if (p == 0) *out_count = count;
  }
}

struct WsCursor {
  char* base;
  size_t off;
  template <typename T>
  T* take(size_t n) {
    off = round_up(off, 256);
    T* p = reinterpret_cast<T*>(base + off);
    off += n * sizeof(T);
    return p;
  }
};

template <typename K>
size_t union_bytes(int64_t n) {
  const int nn = (int)(n > 0 ? n : 1);
  size_t sort = 0, scan = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort, (const K*)nullptr, (K*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, nn);
  cub::DeviceScan::InclusiveSum(nullptr, scan, (const int32_t*)nullptr, (int32_t*)nullptr, nn);
  const size_t keys = round_up((size_t)nn * sizeof(K), 256), ints = round_up((size_t)nn * sizeof(int32_t), 256);
  return 2 * keys + 4 * ints + round_up(sort > scan ? sort : scan, 256) + 256;
}

template <typename I, typename K>
int union_impl(const I* ids_a, int64_t n_a, const I* ids_b, int64_t n_b, I* out_ids, int64_t* out_count,
               int64_t* map_a, int64_t* map_b, void* workspace, cudaStream_t st) {
  const int64_t n = n_a + n_b;
  WsCursor ws{(char*)workspace, 0};
  K* keys_in = ws.take<K>(n);
  K* keys_out = ws.take<K>(n);
  int32_t* slots_in = ws.take<int32_t>(n);
  int32_t* slots_out = ws.take<int32_t>(n);
  int32_t* heads = ws.take<int32_t>(n);
  int32_t* rank1 = ws.take<int32_t>(n);
  size_t sort = 0, scan = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort, keys_in, keys_out, slots_in, slots_out, (int)n, 0,
                                  (int)sizeof(K) * 8, st);
  cub::DeviceScan::InclusiveSum(nullptr, scan, heads, rank1, (int)n, st);
  void* temp = ws.take<char>(sort > scan ? sort : scan);
  const int grid = grid_for(n);
  union_keys_kernel<I, K><<<grid, 256, 0, st>>>(ids_a, n_a, ids_b, n, keys_in, slots_in);
  GNN_LAUNCH_CHECK();
  GNN_CUDA(cub::DeviceRadixSort::SortPairs(temp, sort, keys_in, keys_out, slots_in, slots_out, (int)n, 0,
                                           (int)sizeof(K) * 8, st));
  count_launch(2);
  union_heads_kernel<K><<<grid, 256, 0, st>>>(keys_out, n, heads);
  GNN_LAUNCH_CHECK();
  GNN_CUDA(cub::DeviceScan::InclusiveSum(temp, scan, heads, rank1, (int)n, st));
  count_launch(1);
  union_scatter_kernel<I, K><<<grid, 256, 0, st>>>(keys_out, slots_out, heads, rank1, n, n_a, out_ids, out_count,
                                                   map_a, map_b);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

}  // namespace

extern "C" {

int gnn_node_union_workspace_size(int64_t n_a, int64_t n_b, size_t* bytes_host) {
  GNN_REQUIRE(bytes_host != nullptr, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(n_a >= 0 && n_b >= 0 && n_a + n_b < 0x7fffffffLL, GNN_ERR_BAD_ARG,
              "bad size (n_a=%lld, n_b=%lld; n_a+n_b must fit int32)", (long long)n_a, (long long)n_b);
  const size_t b32 = union_bytes<uint32_t>(n_a + n_b), b64 = union_bytes<uint64_t>(n_a + n_b);
  *bytes_host = b32 > b64 ? b32 : b64;
  return GNN_OK;
}

int gnn_node_union(const void* ids_a, int64_t n_a, const void* ids_b, int64_t n_b, int id_bits, void* out_ids,
                   int64_t* out_count_dev, int64_t* map_a, int64_t* map_b, void* workspace, size_t workspace_bytes,
                   gnn_stream_t stream) {
  GNN_REQUIRE(n_a >= 0 && n_b >= 0 && n_a + n_b < 0x7fffffffLL, GNN_ERR_BAD_ARG,
              "bad size (n_a=%lld, n_b=%lld; n_a+n_b must fit int32)", (long long)n_a, (long long)n_b);
  GNN_REQUIRE(id_bits == 32 || id_bits == 64, GNN_ERR_BAD_ARG, "id_bits must be 32 or 64");
  GNN_REQUIRE(out_count_dev != nullptr, GNN_ERR_BAD_ARG, "null out_count");
  GNN_REQUIRE((n_a == 0 || (ids_a && map_a)) && (n_b == 0 || (ids_b && map_b)), GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(n_a + n_b == 0 || out_ids, GNN_ERR_BAD_ARG, "null out_ids");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_a + n_b == 0) {
    GNN_CUDA(cudaMemsetAsync(out_count_dev, 0, sizeof(int64_t), st));
    return GNN_OK;
  }
  size_t need = 0;
  gnn_node_union_workspace_size(n_a, n_b, &need);
  GNN_REQUIRE(workspace && workspace_bytes >= need, GNN_ERR_WORKSPACE, "workspace too small (%zu < %zu bytes)",
              workspace_bytes, need);
  if (id_bits == 32)
    return union_impl<int32_t, uint32_t>((const int32_t*)ids_a, n_a, (const int32_t*)ids_b, n_b, (int32_t*)out_ids,
                                         out_count_dev, map_a, map_b, workspace, st);
  return union_impl<int64_t, uint64_t>((const int64_t*)ids_a, n_a, (const int64_t*)ids_b, n_b, (int64_t*)out_ids,
                                       out_count_dev, map_a, map_b, workspace, st);
}

}  // extern "C"
