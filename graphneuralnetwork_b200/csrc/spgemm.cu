// Value-carrying sparse x sparse products on a known output pattern: the numeric phase on top of
// gnn_pattern_product_* that GTN's learned soft metapath composition needs (GTN/models/GTLayer.py: H = a·b and
// H = norm(H)·a, there a dense torch.bmm of [C, N, N] tensors), with its backward.  Values carry C <= 8 channels
// stored entry-major ([nnz, C]); every channel is an independent product over the same pattern.
//
// All three products are masked products O[r, j] = Σ_key L[r, key]·R[j, key] over the pattern of O, where L's rows
// and R's rows are sorted key lists (a CSR row, or a transposed CSR row whose values are reached through its
// permutation):
//   forward  C  = A·B     O = pattern(C), L = A,  R = Bᵀ    (key x)
//   dA = dC·Bᵀ on A:      O = pattern(A), L = C,  R = B     (key j)
//   dB = Aᵀ·dC on B:      O = pattern(B), L = Aᵀ, R = Cᵀ    (key i)
// One thread owns one output entry and intersects its two sorted lists: it walks the shorter one and binary-searches
// the longer one from where the last search ended.  The sum runs in ascending key order whichever list it walks, so
// every entry is one ordered sum: no atomics, no shared accumulators, the same bits on every run and on every path.
//
// Output rows are routed like metapath.cu's: rows with at most spgemm.warp_slots entries and an L row of at most
// spgemm.warp_list keys are walked by one warp each (lanes own entries); the rest -- hub rows -- by one CTA each, so a
// hub row never holds up a launch of short rows.  A thread's entry is computed the same way on both paths.
#include "common.cuh"
#include <cub/cub.cuh>

using namespace gnn;

namespace {

constexpr int MAX_C = 8;
constexpr int WARP_CTA = 256;  // threads per CTA of the warp path (8 warps, one row each)
constexpr int HUB_CTA = 512;   // threads per CTA of the hub-row path

// One operand side: rows of sorted keys; the value of slot t is val[perm ? perm[t] : t] (skipped when outside
// [0, n_val)).
struct Side {
  const int64_t* rowptr;
  const int32_t* col;
  const float* val;
  const int64_t* perm;  // nullable
  int64_t n_rows;
  int64_t n_val;
};

struct Masked {
  const int64_t* o_rowptr;
  const int32_t* o_col;
  float* o_val;
  int64_t n_rows;  // rows of O = rows of L
  Side L;          // row r of O reads row r of L
  Side R;          // entry (r, j) of O reads row j of R; j outside [0, R.n_rows) gives 0
};

__device__ __forceinline__ int64_t value_slot(const Side& s, int64_t t) {
  const int64_t v = s.perm ? s.perm[t] : t;
  return (v >= 0 && v < s.n_val) ? v : -1;
}

template <int C>
__device__ __forceinline__ void fma_entry(const Side& a, int64_t ta, const Side& b, int64_t tb, float (&acc)[C]) {
  const int64_t va = value_slot(a, ta), vb = value_slot(b, tb);
  if (va < 0 || vb < 0) return;
#pragma unroll
  for (int c = 0; c < C; ++c) acc[c] = fmaf(a.val[va * C + c], b.val[vb * C + c], acc[c]);
}

// acc = Σ over keys common to rows (ls, le) of L and (rs, re) of R, in ascending key order.
template <int C>
__device__ __forceinline__ void intersect(const Masked& m, int64_t ls, int64_t le, int64_t rs, int64_t re,
                                          float (&acc)[C]) {
  const bool walk_l = (le - ls) <= (re - rs);
  const int32_t* s_col = walk_l ? m.L.col : m.R.col;  // walked
  const int32_t* g_col = walk_l ? m.R.col : m.L.col;  // searched
  int64_t t = walk_l ? ls : rs;
  const int64_t te = walk_l ? le : re;
  int64_t g = walk_l ? rs : ls;
  const int64_t ge = walk_l ? re : le;
  for (; t < te && g < ge; ++t) {
    const int32_t key = s_col[t];
    int64_t lo = g, hi = ge;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (g_col[mid] < key) lo = mid + 1;
      else hi = mid;
    }
    g = lo;
    if (lo < ge && g_col[lo] == key) {
      fma_entry<C>(m.L, walk_l ? t : lo, m.R, walk_l ? lo : t, acc);
      ++g;
    }
  }
}

template <int C>
__device__ __forceinline__ void entry(const Masked& m, int64_t r, int64_t s) {
  float acc[C];
#pragma unroll
  for (int c = 0; c < C; ++c) acc[c] = 0.f;
  const int32_t j = m.o_col[s];
  if (j >= 0 && (int64_t)j < m.R.n_rows)
    intersect<C>(m, m.L.rowptr[r], m.L.rowptr[r + 1], m.R.rowptr[j], m.R.rowptr[j + 1], acc);
#pragma unroll
  for (int c = 0; c < C; ++c) m.o_val[s * C + c] = acc[c];
}

// rows list[0, n_sel[0]): one warp per row, lanes own its entries
template <int C>
__global__ void __launch_bounds__(WARP_CTA, 4) warp_rows_kernel(Masked m, const int32_t* list, const int64_t* n_sel) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t n_list = n_sel[0];
  for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_list; w += nw) {
    const int64_t r = list[w];
    const int64_t e = m.o_rowptr[r + 1];
    for (int64_t s = m.o_rowptr[r] + lane; s < e; s += 32) entry<C>(m, r, s);
  }
}

// rows list[n_sel[0], n_rows): one CTA per hub row, threads own its entries
template <int C>
__global__ void __launch_bounds__(HUB_CTA, 2) hub_rows_kernel(Masked m, const int32_t* list, const int64_t* n_sel) {
  const int64_t first = n_sel[0];
  for (int64_t w = first + blockIdx.x; w < m.n_rows; w += gridDim.x) {
    const int64_t r = list[w];
    const int64_t e = m.o_rowptr[r + 1];
    for (int64_t s = m.o_rowptr[r] + threadIdx.x; s < e; s += HUB_CTA) entry<C>(m, r, s);
  }
}

struct WarpRow {
  const int64_t* o_rowptr;
  const int64_t* l_rowptr;
  int64_t max_slots, max_list;
  __device__ __forceinline__ bool operator()(int32_t r) const {
    return o_rowptr[r + 1] - o_rowptr[r] <= max_slots && l_rowptr[r + 1] - l_rowptr[r] <= max_list;
  }
};

__global__ void path_rows_kernel(const int64_t* n_sel, int64_t n_rows, int64_t* path_rows) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    path_rows[0] = n_sel[0];
    path_rows[1] = n_rows - n_sel[0];
  }
}

size_t partition_temp_bytes(int64_t n_rows) {
  size_t temp = 0;
  cub::DevicePartition::If(nullptr, temp, cub::CountingInputIterator<int32_t>(0), (int32_t*)nullptr,
                           (int64_t*)nullptr, (int)(n_rows > 0 ? n_rows : 1), WarpRow{nullptr, nullptr, 0, 0});
  return temp;
}

size_t workspace_bytes_for(int64_t n_rows) {
  const size_t n = (size_t)(n_rows > 0 ? n_rows : 1);
  return round_up(n * 4, 256) + 256 + round_up(partition_temp_bytes(n_rows), 256) + 256;
}

inline int grid_cap(int64_t want, int cap) { return (int)(want < 1 ? 1 : (want > cap ? cap : want)); }

template <int C>
int launch_masked(const Masked& m, char* workspace, int64_t* path_rows, cudaStream_t st) {
  if (m.n_rows == 0) {
    if (path_rows) GNN_CUDA(cudaMemsetAsync(path_rows, 0, 2 * sizeof(int64_t), st));
    return GNN_OK;
  }
  int32_t* list = reinterpret_cast<int32_t*>(workspace);
  size_t off = round_up((size_t)m.n_rows * 4, 256);
  int64_t* n_sel = reinterpret_cast<int64_t*>(workspace + off);
  off += 256;
  void* temp = workspace + off;
  size_t temp_bytes = partition_temp_bytes(m.n_rows);
  const WarpRow sel{m.o_rowptr, m.L.rowptr, (int64_t)tuning("spgemm.warp_slots", 1024),
                    (int64_t)tuning("spgemm.warp_list", 1024)};
  // selected rows first (ascending), the hub rows after them
  GNN_CUDA(cub::DevicePartition::If(temp, temp_bytes, cub::CountingInputIterator<int32_t>(0), list, n_sel,
                                    (int)m.n_rows, sel, st));
  count_launch(1);
  hub_rows_kernel<C><<<grid_cap(m.n_rows, num_sms() * 4), HUB_CTA, 0, st>>>(m, list, n_sel);
  GNN_LAUNCH_CHECK();
  warp_rows_kernel<C><<<grid_cap((m.n_rows + 7) / 8, num_sms() * 8), WARP_CTA, 0, st>>>(m, list, n_sel);
  GNN_LAUNCH_CHECK();
  if (path_rows) {
    path_rows_kernel<<<1, 32, 0, st>>>(n_sel, m.n_rows, path_rows);
    GNN_LAUNCH_CHECK();
  }
  return GNN_OK;
}

int launch(const Masked& m, int C, void* workspace, int64_t* path_rows, cudaStream_t st) {
  char* ws = reinterpret_cast<char*>(workspace);
  switch (C) {
    case 1: return launch_masked<1>(m, ws, path_rows, st);
    case 2: return launch_masked<2>(m, ws, path_rows, st);
    case 3: return launch_masked<3>(m, ws, path_rows, st);
    case 4: return launch_masked<4>(m, ws, path_rows, st);
    case 5: return launch_masked<5>(m, ws, path_rows, st);
    case 6: return launch_masked<6>(m, ws, path_rows, st);
    case 7: return launch_masked<7>(m, ws, path_rows, st);
    case 8: return launch_masked<8>(m, ws, path_rows, st);
    default: return GNN_ERR_UNSUPPORTED;
  }
}

constexpr int64_t ID_LIMIT = 0x7fffffffLL;  // ids are int32

int check_common(int64_t n_a, int64_t k, int64_t n_b, int64_t nnz_a, int64_t nnz_b, int32_t C) {
  GNN_REQUIRE(n_a >= 0 && k >= 0 && n_b >= 0 && nnz_a >= 0 && nnz_b >= 0, GNN_ERR_BAD_ARG, "negative size");
  GNN_REQUIRE(n_a < ID_LIMIT && k < ID_LIMIT && n_b < ID_LIMIT, GNN_ERR_BAD_ARG,
              "a dimension does not fit the int32 ids (%lld x %lld x %lld)", (long long)n_a, (long long)k,
              (long long)n_b);
  GNN_REQUIRE(C >= 1, GNN_ERR_BAD_ARG, "C = %d channels", (int)C);
  GNN_REQUIRE(C <= MAX_C, GNN_ERR_UNSUPPORTED, "C = %d channels, at most %d per call", (int)C, MAX_C);
  return GNN_OK;
}

}  // namespace

extern "C" {

size_t gnn_spgemm_workspace_size(int64_t n_a, int64_t k) { return workspace_bytes_for(n_a > k ? n_a : k); }

int gnn_spgemm_values_f32(const int64_t* a_rowptr, const int32_t* a_col, const float* a_val, int64_t n_a, int64_t k,
                          int64_t nnz_a, const int64_t* bt_rowptr, const int32_t* bt_col, const int64_t* bt_perm,
                          const float* b_val, int64_t n_b, int64_t nnz_b, const int64_t* c_rowptr,
                          const int32_t* c_col, float* c_val, int32_t C, int64_t* path_rows, void* workspace,
                          size_t workspace_bytes, gnn_stream_t stream) {
  const int bad = check_common(n_a, k, n_b, nnz_a, nnz_b, C);
  if (bad != GNN_OK) return bad;
  GNN_REQUIRE(a_rowptr && a_col && bt_rowptr && bt_col && bt_perm && c_rowptr && c_col, GNN_ERR_BAD_ARG,
              "null pointer");
  GNN_REQUIRE((a_val || nnz_a == 0) && (b_val || nnz_b == 0) && c_val, GNN_ERR_BAD_ARG, "null value pointer");
  GNN_REQUIRE(workspace && workspace_bytes >= workspace_bytes_for(n_a), GNN_ERR_WORKSPACE,
              "workspace too small (%zu bytes)", workspace_bytes);
  const Masked m{c_rowptr, c_col, c_val, n_a, Side{a_rowptr, a_col, a_val, nullptr, n_a, nnz_a},
                 Side{bt_rowptr, bt_col, b_val, bt_perm, n_b, nnz_b}};
  return launch(m, C, workspace, path_rows, (cudaStream_t)stream);
}

int gnn_spgemm_values_bwd_f32(const int64_t* a_rowptr, const int32_t* a_col, const float* a_val, int64_t n_a,
                              int64_t k, int64_t nnz_a, const int64_t* at_rowptr, const int32_t* at_col,
                              const int64_t* at_perm, const int64_t* b_rowptr, const int32_t* b_col,
                              const float* b_val, int64_t n_b, int64_t nnz_b, const int64_t* c_rowptr,
                              const int32_t* c_col, const int64_t* ct_rowptr, const int32_t* ct_col,
                              const int64_t* ct_perm, const float* dc_val, int64_t nnz_c, int32_t C, float* da_val,
                              float* db_val, int64_t* path_rows, void* workspace, size_t workspace_bytes,
                              gnn_stream_t stream) {
  const int bad = check_common(n_a, k, n_b, nnz_a, nnz_b, C);
  if (bad != GNN_OK) return bad;
  GNN_REQUIRE(nnz_c >= 0, GNN_ERR_BAD_ARG, "negative size");
  GNN_REQUIRE(dc_val || nnz_c == 0, GNN_ERR_BAD_ARG, "null dC");
  GNN_REQUIRE(!da_val || (a_rowptr && a_col && c_rowptr && c_col && b_rowptr && b_col && (b_val || nnz_b == 0)),
              GNN_ERR_BAD_ARG, "null pointer (dA needs A's and B's CSR, B's values and C's CSR)");
  GNN_REQUIRE(!db_val || (b_rowptr && b_col && at_rowptr && at_col && at_perm && ct_rowptr && ct_col && ct_perm &&
                          (a_val || nnz_a == 0)),
              GNN_ERR_BAD_ARG, "null pointer (dB needs B's CSR, Aᵀ and Cᵀ with their permutations, A's values)");
  GNN_REQUIRE(workspace && workspace_bytes >= workspace_bytes_for(n_a > k ? n_a : k), GNN_ERR_WORKSPACE,
              "workspace too small (%zu bytes)", workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  if (da_val) {
    const Masked m{a_rowptr, a_col, da_val, n_a, Side{c_rowptr, c_col, dc_val, nullptr, n_a, nnz_c},
                   Side{b_rowptr, b_col, b_val, nullptr, k, nnz_b}};
    const int s = launch(m, C, workspace, path_rows, st);
    if (s != GNN_OK) return s;
  }
  if (db_val) {
    const Masked m{b_rowptr, b_col, db_val, k, Side{at_rowptr, at_col, a_val, at_perm, k, nnz_a},
                   Side{ct_rowptr, ct_col, dc_val, ct_perm, n_b, nnz_c}};
    const int s = launch(m, C, workspace, path_rows ? path_rows + 2 : nullptr, st);
    if (s != GNN_OK) return s;
  }
  return GNN_OK;
}

}  // extern "C"
