// Pattern-only sparse x sparse product on the device: C = pattern(A·B), the binarised metapath adjacency
// HAN builds from a relation matrix P as (P·Pᵀ > 0) (HAN/utils/data_utils.py:85-89, there a dense float64
// N x N array on the host).  Integer work only: the output is the same bits on every run.
//
// Row i of the product has at most u_i = Σ_{x∈A[i]} deg_B(x) (+1 with self_loops) products.  Both calls first
// bound u_i for their rows and split the rows into three lists, each walked by its own persistent launch, so a
// hub row never holds up a launch of short rows:
//   small  (u_i <= metapath.small_max):  one warp per row sorts its products in shared memory, drops repeats;
//   medium (u_i <= metapath.medium_max): one CTA per row, the same at CTA width;
//   large  (hub rows):                   one CTA per row marks a shared-memory bitmap over a column tile of
//                                        metapath.tile_cols columns; the count is a popcount and the fill an
//                                        ordered scan of the bitmap words, so the output is ascending without
//                                        a sort.  The CTA loops over the tiles of [0, n_b).
// The only atomics are the integer atomicOr of the bitmap: the set they produce does not depend on their order.
#include "common.cuh"
#include <cub/cub.cuh>

using namespace gnn;

namespace {

constexpr int SMALL_CAP = 256;    // products one warp sorts (1 KB of shared memory per warp)
constexpr int SMALL_WARPS = 8;    // warps per CTA of the small path
constexpr int MED_CAP = 8192;     // products one CTA sorts (32 KB of shared memory)
constexpr int MED_THREADS = 512;
constexpr int LARGE_THREADS = 1024;
constexpr int MAX_TILE_BYTES = 219 * 1024;  // bitmap (dynamic shared memory): 227 KB less the block scan's storage
constexpr int32_t NONE = 0x7fffffff;               // sorts last and is never a column id (n_b < 2^31)

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

struct Product {
  const int64_t* a_rowptr;
  const int32_t* a_col;
  int64_t k;  // columns of A = rows of B; other ids of A are skipped
  const int64_t* b_rowptr;
  const int32_t* b_col;
  int64_t n_b;  // columns of B; other ids of B are skipped
  int64_t row_lo;
  int self_loops;
};

__device__ __forceinline__ bool valid_x(const Product& p, int32_t x) { return x >= 0 && (int64_t)x < p.k; }
__device__ __forceinline__ int32_t keep_j(const Product& p, int32_t j) {
  return (j >= 0 && (int64_t)j < p.n_b) ? j : NONE;
}

// one warp per row: u_i, in int64
__global__ void bound_kernel(Product p, int64_t n_rows, int64_t* u) {
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = w; r < n_rows; r += nw) {
    const int64_t s = p.a_rowptr[p.row_lo + r], e = p.a_rowptr[p.row_lo + r + 1];
    int64_t sum = 0;
    for (int64_t t = s + lane; t < e; t += 32) {
      const int32_t x = p.a_col[t];
      if (valid_x(p, x)) sum += p.b_rowptr[x + 1] - p.b_rowptr[x];
    }
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) u[r] = sum + (p.self_loops ? 1 : 0);
  }
}

struct AtMost {
  const int64_t* u;
  int64_t cap;
  __device__ __forceinline__ bool operator()(int32_t r) const { return u[r] <= cap; }
};

// The warp copies the B rows of up to 32 A entries (lane l holds entry l: B row start bs, length d, output offset
// off) into buf, each row with all 32 lanes.
__device__ __forceinline__ void warp_copy_rows(const Product& p, int64_t bs, int d, int off, int32_t* buf) {
  const int lane = threadIdx.x & 31;
  for (int l = 0; l < 32; ++l) {
    const int dl = __shfl_sync(0xffffffffu, d, l);
    const int64_t bl = __shfl_sync(0xffffffffu, bs, l);
    const int ol = __shfl_sync(0xffffffffu, off, l);
    for (int q = lane; q < dl; q += 32) buf[ol + q] = keep_j(p, p.b_col[bl + q]);
  }
}

__device__ __forceinline__ void load_entry(const Product& p, int64_t t, int64_t e, int64_t& bs, int& d) {
  bs = 0;
  d = 0;
  if (t < e) {
    const int32_t x = p.a_col[t];
    if (valid_x(p, x)) {
      bs = p.b_rowptr[x];
      d = (int)(p.b_rowptr[x + 1] - bs);  // <= u_i <= MED_CAP on the sorting paths
    }
  }
}

struct WarpSync {
  __device__ __forceinline__ void operator()() const { __syncwarp(); }
};
struct CtaSync {
  __device__ __forceinline__ void operator()() const { __syncthreads(); }
};

// Bitonic sort of buf[0, n) ascending, padded with NONE to a power of two >= 32, by `nt` threads (thread `t`).
// sync() orders the steps: WarpSync for one warp, CtaSync for a CTA.
template <typename Sync>
__device__ __forceinline__ void bitonic_sort(int32_t* buf, int n, int t, int nt, Sync sync) {
  int P = 32;
  while (P < n) P <<= 1;
  for (int i = n + t; i < P; i += nt) buf[i] = NONE;
  sync();
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = t; i < P; i += nt) {
        const int q = i ^ j;
        if (q > i) {
          const int32_t a = buf[i], b = buf[q];
          if ((a > b) == ((i & k) == 0)) {
            buf[i] = b;
            buf[q] = a;
          }
        }
      }
      sync();
    }
}

template <bool FILL>
__global__ void __launch_bounds__(SMALL_WARPS * 32, 4)
    small_kernel(Product p, const int32_t* list, const int64_t* n_sel, int64_t* counts, const int64_t* rowptr,
                 int32_t* col) {
  __shared__ int32_t smem[SMALL_WARPS][SMALL_CAP];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int32_t* buf = smem[wid];
  const int64_t n_list = n_sel[0];
  for (int64_t w = (int64_t)blockIdx.x * SMALL_WARPS + wid; w < n_list; w += (int64_t)gridDim.x * SMALL_WARPS) {
    const int32_t r = list[w];
    const int64_t row = p.row_lo + r;
    const int64_t s = p.a_rowptr[row], e = p.a_rowptr[row + 1];
    int n = 0;
    if (p.self_loops) {
      if (lane == 0) buf[0] = (int32_t)row;
      n = 1;
    }
    for (int64_t t0 = s; t0 < e; t0 += 32) {
      int64_t bs;
      int d;
      load_entry(p, t0 + lane, e, bs, d);
      int incl = d;
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      warp_copy_rows(p, bs, d, n + incl - d, buf);
      n += __shfl_sync(0xffffffffu, incl, 31);
    }
    __syncwarp();
    bitonic_sort(buf, n, lane, 32, WarpSync{});
    int64_t cnt = 0;
    const int64_t out = FILL ? rowptr[r] : 0;
    for (int t0 = 0; t0 < n; t0 += 32) {
      const int t = t0 + lane;
      const int32_t v = t < n ? buf[t] : NONE;
      const bool keep = v != NONE && (t == 0 || buf[t - 1] != v);
      const unsigned bal = __ballot_sync(0xffffffffu, keep);
      if (FILL && keep) col[out + cnt + __popc(bal & ((1u << lane) - 1u))] = v;
      cnt += __popc(bal);
    }
    if (!FILL && lane == 0) counts[r] = cnt;
    __syncwarp();
  }
}

template <bool FILL>
__global__ void __launch_bounds__(MED_THREADS)
    medium_kernel(Product p, const int32_t* list, const int64_t* n_sel, int64_t* counts, const int64_t* rowptr,
                  int32_t* col) {
  using Scan = cub::BlockScan<int, MED_THREADS>;
  __shared__ int32_t buf[MED_CAP];
  __shared__ typename Scan::TempStorage scan;
  const int tid = threadIdx.x;
  const int64_t n_list = n_sel[1];
  for (int64_t w = blockIdx.x; w < n_list; w += gridDim.x) {
    const int32_t r = list[w];
    const int64_t row = p.row_lo + r;
    const int64_t s = p.a_rowptr[row], e = p.a_rowptr[row + 1];
    int n = 0;
    if (p.self_loops) {
      if (tid == 0) buf[0] = (int32_t)row;
      n = 1;
    }
    for (int64_t t0 = s; t0 < e; t0 += MED_THREADS) {
      int64_t bs;
      int d, off, total;
      load_entry(p, t0 + tid, e, bs, d);
      Scan(scan).ExclusiveSum(d, off, total);
      warp_copy_rows(p, bs, d, n + off, buf);
      n += total;
      __syncthreads();
    }
    bitonic_sort(buf, n, tid, MED_THREADS, CtaSync{});
    int64_t cnt = 0;
    const int64_t out = FILL ? rowptr[r] : 0;
    for (int t0 = 0; t0 < n; t0 += MED_THREADS) {
      const int t = t0 + tid;
      const int32_t v = t < n ? buf[t] : NONE;
      const int keep = (v != NONE && (t == 0 || buf[t - 1] != v)) ? 1 : 0;
      int idx, total;
      Scan(scan).ExclusiveSum(keep, idx, total);
      if (FILL && keep) col[out + cnt + idx] = v;
      cnt += total;
      __syncthreads();
    }
    if (!FILL && tid == 0) counts[r] = cnt;
  }
}

template <bool FILL>
__global__ void __launch_bounds__(LARGE_THREADS)
    large_kernel(Product p, const int32_t* list, const int64_t* n_sel, int64_t n_rows, int64_t tile_cols,
                 int64_t* counts, const int64_t* rowptr, int32_t* col) {
  using Scan = cub::BlockScan<int, LARGE_THREADS>;
  extern __shared__ uint32_t words[];
  __shared__ typename Scan::TempStorage scan;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NWARPS = LARGE_THREADS / 32;
  const int64_t n_list = n_rows - n_sel[0] - n_sel[1];
  for (int64_t w = blockIdx.x; w < n_list; w += gridDim.x) {
    const int32_t r = list[w];
    const int64_t row = p.row_lo + r;
    const int64_t s = p.a_rowptr[row], e = p.a_rowptr[row + 1];
    int64_t cnt = 0;
    const int64_t out = FILL ? rowptr[r] : 0;
    for (int64_t c0 = 0; c0 < p.n_b; c0 += tile_cols) {
      const int64_t c1 = c0 + tile_cols < p.n_b ? c0 + tile_cols : p.n_b;
      const int nwords = (int)((c1 - c0 + 31) >> 5);
      for (int i = tid; i < nwords; i += LARGE_THREADS) words[i] = 0u;
      __syncthreads();
      if (tid == 0 && p.self_loops && row >= c0 && row < c1)
        atomicOr(&words[(row - c0) >> 5], 1u << ((row - c0) & 31));
      for (int64_t t0 = s + (int64_t)warp * 32; t0 < e; t0 += (int64_t)NWARPS * 32) {
        int64_t bs = 0, d = 0;
        if (t0 + lane < e) {
          const int32_t x = p.a_col[t0 + lane];
          if (valid_x(p, x)) {
            bs = p.b_rowptr[x];
            d = p.b_rowptr[x + 1] - bs;
          }
        }
        for (int l = 0; l < 32; ++l) {
          const int64_t dl = __shfl_sync(0xffffffffu, d, l);
          const int64_t bl = __shfl_sync(0xffffffffu, bs, l);
          for (int64_t q = lane; q < dl; q += 32) {
            const int64_t j = p.b_col[bl + q];
            if (j >= c0 && j < c1) atomicOr(&words[(j - c0) >> 5], 1u << ((j - c0) & 31));
          }
        }
      }
      __syncthreads();
      // ordered scan: thread t owns the contiguous words [t*wpt, (t+1)*wpt), so ranks follow column order
      const int wpt = (nwords + LARGE_THREADS - 1) / LARGE_THREADS;
      const int w0 = tid * wpt, w1 = min(w0 + wpt, nwords);
      int mine = 0;
      for (int i = w0; i < w1; ++i) mine += __popc(words[i]);
      int off, total;
      Scan(scan).ExclusiveSum(mine, off, total);
      if (FILL) {
        int64_t o = out + cnt + off;
        for (int i = w0; i < w1; ++i)
          for (uint32_t m = words[i]; m; m &= m - 1u) col[o++] = (int32_t)(c0 + 32 * (int64_t)i + (__ffs(m) - 1));
      }
      cnt += total;
      __syncthreads();
    }
    if (!FILL && tid == 0) counts[r] = cnt;
  }
}

__global__ void path_rows_kernel(const int64_t* n_sel, int64_t n_rows, int64_t* path_rows) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    path_rows[0] = n_sel[0];
    path_rows[1] = n_sel[1];
    path_rows[2] = n_rows - n_sel[0] - n_sel[1];
  }
}

inline int grid_cap(int64_t want, int cap) {
  return (int)(want < 1 ? 1 : (want > cap ? cap : want));
}

// The three row lists of rows [row_lo, row_hi), carved out of the workspace.
struct Routing {
  int32_t* small;
  int32_t* medium;
  int32_t* large;
  int64_t* n_sel;   // [2]: rows of the small and the medium list (the large list holds the rest)
  int64_t* counts;  // [n_rows + 1]
  void* scan_temp;
  size_t scan_bytes;
};

size_t partition_temp_bytes(int64_t n_rows) {
  size_t temp = 0;
  cub::DevicePartition::If(nullptr, temp, cub::CountingInputIterator<int32_t>(0), (int32_t*)nullptr,
                           (int32_t*)nullptr, (int32_t*)nullptr, (int64_t*)nullptr, (int)(n_rows > 0 ? n_rows : 1),
                           AtMost{nullptr, 0}, AtMost{nullptr, 0});
  return temp;
}

size_t scan_temp_bytes(int64_t n_rows) {
  size_t temp = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, temp, (const int64_t*)nullptr, (int64_t*)nullptr, n_rows + 1);
  return temp;
}

int route(const Product& p, int64_t n_rows, void* workspace, Routing& rt, cudaStream_t st) {
  WsCursor ws{(char*)workspace, 0};
  int64_t* u = ws.take<int64_t>(n_rows);
  rt.counts = ws.take<int64_t>(n_rows + 1);
  rt.small = ws.take<int32_t>(n_rows);
  rt.medium = ws.take<int32_t>(n_rows);
  rt.large = ws.take<int32_t>(n_rows);
  rt.n_sel = ws.take<int64_t>(2);
  size_t part = partition_temp_bytes(n_rows);
  rt.scan_bytes = scan_temp_bytes(n_rows);
  void* temp = ws.take<char>(part > rt.scan_bytes ? part : rt.scan_bytes);
  rt.scan_temp = temp;
  // the keys route rows; the caps are what the sorting paths hold
  const int64_t small_max = min(tuning("metapath.small_max", SMALL_CAP), SMALL_CAP);
  const int64_t medium_max = min(tuning("metapath.medium_max", MED_CAP), MED_CAP);
  bound_kernel<<<grid_cap((n_rows * 32 + 255) / 256, num_sms() * 32), 256, 0, st>>>(p, n_rows, u);
  GNN_LAUNCH_CHECK();
  GNN_CUDA(cub::DevicePartition::If(temp, part, cub::CountingInputIterator<int32_t>(0), rt.small, rt.medium, rt.large,
                                    rt.n_sel, (int)n_rows, AtMost{u, small_max}, AtMost{u, medium_max}, st));
  count_launch(2);
  return GNN_OK;
}

int64_t tile_cols_for(int64_t n_b) {
  const int64_t max_cols = (int64_t)(MAX_TILE_BYTES / 4) * 32;
  int64_t t = tuning("metapath.tile_cols", 0);
  t = t <= 0 ? max_cols : (t + 31) / 32 * 32;
  t = t > max_cols ? max_cols : t;
  const int64_t need = (n_b + 31) / 32 * 32;
  return t > need ? (need > 0 ? need : 32) : t;
}

template <bool FILL>
int launch_paths(const Product& p, int64_t n_rows, const Routing& rt, const int64_t* rowptr, int32_t* col,
                 cudaStream_t st) {
  const int64_t tile = tile_cols_for(p.n_b);
  const int smem = (int)(tile / 32 * 4);
  GNN_CUDA(cudaFuncSetAttribute(large_kernel<FILL>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  // the large list first: its hub rows are the longest CTAs of the three launches
  large_kernel<FILL><<<grid_cap(n_rows, num_sms()), LARGE_THREADS, smem, st>>>(p, rt.large, rt.n_sel, n_rows, tile,
                                                                              rt.counts, rowptr, col);
  GNN_LAUNCH_CHECK();
  medium_kernel<FILL><<<grid_cap(n_rows, num_sms() * 4), MED_THREADS, 0, st>>>(p, rt.medium, rt.n_sel, rt.counts,
                                                                              rowptr, col);
  GNN_LAUNCH_CHECK();
  small_kernel<FILL><<<grid_cap((n_rows + SMALL_WARPS - 1) / SMALL_WARPS, num_sms() * 8), SMALL_WARPS * 32, 0, st>>>(
      p, rt.small, rt.n_sel, rt.counts, rowptr, col);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

size_t workspace_bytes_for(int64_t n_rows) {
  const size_t n = (size_t)(n_rows > 0 ? n_rows : 1);
  const size_t part = partition_temp_bytes(n_rows), scan = scan_temp_bytes(n_rows);
  return round_up(n * 8, 256) + round_up((n + 1) * 8, 256) + 3 * round_up(n * 4, 256) + 256 +
         round_up(part > scan ? part : scan, 256) + 1024;
}

// argument checks shared by both calls (before any CUDA call)
int check_args(const int64_t* a_rowptr, const int32_t* a_col, int64_t n_a, int64_t k, const int64_t* b_rowptr,
               const int32_t* b_col, int64_t n_b, int64_t row_lo, int64_t row_hi, int self_loops) {
  GNN_REQUIRE(n_a >= 0 && k >= 0 && n_b >= 0, GNN_ERR_BAD_ARG, "negative size");
  GNN_REQUIRE(row_lo >= 0 && row_lo <= row_hi && row_hi <= n_a, GNN_ERR_BAD_ARG,
              "row range [%lld, %lld) outside the %lld rows of A", (long long)row_lo, (long long)row_hi, (long long)n_a);
  GNN_REQUIRE(n_b < 0x7fffffffLL, GNN_ERR_BAD_ARG, "n_b = %lld does not fit the int32 column ids", (long long)n_b);
  GNN_REQUIRE(!self_loops || n_a == n_b, GNN_ERR_BAD_ARG, "self_loops on a product that is not square (%lld x %lld)",
              (long long)n_a, (long long)n_b);
  GNN_REQUIRE(row_hi - row_lo < 0x7fffffffLL, GNN_ERR_UNSUPPORTED, "more than 2^31-1 rows in one call");
  GNN_REQUIRE(a_rowptr && a_col && b_rowptr && b_col, GNN_ERR_BAD_ARG, "null pointer");
  return GNN_OK;
}

}  // namespace

extern "C" {

size_t gnn_pattern_product_count_workspace_size(int64_t n_rows) { return workspace_bytes_for(n_rows); }

int gnn_pattern_product_count(const int64_t* a_rowptr, const int32_t* a_col, int64_t n_a, int64_t k,
                              const int64_t* b_rowptr, const int32_t* b_col, int64_t n_b, int64_t row_lo,
                              int64_t row_hi, int self_loops, int64_t* rowptr, int64_t* path_rows, void* workspace,
                              size_t workspace_bytes, gnn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int bad = check_args(a_rowptr, a_col, n_a, k, b_rowptr, b_col, n_b, row_lo, row_hi, self_loops);
  if (bad != GNN_OK) return bad;
  GNN_REQUIRE(rowptr != nullptr, GNN_ERR_BAD_ARG, "null rowptr");
  const int64_t n_rows = row_hi - row_lo;
  GNN_REQUIRE(workspace && workspace_bytes >= workspace_bytes_for(n_rows), GNN_ERR_WORKSPACE,
              "workspace too small (%zu bytes)", workspace_bytes);
  if (n_rows == 0) {
    GNN_CUDA(cudaMemsetAsync(rowptr, 0, sizeof(int64_t), st));
    if (path_rows) GNN_CUDA(cudaMemsetAsync(path_rows, 0, 3 * sizeof(int64_t), st));
    return GNN_OK;
  }
  const Product p{a_rowptr, a_col, k, b_rowptr, b_col, n_b, row_lo, self_loops ? 1 : 0};
  Routing rt;
  int s = route(p, n_rows, workspace, rt, st);
  if (s != GNN_OK) return s;
  GNN_CUDA(cudaMemsetAsync(rt.counts + n_rows, 0, sizeof(int64_t), st));
  s = launch_paths<false>(p, n_rows, rt, nullptr, nullptr, st);
  if (s != GNN_OK) return s;
  GNN_CUDA(cub::DeviceScan::ExclusiveSum(rt.scan_temp, rt.scan_bytes, rt.counts, rowptr, n_rows + 1, st));
  count_launch(1);
  if (path_rows) {
    path_rows_kernel<<<1, 32, 0, st>>>(rt.n_sel, n_rows, path_rows);
    GNN_LAUNCH_CHECK();
  }
  return GNN_OK;
}

int gnn_pattern_product_fill(const int64_t* a_rowptr, const int32_t* a_col, int64_t n_a, int64_t k,
                             const int64_t* b_rowptr, const int32_t* b_col, int64_t n_b, int64_t row_lo,
                             int64_t row_hi, int self_loops, const int64_t* rowptr, int32_t* col, void* workspace,
                             size_t workspace_bytes, gnn_stream_t stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int bad = check_args(a_rowptr, a_col, n_a, k, b_rowptr, b_col, n_b, row_lo, row_hi, self_loops);
  if (bad != GNN_OK) return bad;
  GNN_REQUIRE(rowptr && col, GNN_ERR_BAD_ARG, "null pointer");
  const int64_t n_rows = row_hi - row_lo;
  GNN_REQUIRE(workspace && workspace_bytes >= workspace_bytes_for(n_rows), GNN_ERR_WORKSPACE,
              "workspace too small (%zu bytes)", workspace_bytes);
  if (n_rows == 0) return GNN_OK;
  const Product p{a_rowptr, a_col, k, b_rowptr, b_col, n_b, row_lo, self_loops ? 1 : 0};
  Routing rt;
  const int s = route(p, n_rows, workspace, rt, st);
  if (s != GNN_OK) return s;
  return launch_paths<true>(p, n_rows, rt, rowptr, col, st);
}

}  // extern "C"
