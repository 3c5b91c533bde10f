// Row-parallel gather-reduce: the one kernel template behind
//   - CSR SpMM  Y = Â·X                     (replaces torch.spmm, GCN/GCN.py:43)
//   - transpose SpMM for the backward       (autograd of GCN/GCN.py:43)
//   - fixed-fanout gather-mean/sum/max with vector loads
//                                           (GraphSAGE_Pytorch/models/Aggregator.py:19-24)
//   - the ordered gather backward into the feature table.
//
// A row is owned by GROUP lanes (a sub-warp chosen from F), each lane owns CHUNKS
// vectors of VEC elements (128-bit when alignment allows).  The GROUP lanes load GROUP
// (col,val) pairs coalesced, then broadcast them by shuffle and issue U independent
// feature-row gathers before the FMAs (memory-level parallelism).  Edges are
// accumulated strictly in CSR order: deterministic, no atomics.
#pragma once
#include "common.cuh"

namespace gnn {

template <typename T>
struct RowArgs {
  const int64_t* rowptr;  // nullptr => implicit fixed fanout: row r owns slots [r*fanout,(r+1)*fanout)
  int32_t fanout;
  const int32_t* col32;  // CSR col / int32 index block
  const int64_t* col64;  // int64 index block; both null => identity (source row = slot)
  const float* val;      // nullptr => 1
  int32_t src_div;       // >0: source row = col / src_div (gather backward: flat position -> source)
  int32_t src_mul;       // >0: typed table [N, src_mul, F]: source row = col * src_mul + (row % src_mul)
                         //     (GATNE's edge-type axis: output row b*T+t reads type-t embeddings)
  float scale;           // result multiplier (1/fanout for mean)
  const T* X;
  int64_t ldx;
  T* Y;
  int64_t ldy;
  int64_t n_rows;
  int32_t F;
  int64_t skip_deg_gt;   // >0: rows with more edges are left to the long-row kernel
  int32_t* argmax;       // max only, nullable, [n_rows, ldy]
  int32_t n_src_rows;    // >0: source ids >= n_src_rows contribute nothing (like negative ids) instead of reading
                         //     out of bounds; the reference raises IndexError there (an id block is caller input)
};

constexpr int kRowReduceThreads = 256;

template <typename T, int VEC, int GROUP, int CHUNKS, int U, int OP>
__global__ void __launch_bounds__(kRowReduceThreads) row_reduce_kernel(const RowArgs<T> a) {
  constexpr int ROWS_PER_CTA = kRowReduceThreads / GROUP;
  const int lane = threadIdx.x & 31;
  const int gl = threadIdx.x % GROUP;
  const unsigned gmask = (GROUP == 32) ? 0xffffffffu : (((1u << GROUP) - 1u) << (lane - gl));
  const int64_t row = (int64_t)blockIdx.x * ROWS_PER_CTA + threadIdx.x / GROUP;
  if (row >= a.n_rows) return;
  int64_t s, e;
  if (a.rowptr) {
    s = __ldg(a.rowptr + row);
    e = __ldg(a.rowptr + row + 1);
  } else {
    s = row * (int64_t)a.fanout;
    e = s + a.fanout;
  }
  if (a.skip_deg_gt > 0 && e - s > a.skip_deg_gt) return;

  float acc[CHUNKS][VEC];
  int best[CHUNKS][VEC];
#pragma unroll
  for (int ch = 0; ch < CHUNKS; ++ch)
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      acc[ch][i] = (OP == 1) ? -INFINITY : 0.f;
      best[ch][i] = 0;
    }

  for (int64_t base = s; base < e; base += GROUP) {
    const int64_t k = base + gl;
    int32_t c = -1;
    float v = 0.f;
    if (k < e) {
      if (a.col32) c = __ldg(a.col32 + k);
      else if (a.col64) {
        // an id outside int32 is invalid (>= every table's rows): -1, not its low 32 bits, which may name a real row
        const int64_t c64 = __ldg(a.col64 + k);
        c = (c64 >= 0 && c64 <= 0x7fffffffLL) ? (int32_t)c64 : -1;
      }
      else c = (int32_t)k;
      if (a.src_div > 0 && c >= 0) c /= a.src_div;
      if (a.src_mul > 0 && c >= 0) c = c * a.src_mul + (int32_t)(row % a.src_mul);
      v = a.val ? __ldg(a.val + k) : 1.f;
    }
    const int cnt = (int)((e - base) < (int64_t)GROUP ? (e - base) : (int64_t)GROUP);
    for (int j0 = 0; j0 < cnt; j0 += U) {
      VecRaw<T, VEC> xv[U][CHUNKS];
      float vv[U];
      bool xok[U][CHUNKS];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int jj = j0 + u;
        const int32_t cj = __shfl_sync(gmask, c, jj, GROUP);
        const float vj = __shfl_sync(gmask, v, jj, GROUP);
        const bool ok = (jj < cnt) && (cj >= 0) && (a.n_src_rows <= 0 || cj < a.n_src_rows);
        vv[u] = ok ? vj : 0.f;
        const T* xr = a.X + (int64_t)(ok ? cj : 0) * a.ldx;
#pragma unroll
        for (int ch = 0; ch < CHUNKS; ++ch) {
          const int col0 = (gl + ch * GROUP) * VEC;
          xok[u][ch] = ok && col0 < a.F;
          xv[u][ch] = xok[u][ch] ? load_raw<T, VEC>(xr + col0) : zero_raw<T, VEC>();
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int ch = 0; ch < CHUNKS; ++ch) {
          float x[VEC];
          unpack_raw<T, VEC>(xv[u][ch], x);
#pragma unroll
          for (int i = 0; i < VEC; ++i) {
            if (OP == 1) {
              if (xok[u][ch] && x[i] > acc[ch][i]) {
                acc[ch][i] = x[i];
                best[ch][i] = (int)(base - s) + j0 + u;
              }
            } else {
              acc[ch][i] = fmaf(vv[u], x[i], acc[ch][i]);
            }
          }
        }
    }
  }

  T* yr = a.Y + row * a.ldy;
#pragma unroll
  for (int ch = 0; ch < CHUNKS; ++ch) {
    const int col0 = (gl + ch * GROUP) * VEC;
    if (col0 < a.F) {
      float o[VEC];
#pragma unroll
      for (int i = 0; i < VEC; ++i) o[i] = (OP == 1) ? acc[ch][i] : acc[ch][i] * a.scale;
      store_cols<T, VEC>(yr + col0, o, a.F - col0);  // columns >= F stay untouched
      if (OP == 1 && a.argmax) {
#pragma unroll
        for (int i = 0; i < VEC; ++i)
          if (col0 + i < a.F) a.argmax[row * a.ldy + col0 + i] = best[ch][i];
      }
    }
  }
}

// ---- host-side dispatch -----------------------------------------------------------
template <typename T>
inline int pick_vec(const void* X, int64_t ldx, const void* Y, int64_t ldy, int F) {
  for (int v = 16 / (int)sizeof(T); v > 1; v >>= 1) {
    const size_t bytes = (size_t)v * sizeof(T);
    const int64_t fpad = ((int64_t)F + v - 1) / v * v;
    if (aligned_to(X, bytes) && aligned_to(Y, bytes) && ldx % v == 0 && ldy % v == 0 && fpad <= ldx && fpad <= ldy)
      return v;
  }
  return 1;
}

template <typename T, int VEC, int GROUP, int CHUNKS, int OP>
inline void launch_row_reduce_inst(const RowArgs<T>& a, cudaStream_t st) {
  constexpr int WORDS = CHUNKS * VecRaw<T, VEC>::W;
  constexpr int U0 = (WORDS <= 4) ? 8 : (WORDS <= 12 ? 4 : 2);
  constexpr int U = U0 < GROUP ? U0 : GROUP;
  constexpr int ROWS_PER_CTA = kRowReduceThreads / GROUP;
  const int64_t grid = (a.n_rows + ROWS_PER_CTA - 1) / ROWS_PER_CTA;
  row_reduce_kernel<T, VEC, GROUP, CHUNKS, U, OP><<<(unsigned)grid, kRowReduceThreads, 0, st>>>(a);
}

template <typename T, int VEC, int OP>
inline int launch_row_reduce_vec(const RowArgs<T>& a0, cudaStream_t st) {
  // column tiles of at most 32 lanes x 8 chunks x VEC elements
  const int tile_cols = 32 * 8 * VEC;
  for (int c0 = 0; c0 < a0.F; c0 += tile_cols) {
    RowArgs<T> a = a0;
    a.X = a0.X + c0;
    a.Y = a0.Y + c0;
    if (a0.argmax) a.argmax = a0.argmax + c0;
    a.F = (a0.F - c0) < tile_cols ? (a0.F - c0) : tile_cols;
    const int nvec = (a.F + VEC - 1) / VEC;
    if (nvec <= 4) launch_row_reduce_inst<T, VEC, 4, 1, OP>(a, st);
    else if (nvec <= 8) launch_row_reduce_inst<T, VEC, 8, 1, OP>(a, st);
    else if (nvec <= 16) launch_row_reduce_inst<T, VEC, 16, 1, OP>(a, st);
    else if (nvec <= 32) launch_row_reduce_inst<T, VEC, 32, 1, OP>(a, st);
    else if (nvec <= 64) launch_row_reduce_inst<T, VEC, 32, 2, OP>(a, st);
    else if (nvec <= 96) launch_row_reduce_inst<T, VEC, 32, 3, OP>(a, st);
    else if (nvec <= 128) launch_row_reduce_inst<T, VEC, 32, 4, OP>(a, st);
    else if (nvec <= 160) launch_row_reduce_inst<T, VEC, 32, 5, OP>(a, st);
    else if (nvec <= 192) launch_row_reduce_inst<T, VEC, 32, 6, OP>(a, st);
    else launch_row_reduce_inst<T, VEC, 32, 8, OP>(a, st);
    GNN_LAUNCH_CHECK();
  }
  return GNN_OK;
}

template <typename T, int OP>
inline int launch_row_reduce(const RowArgs<T>& a, cudaStream_t st) {
  if (a.n_rows <= 0 || a.F <= 0) return GNN_OK;
  GNN_REQUIRE((a.n_rows + 7) / 8 < 0x7fffffffLL, GNN_ERR_UNSUPPORTED, "too many rows for one grid: %lld", (long long)a.n_rows);
  const int vec = pick_vec<T>(a.X, a.ldx, a.Y, a.ldy, a.F);
  if (sizeof(T) == 2 && vec == 8) return launch_row_reduce_vec<T, (sizeof(T) == 2 ? 8 : 4), OP>(a, st);
  if (vec >= 4) return launch_row_reduce_vec<T, 4, OP>(a, st);
  if (vec == 2) return launch_row_reduce_vec<T, 2, OP>(a, st);
  return launch_row_reduce_vec<T, 1, OP>(a, st);
}

}  // namespace gnn
