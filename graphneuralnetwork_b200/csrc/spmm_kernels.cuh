// CSR SpMM kernels for Y = Â·X (replaces torch.spmm, /root/reference GCN/GCN.py:43).
//
//  spmm_rbs_kernel         "row-block streaming": a team of GROUP lanes (sub-warp chosen from
//      F) owns GROUP consecutive rows.  The row pointers of the block are loaded once
//      (coalesced), then the block's edge range is streamed in coalesced batches of GROUP
//      (col,val) pairs that ignore row boundaries, with the next batch prefetched while U
//      independent 128-bit feature-row gathers of the current one are in flight.  Rows are
//      accumulated in CSR order and flushed as their last edge passes: a warp-per-row
//      segmented reduction with no atomics and no second pass (deterministic).
//  spmm_long_chunk_kernel  rows longer than the "spmm.long_row" knob are cut into chunks of
//      "spmm.chunk" edges, one CTA per chunk; for narrow F the 32 lanes of a warp split into
//      (edge slot x vector) so a full warp gathers 32/GROUP edges per instruction and the
//      slots are combined by warp shuffle.  Per-chunk partial sums go to a workspace and
//  spmm_long_finalize_kernel adds them per row in chunk order (fixed order => deterministic).
#pragma once
#include "common.cuh"

namespace gnn {

template <typename T>
struct SpmmArgs {
  const int64_t* rowptr;
  const int32_t* col;
  const float* val;  // nullptr => 1
  const T* X;
  int64_t ldx;
  T* Y;
  int64_t ldy;
  int64_t n_rows;
  int32_t F;
  int64_t skip_deg_gt;  // >0: rows with more edges belong to the long-row kernels
  int32_t accumulate;   // 1: Y += Â·X (second pass of the partitioned SpMM), 0: Y = Â·X
  int32_t rows_per_team;  // rows a team of GROUP lanes owns (1..GROUP); 0 = GROUP
  // fused epilogue of the GCN layer (GCN/GCN.py:44-45 `output + self.bias`, GCN.py:12 nn.ReLU):
  const float* bias;      // nullable, [F] fp32, added to every row
  int32_t relu;           // 1: max(., 0) after the bias
  // ---- row-subset / two-table form (gnn_spmm_csr_ex_*; the partitioned SpMM's wave consumers) ----
  const int32_t* row_map;  // nullable: the CSR is COMPACT (n_rows selected rows); row r writes Y row row_map[r]
  int64_t acc_prefix;      // compact rows [0, acc_prefix) accumulate into Y even when accumulate == 0
  const T* X2;             // SPLIT kernels: a column id c >= split reads row (c - split) of X2 (the halo buffer);
  int64_t ldx2;            //   the host passes X2 pre-offset by -split rows, so the row is X2 + c * ldx2
  int32_t split;
  int32_t excl_smem;       // host only: token dynamic shared memory per CTA (keeps CTAs off SMs a mover filled)
  int64_t epi_skip;        // compact rows [0, epi_skip) get no bias/ReLU epilogue (first pass of two-pass rows)
};

// source row of column id c (SPLIT: two tables, [0, split) -> X, [split, ...) -> X2)
template <typename T, bool SPLIT>
__device__ __forceinline__ const T* spmm_src_row(const SpmmArgs<T>& a, int32_t c) {
  if (SPLIT) {
    // one select of (base, stride) and one multiply-add: X2 arrives pre-offset by -split rows
    const bool loc = c < a.split;
    return (loc ? a.X : a.X2) + (int64_t)c * (loc ? a.ldx : a.ldx2);
  }
  return a.X + (int64_t)c * a.ldx;
}

// y = relu?(acc + bias[col0..]) for the VEC columns starting at col0 (columns >= F are padding)
template <int VEC>
__device__ __forceinline__ void spmm_epilogue(float (&acc)[VEC], const float* bias, int relu, int col0, int F) {
  if (bias) {
#pragma unroll
    for (int i = 0; i < VEC; ++i)
      if (col0 + i < F) acc[i] += __ldg(bias + col0 + i);
  }
  if (relu) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[i] = fmaxf(acc[i], 0.f);
  }
}

constexpr int kSpmmThreads = 256;

// One-vector-per-lane variants are held to 64 registers (4 CTAs/SM): next to the 3 CTAs that a
// concurrently running halo-push CTA leaves room for, this keeps the local-column pass of the
// partitioned SpMM at full occupancy (at 80 registers it dropped from 3 to 2 CTAs per SM).
// MINB: CTAs per SM the register allocation is held to.  Multi-vector rows (CHUNKS 2..5) run the
// instantiation held to 3 CTAs/SM (80 registers, a few spilled words): on the Reddit-shaped graph the
// kernel is latency-bound and the third CTA is worth 4-11 % (F=602 fp32 34.1 -> 30.6 ms, bf16 23.6 ->
// 21.7 ms; profiles/r01s2_kbench_spmm_reddit_ctas3_ab.jsonl).  "spmm.ctas3" = 0 selects the unconstrained
// instantiation (100-140 registers, 2 CTAs/SM).
// SKIP: the epilogue honours epi_skip (a separate instantiation, so the plain epilogue keeps its registers).
template <typename T, int VEC, int GROUP, int CHUNKS, int U, bool EPI, int MINB = ((CHUNKS == 1) ? 4 : 1), bool SPLIT = false,
          bool SKIP = false>
__global__ void __launch_bounds__(kSpmmThreads, MINB) spmm_rbs_kernel(const SpmmArgs<T> a) {
  const int lane = threadIdx.x & 31;
  const int gl = threadIdx.x % GROUP;
  const unsigned gmask = (GROUP == 32) ? 0xffffffffu : (((1u << GROUP) - 1u) << (lane - gl));
  // A team owns rpt consecutive rows.  rpt = GROUP suits sparse rows (papers100M: 14 edges per
  // row, 460 per team); on dense graphs (Reddit: 490 per row) 32 rows per team left 7,288 warps
  // for the whole graph, each walking 15,000 edges at one DRAM round trip per U of them, so the
  // host lowers rpt until a team holds a few hundred edges.
  const int rpt = (a.rows_per_team > 0 && a.rows_per_team < GROUP) ? a.rows_per_team : GROUP;
  const int64_t team = ((int64_t)blockIdx.x * kSpmmThreads + threadIdx.x) / GROUP;
  const int64_t r0 = team * rpt;
  if (r0 >= a.n_rows) return;
  const int nr = (int)((a.n_rows - r0) < (int64_t)rpt ? (a.n_rows - r0) : (int64_t)rpt);
  const int64_t rlo = r0 + (gl < nr ? gl : nr);          // lanes past the team's rows hold an
  const int64_t rhi = r0 + (gl + 1 < nr ? gl + 1 : nr);  // empty range at the team's end
  const int64_t lo = __ldg(a.rowptr + rlo), hi = __ldg(a.rowptr + rhi);
  const bool is_long = a.skip_deg_gt > 0 && (hi - lo) > a.skip_deg_gt;
  const unsigned longs = __ballot_sync(gmask, is_long) & gmask;

  float acc[CHUNKS][VEC];
#pragma unroll
  for (int ch = 0; ch < CHUNKS; ++ch)
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[ch][i] = 0.f;

  auto flush = [&](int r) {
    const int64_t orow = a.row_map ? (int64_t)__ldg(a.row_map + r0 + r) : (r0 + r);
    T* yr = a.Y + orow * a.ldy;
    const bool accum = a.accumulate || (r0 + r) < a.acc_prefix;
#pragma unroll
    for (int ch = 0; ch < CHUNKS; ++ch) {
      const int col0 = (gl + ch * GROUP) * VEC;
      if (col0 < a.F) {  // columns >= F of Y are neither read nor written
        if (accum) {
          float prev[VEC];
          load_cols<T, VEC>(yr + col0, prev, a.F - col0);
#pragma unroll
          for (int i = 0; i < VEC; ++i) acc[ch][i] += prev[i];
        }
        if (EPI && (!SKIP || (r0 + r) >= a.epi_skip)) spmm_epilogue<VEC>(acc[ch], a.bias, a.relu, col0, a.F);
        store_cols<T, VEC>(yr + col0, acc[ch], a.F - col0);
      }
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[ch][i] = 0.f;
    }
  };

  if (longs == 0) {
    // ---- fast path: stream the whole block's edges, flushing rows as they end ----
    const int64_t E0 = __shfl_sync(gmask, lo, 0, GROUP);
    const int64_t E1 = __shfl_sync(gmask, hi, GROUP - 1, GROUP);
    int cur = 0;
    int64_t cur_end = __shfl_sync(gmask, hi, 0, GROUP);
    int32_t c_n = 0;
    float v_n = 0.f;
    if (E0 + gl < E1) {
      c_n = __ldg(a.col + E0 + gl);
      v_n = a.val ? __ldg(a.val + E0 + gl) : 1.f;
    }
    for (int64_t base = E0; base < E1; base += GROUP) {
      const int32_t c = c_n;
      const float v = v_n;
      const int64_t kn = base + GROUP + gl;
      if (kn < E1) {  // prefetch the next batch while this one is gathered
        c_n = __ldg(a.col + kn);
        v_n = a.val ? __ldg(a.val + kn) : 1.f;
      }
      const int cnt = (int)((E1 - base) < (int64_t)GROUP ? (E1 - base) : (int64_t)GROUP);
      for (int j0 = 0; j0 < cnt; j0 += U) {
        VecRaw<T, VEC> xv[U][CHUNKS];
        float vv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int jj = j0 + u;
          const int32_t cj = __shfl_sync(gmask, c, jj, GROUP);
          vv[u] = __shfl_sync(gmask, v, jj, GROUP);
          const bool ok = jj < cnt;
          const T* xr = spmm_src_row<T, SPLIT>(a, ok ? cj : 0);
#pragma unroll
          for (int ch = 0; ch < CHUNKS; ++ch) {
            const int col0 = (gl + ch * GROUP) * VEC;
            xv[u][ch] = (ok && col0 < a.F) ? load_raw<T, VEC>(xr + col0) : zero_raw<T, VEC>();
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int jj = j0 + u;
          if (jj < cnt) {
            const int64_t e = base + jj;
            while (e >= cur_end) {  // uniform in the team; also steps over empty rows
              flush(cur);
              ++cur;
              cur_end = __shfl_sync(gmask, hi, cur, GROUP);
            }
#pragma unroll
            for (int ch = 0; ch < CHUNKS; ++ch) {
              float x[VEC];
              unpack_raw<T, VEC>(xv[u][ch], x);
#pragma unroll
              for (int i = 0; i < VEC; ++i) acc[ch][i] = fmaf(vv[u], x[i], acc[ch][i]);
            }
          }
        }
      }
    }
    for (; cur < nr; ++cur) flush(cur);
    return;
  }

  // ---- block contains long rows: walk row by row, leaving the long ones to their kernels ----
  for (int r = 0; r < nr; ++r) {
    const int64_t s = __shfl_sync(gmask, lo, r, GROUP);
    const int64_t e = __shfl_sync(gmask, hi, r, GROUP);
    if ((longs >> ((lane - gl) + r)) & 1u) continue;
    for (int64_t base = s; base < e; base += GROUP) {
      const int64_t k = base + gl;
      int32_t c = 0;
      float v = 0.f;
      if (k < e) {
        c = __ldg(a.col + k);
        v = a.val ? __ldg(a.val + k) : 1.f;
      }
      const int cnt = (int)((e - base) < (int64_t)GROUP ? (e - base) : (int64_t)GROUP);
      for (int j0 = 0; j0 < cnt; j0 += U) {
        VecRaw<T, VEC> xv[U][CHUNKS];
        float vv[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int jj = j0 + u;
          const int32_t cj = __shfl_sync(gmask, c, jj, GROUP);
          const float vj = __shfl_sync(gmask, v, jj, GROUP);
          const bool ok = jj < cnt;
          vv[u] = ok ? vj : 0.f;
          const T* xr = spmm_src_row<T, SPLIT>(a, ok ? cj : 0);
#pragma unroll
          for (int ch = 0; ch < CHUNKS; ++ch) {
            const int col0 = (gl + ch * GROUP) * VEC;
            xv[u][ch] = (ok && col0 < a.F) ? load_raw<T, VEC>(xr + col0) : zero_raw<T, VEC>();
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int ch = 0; ch < CHUNKS; ++ch) {
            float x[VEC];
            unpack_raw<T, VEC>(xv[u][ch], x);
#pragma unroll
            for (int i = 0; i < VEC; ++i) acc[ch][i] = fmaf(vv[u], x[i], acc[ch][i]);
          }
      }
    }
    flush(r);
  }
}

// ---- long rows --------------------------------------------------------------------------
constexpr int kLongChunkWarps = 8;

template <typename T, int VEC, int GROUP, int CHUNKS, bool SPLIT = false>
__global__ void __launch_bounds__(kLongChunkWarps * 32)
    spmm_long_chunk_kernel(const SpmmArgs<T> a, const int64_t* __restrict__ long_rows,
                           const int64_t* __restrict__ chunk_off, int64_t n_long, int chunk_edges,
                           float* __restrict__ partial, int ldp) {
  constexpr int EPW = 32 / GROUP;  // edges gathered per warp instruction
  constexpr int U = (CHUNKS == 1) ? (EPW >= 4 ? 4 : 8) : (CHUNKS <= 2 ? 4 : 2);
  __shared__ float part[kLongChunkWarps][CHUNKS * GROUP * VEC];
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const int gl = lane % GROUP;
  const int eslot = lane / GROUP;
  // which long row does this chunk belong to?  chunk_off is ascending, n_long+1 entries
  const int64_t id = blockIdx.x;
  int64_t lo_i = 0, hi_i = n_long;
  while (hi_i - lo_i > 1) {
    const int64_t mid = (lo_i + hi_i) >> 1;
    if (__ldg(chunk_off + mid) <= id) lo_i = mid; else hi_i = mid;
  }
  const int64_t row = __ldg(long_rows + lo_i);
  const int64_t kchunk = id - __ldg(chunk_off + lo_i);
  const int64_t s = __ldg(a.rowptr + row) + kchunk * chunk_edges;
  int64_t e = __ldg(a.rowptr + row + 1);
  e = (s + chunk_edges < e) ? s + chunk_edges : e;

  float acc[CHUNKS][VEC];
#pragma unroll
  for (int ch = 0; ch < CHUNKS; ++ch)
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[ch][i] = 0.f;

  for (int64_t base = s + (int64_t)w * 32; base < e; base += (int64_t)kLongChunkWarps * 32) {
    const int64_t k = base + lane;
    int32_t c = 0;
    float v = 0.f;
    if (k < e) {
      c = __ldg(a.col + k);
      v = a.val ? __ldg(a.val + k) : 1.f;
    }
    const int cnt = (int)((e - base) < 32 ? (e - base) : 32);
    for (int j0 = 0; j0 < cnt; j0 += EPW * U) {
      VecRaw<T, VEC> xv[U][CHUNKS];
      float vv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int jj = j0 + u * EPW + eslot;
        const int32_t cj = __shfl_sync(0xffffffffu, c, jj & 31);
        const float vj = __shfl_sync(0xffffffffu, v, jj & 31);
        const bool ok = jj < cnt;
        vv[u] = ok ? vj : 0.f;
        const T* xr = spmm_src_row<T, SPLIT>(a, ok ? cj : 0);
#pragma unroll
        for (int ch = 0; ch < CHUNKS; ++ch) {
          const int col0 = (gl + ch * GROUP) * VEC;
          xv[u][ch] = (ok && col0 < a.F) ? load_raw<T, VEC>(xr + col0) : zero_raw<T, VEC>();
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int ch = 0; ch < CHUNKS; ++ch) {
          float x[VEC];
          unpack_raw<T, VEC>(xv[u][ch], x);
#pragma unroll
          for (int i = 0; i < VEC; ++i) acc[ch][i] = fmaf(vv[u], x[i], acc[ch][i]);
        }
    }
  }
  // combine the edge slots of the warp (fixed butterfly), then the warps (fixed order)
#pragma unroll
  for (int off = GROUP; off < 32; off <<= 1)
#pragma unroll
    for (int ch = 0; ch < CHUNKS; ++ch)
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[ch][i] += __shfl_xor_sync(0xffffffffu, acc[ch][i], off);
  if (eslot == 0) {
#pragma unroll
    for (int ch = 0; ch < CHUNKS; ++ch)
#pragma unroll
      for (int i = 0; i < VEC; ++i) part[w][(ch * GROUP + gl) * VEC + i] = acc[ch][i];
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < CHUNKS * GROUP * VEC; idx += kLongChunkWarps * 32) {
    if (idx < a.F) {  // idx == column: (ch*GROUP+gl)*VEC+i == (gl + ch*GROUP)*VEC + i
      float sum = 0.f;
#pragma unroll
      for (int ww = 0; ww < kLongChunkWarps; ++ww) sum += part[ww][idx];
      partial[id * ldp + idx] = sum;
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
    spmm_long_finalize_kernel(const int64_t* __restrict__ long_rows, const int64_t* __restrict__ chunk_off,
                              const float* __restrict__ partial, int ldp, int col_base, int Ftile, T* __restrict__ Y,
                              int64_t ldy, int accumulate, const float* __restrict__ bias, int relu,
                              const int32_t* __restrict__ row_map, int64_t acc_prefix, int64_t epi_skip) {
  const int64_t r = blockIdx.x;
  const int64_t crow = __ldg(long_rows + r);  // (compact) CSR row
  const int64_t row = row_map ? (int64_t)__ldg(row_map + crow) : crow;
  accumulate = accumulate || crow < acc_prefix;
  if (crow < epi_skip) {  // first pass of a two-pass row: its epilogue comes with the last contribution
    bias = nullptr;
    relu = 0;
  }
  const int64_t c0 = __ldg(chunk_off + r), c1 = __ldg(chunk_off + r + 1);
  for (int f = threadIdx.x; f < Ftile; f += blockDim.x) {
    float sum = 0.f;
    for (int64_t c = c0; c < c1; ++c) sum += __ldg(partial + c * ldp + f);
    if (accumulate) {
      float prev[1];
      VecIO<T, 1>::load(Y + row * ldy + col_base + f, prev);
      sum += prev[0];
    }
    if (bias) sum += __ldg(bias + col_base + f);
    if (relu) sum = fmaxf(sum, 0.f);
    float o[1] = {sum};
    VecIO<T, 1>::store(Y + row * ldy + col_base + f, o);
  }
}

// ---- host-side dispatch ------------------------------------------------------------------
template <typename T>
inline int spmm_pick_vec(const void* X, int64_t ldx, const void* Y, int64_t ldy, int F, const void* X2 = nullptr,
                         int64_t ldx2 = 0) {
  for (int v = 16 / (int)sizeof(T); v > 1; v >>= 1) {
    const size_t bytes = (size_t)v * sizeof(T);
    const int64_t fpad = ((int64_t)F + v - 1) / v * v;
    if (aligned_to(X, bytes) && aligned_to(Y, bytes) && ldx % v == 0 && ldy % v == 0 && fpad <= ldx && fpad <= ldy &&
        (!X2 || (aligned_to(X2, bytes) && ldx2 % v == 0 && fpad <= ldx2)))
      return v;
  }
  return 1;
}

template <typename T, int VEC, int GROUP, int CHUNKS>
inline void spmm_rbs_launch(const SpmmArgs<T>& a, cudaStream_t st) {
  // gathers in flight per lane: about 8 x 16 bytes of staging registers
  constexpr int WORDS = CHUNKS * VecRaw<T, VEC>::W;
  constexpr int U0 = (WORDS <= 4) ? 8 : (WORDS <= 12 ? 4 : 2);
  constexpr int U = U0 < GROUP ? U0 : GROUP;
  const int rpt = (a.rows_per_team > 0 && a.rows_per_team < GROUP) ? a.rows_per_team : GROUP;
  const int64_t teams = (a.n_rows + rpt - 1) / rpt;
  const int64_t grid = (teams * GROUP + kSpmmThreads - 1) / kSpmmThreads;
  // the bias/ReLU epilogue is a separate instantiation: the plain one keeps its register budget
  // token dynamic shared memory (<= 48 KB, unused by the kernel) keeps these CTAs off the SMs a
  // dedicated halo push has claimed (peer.cu); 0 outside the partitioned SpMM's local pass
  const size_t sm = (size_t)(a.excl_smem > 0 ? a.excl_smem : 0);
  constexpr int MINB_DEF = (CHUNKS == 1) ? 4 : ((CHUNKS <= 5) ? 3 : 1);
  // the partitioned SpMM's consumers with the GCN epilogue (two-table pass, first pass + finished rows in one
  // launch): held to a register budget that does not spill
  constexpr int MINB_EPI = (CHUNKS == 1) ? 2 : 1;
  const bool epi = a.bias || a.relu;
  if (a.split != 0x7fffffff) {
    if (epi)
      spmm_rbs_kernel<T, VEC, GROUP, CHUNKS, U, true, MINB_EPI, true, true><<<(unsigned)grid, kSpmmThreads, sm, st>>>(a);
    else
      spmm_rbs_kernel<T, VEC, GROUP, CHUNKS, U, false, MINB_DEF, true><<<(unsigned)grid, kSpmmThreads, sm, st>>>(a);
  } else if (epi && a.epi_skip > 0) {
    spmm_rbs_kernel<T, VEC, GROUP, CHUNKS, U, true, MINB_EPI, false, true><<<(unsigned)grid, kSpmmThreads, sm, st>>>(a);
  } else if (epi) {
    spmm_rbs_kernel<T, VEC, GROUP, CHUNKS, U, true><<<(unsigned)grid, kSpmmThreads, sm, st>>>(a);
  } else if (CHUNKS >= 2 && CHUNKS <= 5 && tuning("spmm.ctas3", 1)) {
    spmm_rbs_kernel<T, VEC, GROUP, CHUNKS, U, false, (CHUNKS >= 2 && CHUNKS <= 5) ? 3 : 1>
        <<<(unsigned)grid, kSpmmThreads, sm, st>>>(a);
  } else {
    spmm_rbs_kernel<T, VEC, GROUP, CHUNKS, U, false><<<(unsigned)grid, kSpmmThreads, sm, st>>>(a);
  }
}

template <typename T, int VEC>
inline int spmm_main_vec(const SpmmArgs<T>& a0, cudaStream_t st) {
  const int tile_cols = 32 * 8 * VEC;
  for (int c0 = 0; c0 < a0.F; c0 += tile_cols) {
    SpmmArgs<T> a = a0;
    a.X = a0.X + c0;
    a.X2 = (a0.split != 0x7fffffff) ? a0.X2 + c0 : nullptr;
    a.Y = a0.Y + c0;
    a.bias = a0.bias ? a0.bias + c0 : nullptr;
    a.F = (a0.F - c0) < tile_cols ? (a0.F - c0) : tile_cols;
    const int nvec = (a.F + VEC - 1) / VEC;
    if (nvec <= 4) spmm_rbs_launch<T, VEC, 4, 1>(a, st);
    else if (nvec <= 8) spmm_rbs_launch<T, VEC, 8, 1>(a, st);
    else if (nvec <= 16) spmm_rbs_launch<T, VEC, 16, 1>(a, st);
    else if (nvec <= 32) spmm_rbs_launch<T, VEC, 32, 1>(a, st);
    else if (nvec <= 64) spmm_rbs_launch<T, VEC, 32, 2>(a, st);
    else if (nvec <= 96) spmm_rbs_launch<T, VEC, 32, 3>(a, st);
    else if (nvec <= 128) spmm_rbs_launch<T, VEC, 32, 4>(a, st);
    else if (nvec <= 160) spmm_rbs_launch<T, VEC, 32, 5>(a, st);
    else if (nvec <= 192) spmm_rbs_launch<T, VEC, 32, 6>(a, st);
    else spmm_rbs_launch<T, VEC, 32, 8>(a, st);
    GNN_LAUNCH_CHECK();
  }
  return GNN_OK;
}

template <typename T>
inline int spmm_main(const SpmmArgs<T>& a, cudaStream_t st) {
  GNN_REQUIRE(a.n_rows < (1LL << 33), GNN_ERR_UNSUPPORTED, "too many rows");  // grid <= n_rows / 8
  const int vec = spmm_pick_vec<T>(a.X, a.ldx, a.Y, a.ldy, a.F, (a.split != 0x7fffffff) ? a.X2 : nullptr, a.ldx2);
  if (sizeof(T) == 2 && vec == 8) return spmm_main_vec<T, (sizeof(T) == 2 ? 8 : 4)>(a, st);
  if (vec >= 4) return spmm_main_vec<T, 4>(a, st);
  if (vec == 2) return spmm_main_vec<T, 2>(a, st);
  return spmm_main_vec<T, 1>(a, st);
}

template <typename T, int VEC>
inline int spmm_long_vec(const SpmmArgs<T>& a0, const int64_t* long_rows, int64_t n_long, const int64_t* chunk_off,
                         int64_t n_chunks, int chunk_edges, float* partial, cudaStream_t st) {
  const int tile_cols = 32 * 4 * VEC;
  const int ldp = tile_cols;
  for (int c0 = 0; c0 < a0.F; c0 += tile_cols) {
    SpmmArgs<T> a = a0;
    a.X = a0.X + c0;
    a.X2 = (a0.split != 0x7fffffff) ? a0.X2 + c0 : nullptr;
    a.F = (a0.F - c0) < tile_cols ? (a0.F - c0) : tile_cols;
    const int nvec = (a.F + VEC - 1) / VEC;
    const unsigned grid = (unsigned)n_chunks;
    const int thr = kLongChunkWarps * 32;
#define GNN_LONG(G, C)                                                                                               \
  do {                                                                                                               \
    if (a.split != 0x7fffffff)                                                                                       \
      spmm_long_chunk_kernel<T, VEC, G, C, true><<<grid, thr, 0, st>>>(a, long_rows, chunk_off, n_long, chunk_edges, \
                                                                       partial, ldp);                                \
    else                                                                                                             \
      spmm_long_chunk_kernel<T, VEC, G, C><<<grid, thr, 0, st>>>(a, long_rows, chunk_off, n_long, chunk_edges,       \
                                                                 partial, ldp);                                      \
  } while (0)
    if (nvec <= 4) GNN_LONG(4, 1);
    else if (nvec <= 8) GNN_LONG(8, 1);
    else if (nvec <= 16) GNN_LONG(16, 1);
    else if (nvec <= 32) GNN_LONG(32, 1);
    else if (nvec <= 64) GNN_LONG(32, 2);
    else GNN_LONG(32, 4);
#undef GNN_LONG
    GNN_LAUNCH_CHECK();
    spmm_long_finalize_kernel<T><<<(unsigned)n_long, 256, 0, st>>>(long_rows, chunk_off, partial, ldp, c0, a.F, a0.Y,
                                                                   a0.ldy, a0.accumulate, a0.bias, a0.relu,
                                                                   a0.row_map, a0.acc_prefix, a0.epi_skip);
    GNN_LAUNCH_CHECK();
  }
  return GNN_OK;
}

template <typename T>
inline int spmm_long(const SpmmArgs<T>& a, const int64_t* long_rows, int64_t n_long, const int64_t* chunk_off,
                     int64_t n_chunks, int chunk_edges, float* partial, cudaStream_t st) {
  const int vec = spmm_pick_vec<T>(a.X, a.ldx, a.Y, a.ldy, a.F, (a.split != 0x7fffffff) ? a.X2 : nullptr, a.ldx2);
  if (sizeof(T) == 2 && vec == 8)
    return spmm_long_vec<T, (sizeof(T) == 2 ? 8 : 4)>(a, long_rows, n_long, chunk_off, n_chunks, chunk_edges, partial, st);
  if (vec >= 4) return spmm_long_vec<T, 4>(a, long_rows, n_long, chunk_off, n_chunks, chunk_edges, partial, st);
  if (vec == 2) return spmm_long_vec<T, 2>(a, long_rows, n_long, chunk_off, n_chunks, chunk_edges, partial, st);
  return spmm_long_vec<T, 1>(a, long_rows, n_long, chunk_off, n_chunks, chunk_edges, partial, st);
}

inline size_t spmm_long_workspace_bytes(int64_t n_chunks, int elem_size) {
  const int vec = 16 / elem_size;
  return (size_t)n_chunks * (size_t)(32 * 4 * vec) * sizeof(float);
}

}  // namespace gnn
