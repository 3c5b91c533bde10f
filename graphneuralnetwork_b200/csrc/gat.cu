// Fused multi-head graph attention aggregation (GAT / HAN node-level attention).
// Replaces, at /root/reference:
//   GAT/models/layers.py:25-32  (== HAN/models/NodeAttention.py:25-33)
//       the [N,N,2F'] pair tensor, masked softmax and dense attention·Wh matmul
//   GAT/models/layers.py:108-122  the edge-list variant exp(-LeakyReLU) / rowsum
//   GAT/models/layers.py:55-64    SpecialSpmmFunction.backward (dense N×N edge gradient)
//
// Forward, all H heads in one pass over a CSR row, staged through shared memory:
//   A  lane-per-edge:  logit[k,h] = ±LeakyReLU(s[i,h] + t[col_k,h])
//   B  per-head chunk max by warp shuffle, running max / rescale (softmax mode)
//   B2 logit -> p = exp(logit - max) in place: ONE exp per (edge, head)
//   C  lane-per-column: acc += p[k,head(col)] * Wh[col_k, column], 8 coalesced row gathers
//      in flight per lane
// Scheduling: W = 1 -> one warp per row (low-degree graphs: Cora); W = 4 -> one CTA per row,
// the warps take alternate 128-edge chunks and their (max, sum, acc) partials are merged in
// warp order (dense metapath / Reddit-like graphs).  Both are deterministic.
// Backward: two passes of the forward kernel's shape (see gat_bwd2_kernel): over the CSR rows for d_s, over the
// transposed CSR rows for d_Wh and d_t.  The edge gradient is never materialised per edge: it factorises into
// weighted row sums (FMA per column) plus a per-head correction.  Ordered sums only, no atomics, no edge stash.
#include "common.cuh"

using namespace gnn;

namespace {

constexpr int kGatWarps = 4;

struct GatArgs {
  const int64_t* rowptr;
  const int32_t* col;
  const int64_t* perm;   // backward pass 2: transposed slot -> forward edge slot (dropout factors only)
  const void* Wh;        // T [n, ldw]: fp32 or bf16 (softmax and accumulation are fp32 either way)
  int64_t ldw;
  const float* s;
  const float* t;
  int64_t n;
  int H, Hp, Fp, HF;
  float alpha;
  int mode;
  int elu;
  const float* col_mean;
  const float* keep;     // explicit post-softmax dropout factors [nnz, H] (parity tests); else the seeded stream below
  float keep_prob;       // > 0 with drop_seed: keep an (edge, head) with this probability, scaled by drop_scale
  float drop_scale;      // 1 / keep_prob
  uint64_t drop_seed;    // host half of the seed
  const int64_t* drop_seed_dev;  // device half (nullable): a captured CUDA graph draws a fresh mask per replay
  void* out;             // T [n, ldo]: the aggregate (activated unless out_act is given)
  void* out_act;         // T [n, ldo], nullable (training): out keeps the PRE-activation aggregate for the backward,
                         //   out_act receives the activated one — the ELU(s) never run as separate launches
  int64_t ldo;
  float* row_max;
  float* row_sum;
  // batched graphs (HAN's M metapaths over the same nodes, HAN/models/HAN.py:16-23, in ONE launch): the CSR is the
  // block diagonal of M graphs of batch_n nodes (row r = graph r / batch_n, node r % batch_n; col ids offset
  // likewise); s, t, row statistics and d_s / d_t are indexed by the batched row, graph m's feature columns sit
  // at column offset m * HF of Wh / out / d_out / d_Wh.  0 = one graph.
  int64_t batch_n;
  int SE;
  int packed;  // bf16 rows 4-byte aligned with even head width: lanes own column pairs (PK = 2)
  // backward
  const void* out_pre;   // T
  const void* d_out;     // T
  float* rowstat;        // [n][4][H] fp32: s, row max, 1/row sum, D = <d_out_i, out_pre_i> per head (backward)
  void* d_Wh;            // T
  int64_t ld_dwh;
  float* d_s;
  float* d_t;
  // schedule: the warp-per-row launch leaves rows longer than skip_deg_gt to the CTA-per-row
  // launch, which walks row_list (nullable: row = blockIdx.x)
  const int64_t* row_list;
  int64_t skip_deg_gt;
  // batched AND rectangular (RB kernels, a rank's block of M metapaths): batch_n is the stride of this launch's rows
  // (graph gm = row / batch_n, own row = row - gm * batch_n) and col_stride the stride of its column ids (graph gm's
  // ids start at gm * col_stride) — the forward rows' and the table rows' counts, swapped in the transposed pass.
  // slot_shift[gm] (nullable) moves graph gm's seeded-dropout slots.
  int64_t col_stride;
  const int64_t* slot_shift;
};

__device__ __forceinline__ bool aligned_to_dev(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

template <typename T>
__device__ __forceinline__ float ldv(const T* p);
template <>
__device__ __forceinline__ float ldv<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float ldv<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __uint_as_float(((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p))) << 16);
}
// raw (unconverted) staging of gathered values: the loads of a batch are all issued before the first
// conversion (with ldv<bf16> in the gather loop every shift waited on its own 2-byte load: ncu r02, 43 % of the
// bf16 forward's stall samples sat on those shifts)
template <typename T>
struct RawOf { using type = float; };
// (a bf16 value is staged zero-extended in a full 32-bit register: staged as 16-bit halves, ptxas gave several
// in-flight loads the same register and the batch serialised load -> shift -> load)
template <>
struct RawOf<__nv_bfloat16> { using type = uint32_t; };
__device__ __forceinline__ float ld_raw(const float* p) { return __ldg(p); }
// The staged word is the aligned 32-bit word that CONTAINS the element (rows are 4-byte aligned: checked on the
// host); the element's half is selected at use.  16-bit loads (LDG.U16) made ptxas funnel a whole batch of
// in-flight loads through one destination register.
__device__ __forceinline__ uint32_t ld_raw(const __nv_bfloat16* p) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3));
  return (a & 2) ? (w & 0xffff0000u) : (w << 16);
}
__device__ __forceinline__ float raw_to_f(float v) { return v; }
__device__ __forceinline__ float raw_to_f(uint32_t v) { return __uint_as_float(v); }

// Column owned by (lane, c).  PK = 1: lane + 32c (one element per load).  PK = 2 (bf16 rows that are 4-byte
// aligned): the pair (2q, 2q+1) of one 32-bit word, q = lane + 32*(c/2) — one 32-bit load per lane serves two
// columns, the load pattern of the fp32 kernel at half the bytes.
template <int PK>
__device__ __forceinline__ int col_of(int lane, int c) {
  return PK == 1 ? lane + 32 * c : (lane + 32 * (c >> 1)) * 2 + (c & 1);
}
// one staged load: PK = 1 -> the element (see ld_raw), PK = 2 -> the raw 32-bit word holding the pair
template <typename T, int PK>
__device__ __forceinline__ typename RawOf<T>::type ld_stage(const T* row, int lane, int q) {
  if constexpr (PK == 1) {
    return ld_raw(row + lane + 32 * q);
  } else {
    return __ldg(reinterpret_cast<const uint32_t*>(row) + lane + 32 * q);
  }
}
// element c of the lane from the staged loads (x[c / PK])
template <typename T, int PK>
__device__ __forceinline__ float stage_elem(typename RawOf<T>::type v, int c) {
  if constexpr (PK == 1) {
    return raw_to_f(v);
  } else {
    return __uint_as_float((c & 1) ? (v & 0xffff0000u) : (v << 16));
  }
}

template <typename T>
__device__ __forceinline__ float round_as(float v) {
  if constexpr (sizeof(T) == 2) return __bfloat162float(__float2bfloat16_rn(v));
  return v;
}
__device__ __forceinline__ void stv(float* p, float v) { *p = v; }
__device__ __forceinline__ void stv(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// Counter-based dropout stream (splitmix64 of seed + (edge slot, head)): the SAME factor is recomputed by the
// forward and by both backward passes from the forward edge slot, so no [nnz, H] mask is ever materialised
// (layers.py:31 applies F.dropout to the dense N x N attention; parity is semantic — and bit-exact against
// functional.attention_keep_mask_from_seed, the torch restatement of this hash).
__device__ __forceinline__ uint64_t drop_seed_of(const GatArgs& a) {
  uint64_t s = a.drop_seed;
  if (a.drop_seed_dev) s ^= (uint64_t)__ldg(a.drop_seed_dev) * 0xD6E8FEB86659FD93ULL;
  return s;
}
__device__ __forceinline__ float keep_factor(uint64_t seed, int64_t e, int h, int H, uint32_t thresh24, float scale) {
  uint64_t z = seed + (uint64_t)(e * H + h + 1) * 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  z ^= z >> 31;
  return (uint32_t)(z >> 40) < thresh24 ? scale : 0.f;
}

__device__ __forceinline__ float act_elu(float x, int elu) {
  if (elu >= 1) x = elu1(x);
  if (elu >= 2) x = elu1(x);
  return x;
}

// floats of shared memory per warp for the staged chunk
__host__ __device__ inline int gat_warp_floats(int SE, int H, int HF) { return SE * H + SE + 160 + HF; }
// W  = warps that share one row: 1 -> one warp per row (4 rows per CTA); 4 / 16 -> one CTA of W
//      warps per row, the warps take alternate SE-edge chunks and merge (max, sum, acc) in warp order.
// HT = compile-time head count (1, 8; must divide 32) or 0 for the generic run-time H.  With HT known
//      the per-lane head of phase B/B2 is fixed (lane % HT), t rows are loaded as vectors, the row sum
//      is reduced once per chunk instead of once per edge, and all index arithmetic folds away
//      (the generic path executed 79 warp instructions per edge, ncu profiles/r01_prof_gat_fwd_raw.csv).
template <int W>
struct GatBlock {
  static constexpr int kWarps = (W == 1) ? kGatWarps : W;
};

template <typename T, int CPL, int W, int HT, int PK, bool RB = false>
__global__ void __launch_bounds__(GatBlock<W>::kWarps * 32) gat_fwd_kernel(const GatArgs a) {
  constexpr int BW = GatBlock<W>::kWarps;
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t i = (W == 1) ? (int64_t)blockIdx.x * kGatWarps + warp
                             : (a.row_list ? __ldg(a.row_list + blockIdx.x) : (int64_t)blockIdx.x);
  const int wsub = (W == 1) ? 0 : warp;
  if (W == 1 && i >= a.n) return;  // warp-uniform; the W == 1 schedule has no block-wide barrier
  const int H = HT ? HT : a.H, Hp = HT ? HT : a.Hp, SE = a.SE;
  const int PW = gat_warp_floats(SE, H, a.HF);
  float* logit = sm + (size_t)warp * PW;
  int* cols = reinterpret_cast<int*>(logit + SE * H);
  float* mh = reinterpret_cast<float*>(cols + SE);  // [32] running max per head
  float* sc = mh + 32;                              // [32] rescale factor of this chunk
  float* lh = sc + 32;                              // [32] running sum per head (HT path)
  float* marr = sm + (size_t)BW * PW;               // [BW][32]
  float* larr = marr + BW * 32;                     // [BW][CPL*32]
  float* aarr = larr + BW * CPL * 32;               // [BW][CPL*32]

  int hc[CPL];
  bool cv[CPL];
  float acc[CPL], l[CPL];
#pragma unroll
  for (int c = 0; c < CPL; ++c) {
    const int ci = col_of<PK>(lane, c);
    cv[c] = ci < a.HF;
    hc[c] = cv[c] ? ci / a.Fp : 0;
    acc[c] = 0.f;
    l[c] = 0.f;
  }
  const int64_t e0 = __ldg(a.rowptr + i), e1 = __ldg(a.rowptr + i + 1);
  const int64_t d = e1 - e0;
  if (W == 1 && a.skip_deg_gt > 0 && d > a.skip_deg_gt) return;  // a long row: the CTA-per-row launch owns it
  const int64_t gm = a.batch_n ? i / a.batch_n : 0;      // graph of this row (batched launch)
  const int64_t joff = gm * (RB ? a.col_stride : a.batch_n);  // its col ids are offset by joff
  const int64_t roff = RB ? gm * a.batch_n : joff;        // its output row is i - roff
  const int64_t coff = gm * a.HF;                         // its feature columns start at coff
  T* orow = reinterpret_cast<T*>(a.out) + (i - roff) * a.ldo + coff;
  T* arow = a.out_act ? reinterpret_cast<T*>(a.out_act) + (i - roff) * a.ldo + coff : nullptr;
  const bool seeded = a.keep == nullptr && a.keep_prob > 0.f;
  uint64_t dseed = seeded ? drop_seed_of(a) : 0;
  // slot e + shift under seed s is slot e under seed s + shift*H*golden (see set_dropout)
  if (RB && seeded && a.slot_shift) dseed += (uint64_t)__ldg(a.slot_shift + gm) * (uint64_t)a.H * 0x9E3779B97F4A7C15ULL;
  const uint32_t thresh24 = (uint32_t)(a.keep_prob * 16777216.f);
  if (d == 0) {
    // GAT/models/layers.py:28-30: an all -9e15 row soft-maxes to the uniform 1/N over ALL nodes
    if (wsub == 0) {
#pragma unroll
      for (int c = 0; c < CPL; ++c)
        if (cv[c]) {
          const int ci = col_of<PK>(lane, c);
          const float v0 = a.col_mean ? a.col_mean[coff + ci] : 0.f;
          stv(orow + ci, arow ? v0 : act_elu(v0, a.elu));
          if (arow) stv(arow + ci, act_elu(v0, a.elu));
          if (ci % a.Fp == 0) {
            if (a.row_max) a.row_max[i * H + hc[c]] = 0.f;
            if (a.row_sum) a.row_sum[i * H + hc[c]] = 0.f;
          }
        }
    }
    return;  // uniform over the CTA when W > 1 (one row per CTA)
  }
  if (lane < Hp) {
    mh[lane] = (a.mode == GNN_GAT_SOFTMAX) ? -INFINITY : 0.f;
    sc[lane] = 1.f;
    lh[lane] = 0.f;
  }
  __syncwarp();
  const int ngrp = 32 / Hp;
  const int hsub = lane % Hp, g = lane / Hp;
  float si_reg[HT ? HT : 1];
  if (HT) {
#pragma unroll
    for (int h = 0; h < (HT ? HT : 1); ++h) si_reg[h] = __ldg(a.s + i * H + h);
  }
  const bool t_vec4 = HT && (HT % 4 == 0) && aligned_to_dev(a.t, 16);

  for (int64_t c0 = (int64_t)wsub * SE; c0 < d; c0 += (int64_t)W * SE) {
    const int ne = (int)((d - c0) < SE ? (d - c0) : SE);
    // A: logits, one lane per edge
    for (int k = lane; k < ne; k += 32) {
      const int j = __ldg(a.col + e0 + c0 + k);
      cols[k] = j - (int)joff;  // node id within its graph: the feature-row gathers of phase C
      const float* tj = a.t + (int64_t)j * H;
      if (HT) {
        float tv[HT ? HT : 1];
        if (t_vec4) {
#pragma unroll
          for (int q = 0; q < (HT ? HT : 1) / 4; ++q) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(tj) + q);
            tv[4 * q] = v.x; tv[4 * q + 1] = v.y; tv[4 * q + 2] = v.z; tv[4 * q + 3] = v.w;
          }
        } else {
#pragma unroll
          for (int h = 0; h < (HT ? HT : 1); ++h) tv[h] = __ldg(tj + h);
        }
#pragma unroll
        for (int h = 0; h < (HT ? HT : 1); ++h) {
          const float z = si_reg[h] + tv[h];
          float e = fmaxf(z, 0.f) + a.alpha * fminf(z, 0.f);  // LeakyReLU without a branch
          if (a.mode == GNN_GAT_EXPNEG) e = -e;
          logit[k * H + h] = e;
        }
      } else {
        const float* si = a.s + i * H;
#pragma unroll 4
        for (int h = 0; h < H; ++h) {
          const float z = __ldg(si + h) + __ldg(tj + h);
          float e = z > 0.f ? z : a.alpha * z;
          if (a.mode == GNN_GAT_EXPNEG) e = -e;
          logit[k * H + h] = e;
        }
      }
    }
    __syncwarp();
    // B: running per-head max
    if (a.mode == GNN_GAT_SOFTMAX) {
      float mx = -INFINITY;
      if (hsub < H)
        for (int k = g; k < ne; k += ngrp) mx = fmaxf(mx, logit[k * H + hsub]);
      for (int o = Hp; o < 32; o <<= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      if (lane < H) {
        const float mo = mh[lane];
        const float mn = fmaxf(mo, mx);
        const float f = (mo == -INFINITY) ? 0.f : __expf(mo - mn);
        sc[lane] = f;
        mh[lane] = mn;
        lh[lane] *= f;
      }
      __syncwarp();
#pragma unroll
      for (int c = 0; c < CPL; ++c) {
        const float f = sc[hc[c]];
        acc[c] *= f;
        l[c] *= f;
      }
    }
    // B2: logits -> un-normalised probabilities, one exp per (edge, head)
    if (HT) {
      // idx = lane + 32*j  =>  head = lane % HT for every j (HT divides 32)
      const float mymax = mh[hsub];
      float ps = 0.f;
      for (int idx = lane; idx < ne * H; idx += 32) {
        const float p = __expf(logit[idx] - mymax);
        ps += p;  // the row sum is taken before the dropout (softmax first, layers.py:30-31)
        float w = p;
        if (a.keep) w *= __ldg(a.keep + (e0 + c0) * H + idx);
        else if (seeded) w *= keep_factor(dseed, e0 + c0 + idx / (HT ? HT : 1), hsub, HT, thresh24, a.drop_scale);
        logit[idx] = w;
      }
      for (int o = Hp; o < 32; o <<= 1) ps += __shfl_xor_sync(0xffffffffu, ps, o);
      if (lane < H) lh[lane] += ps;
    } else {
      for (int idx = lane; idx < ne * H; idx += 32) logit[idx] = __expf(logit[idx] - mh[idx % H]);
    }
    __syncwarp();
    // C: weighted accumulation, one lane per output column, 8 row gathers in flight
    for (int k0 = 0; k0 < ne; k0 += 8) {
      typename RawOf<T>::type x[8][CPL / PK];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const bool ok = k0 + u < ne;
        const T* wr = reinterpret_cast<const T*>(a.Wh) + coff + (int64_t)(ok ? cols[k0 + u] : 0) * a.ldw;
#pragma unroll
        for (int q = 0; q < CPL / PK; ++q) x[u][q] = (ok && cv[q * PK]) ? ld_stage<T, PK>(wr, lane, q) : 0;
      }
      const float* pk = logit + k0 * H;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (k0 + u < ne) {
#pragma unroll
          for (int c = 0; c < CPL; ++c)
            if (cv[c]) {
              const float p = pk[u * H + hc[c]];
              float w = p;  // HT path: the dropout factor was folded into the staged weight in phase B2
              if (!HT) {
                l[c] += p;
                if (a.keep) w *= __ldg(a.keep + (e0 + c0 + k0 + u) * H + hc[c]);
                else if (seeded) w *= keep_factor(dseed, e0 + c0 + k0 + u, hc[c], H, thresh24, a.drop_scale);
              }
              acc[c] = fmaf(w, stage_elem<T, PK>(x[u][c / PK], c), acc[c]);
            }
        }
      }
    }
    __syncwarp();
  }
  if (HT) {
#pragma unroll
    for (int c = 0; c < CPL; ++c) l[c] = lh[hc[c]];
  }

  if (W == 1) {
#pragma unroll
    for (int c = 0; c < CPL; ++c)
      if (cv[c]) {
        const int ci = col_of<PK>(lane, c);
        const float v = acc[c] / l[c];
        stv(orow + ci, arow ? v : act_elu(v, a.elu));
        if (arow) stv(arow + ci, act_elu(v, a.elu));
        if (ci % a.Fp == 0) {
          if (a.row_max) a.row_max[i * H + hc[c]] = mh[hc[c]];
          if (a.row_sum) a.row_sum[i * H + hc[c]] = l[c];
        }
      }
    return;
  }
  // merge the warps' partial (max, sum, acc) in warp order
  if (lane < Hp) marr[warp * 32 + lane] = mh[lane];
#pragma unroll
  for (int c = 0; c < CPL; ++c) {
    larr[(warp * CPL + c) * 32 + lane] = l[c];
    aarr[(warp * CPL + c) * 32 + lane] = acc[c];
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int c = 0; c < CPL; ++c)
      if (cv[c]) {
        const int ci = col_of<PK>(lane, c);
        float M = -INFINITY;
        for (int w = 0; w < BW; ++w) M = fmaxf(M, marr[w * 32 + hc[c]]);
        float L = 0.f, A = 0.f;
        for (int w = 0; w < BW; ++w) {
          const float mw = marr[w * 32 + hc[c]];
          const float f = (mw == -INFINITY) ? 0.f : __expf(mw - M);
          L = fmaf(larr[(w * CPL + c) * 32 + lane], f, L);
          A = fmaf(aarr[(w * CPL + c) * 32 + lane], f, A);
        }
        const float v = A / L;
        stv(orow + ci, arow ? v : act_elu(v, a.elu));
        if (arow) stv(arow + ci, act_elu(v, a.elu));
        if (ci % a.Fp == 0) {
          if (a.row_max) a.row_max[i * H + hc[c]] = M;
          if (a.row_sum) a.row_sum[i * H + hc[c]] = L;
        }
      }
  }
}

__global__ void __launch_bounds__(256) gat_scores_kernel(const float* __restrict__ Wh, int64_t ldw,
                                                         const float* __restrict__ a_src,
                                                         const float* __restrict__ a_dst, int64_t n, int H, int Fp,
                                                         float* __restrict__ s, float* __restrict__ t) {
  const int64_t total = n * H;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
    const int h = (int)(p % H);
    const int64_t i = p / H;
    const float* w = Wh + i * ldw + h * Fp;
    float ss = 0.f, tt = 0.f;
    for (int f = 0; f < Fp; ++f) {
      const float x = __ldg(w + f);
      ss = fmaf(x, __ldg(a_src + h * Fp + f), ss);
      tt = fmaf(x, __ldg(a_dst + h * Fp + f), tt);
    }
    s[p] = ss;
    t[p] = tt;
  }
}

// ---- backward ------------------------------------------------------------------------------------
// Per-row statistics packed for the backward passes: rowstat[i] = [s_i | m_i | 1/l_i | D_i], H floats each, with
// D_i[h] = <d_out_i[h,:], out_pre_i[h,:]> (the softmax-Jacobian term).  One 128-byte record per node (H = 8): the
// transposed pass gathers it with one access per edge.
// When the forward applied its ELU(s) in the kernel epilogue (apply_elu > 0), d_out is the gradient w.r.t. the
// ACTIVATED output: the ELU derivative chain is applied here from the saved pre-activation (elu'(x) = 1 for x > 0,
// exp(x) otherwise; the second ELU is evaluated at elu(x)) and the pre-activation gradient is written to d_pre,
// which the two passes then gather — the activations' backward never runs as separate launches either.
template <typename T>
__global__ void __launch_bounds__(256) gat_rowstat_kernel(const T* __restrict__ d_out, const T* __restrict__ out_pre,
                                                          int64_t ldo, const float* __restrict__ s,
                                                          const float* __restrict__ row_max,
                                                          const float* __restrict__ row_sum, int64_t n, int H, int Fp,
                                                          float* __restrict__ rowstat, int apply_elu,
                                                          T* __restrict__ d_pre, int64_t batch_n) {
  const int64_t total = n * H;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
    const int h = (int)(p % H);
    const int64_t i = p / H;
    const int64_t gm = batch_n ? i / batch_n : 0;
    const int64_t fo = (i - gm * batch_n) * ldo + gm * (int64_t)H * Fp + h * Fp;  // (node row, graph's column block)
    const T* a = d_out + fo;
    const T* b = out_pre + fo;
    float acc = 0.f;
    for (int f = 0; f < Fp; ++f) {
      float g = ldv<T>(a + f);
      const float x = ldv<T>(b + f);
      if (apply_elu > 0) {
        if (apply_elu >= 2) {
          const float y1 = elu1(x);
          g *= y1 > 0.f ? 1.f : __expf(y1);
        }
        g *= x > 0.f ? 1.f : __expf(x);
        stv(d_pre + fo + f, g);
        g = round_as<T>(g);  // the passes read the ROUNDED value (bf16): keep D consistent with them
      }
      acc = fmaf(g, x, acc);
    }
    const float l = __ldg(row_sum + p);
    float* rs = rowstat + i * 4 * H;
    rs[h] = __ldg(s + p);
    rs[H + h] = __ldg(row_max + p);
    rs[2 * H + h] = l > 0.f ? 1.f / l : 0.f;
    rs[3 * H + h] = acc;
  }
}

// floats of shared memory per warp: w2 [SE*H], q [SE*H], (TR) w1 [SE*H], cols [SE]
// (at least HF: the finalize step reuses the warp's area as an [HF] scratch)
__host__ __device__ inline int gat_bwd_warp_floats(int SE, int H, int HF, bool tr) {
  const int f = (tr ? 3 : 2) * SE * H + SE;
  return f > HF ? f : HF;
}

// Both backward passes are the FORWARD kernel's shape — lane-per-edge weights staged in shared memory, then
// lane-per-column FMAs over coalesced row gathers — because the edge gradient factorises:
//     dz_ij = a_ij * slope_ij * (keep_ij * <dOut_i, Wh_j> - D_i)                 (per head)
//     d_s[i]  = sum_j dz_ij = <dOut_i, sum_j w2_ij Wh_j>  - D_i * sum_j a_ij slope_ij          (TR = false)
//     d_t[j]  = sum_i dz_ij = <Wh_j,  sum_i w2_ij dOut_i> -       sum_i a_ij slope_ij D_i      (TR = true)
//     d_Wh[j] =               sum_i w1_ij dOut_i                                               (TR = true)
// with w1 = keep*a, w2 = w1*slope.  No per-edge dot product (the first build reduced 64-wide dots by segmented
// shuffle for every edge: 71 warp instructions per edge, ncu r02), no per-edge stash between the passes (the first
// build wrote 64 bytes per edge and read them back: 6.9 GB each way on the Reddit shape), nothing but ordered sums.
//   TR = false: rows of the forward CSR (destination i); gathers Wh_j and t_j.
//   TR = true : rows of the transposed CSR (source j); gathers dOut_i and rowstat_i; `perm` maps its slots to the
//               forward edge slots for the dropout factors.
template <typename T, int CPL, int W, int HT, bool TR, int PK, bool RB = false>
__global__ void __launch_bounds__(GatBlock<W>::kWarps * 32) gat_bwd2_kernel(const GatArgs a) {
  constexpr int BW = GatBlock<W>::kWarps;
  constexpr int NA = TR ? 2 : 1;  // accumulators per column
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t r = (W == 1) ? (int64_t)blockIdx.x * kGatWarps + warp
                             : (a.row_list ? __ldg(a.row_list + blockIdx.x) : (int64_t)blockIdx.x);
  const int wsub = (W == 1) ? 0 : warp;
  if (W == 1 && r >= a.n) return;
  const int64_t e0 = __ldg(a.rowptr + r), e1 = __ldg(a.rowptr + r + 1);
  const int64_t d = e1 - e0;
  if (W == 1 && a.skip_deg_gt > 0 && d > a.skip_deg_gt) return;
  const int H = HT ? HT : a.H, Hp = HT ? HT : a.Hp, SE = a.SE, HF = a.HF, Fp = a.Fp;
  const int64_t gm = a.batch_n ? r / a.batch_n : 0;
  const int64_t joff = gm * (RB ? a.col_stride : a.batch_n);
  const int64_t roff = RB ? gm * a.batch_n : joff;
  const int64_t coff = gm * a.HF;
  const int PW = gat_bwd_warp_floats(SE, H, HF, TR);
  float* w2s = sm + (size_t)warp * PW;
  float* qs = w2s + SE * H;
  float* w1s = qs + SE * H;  // TR only
  int* cols = reinterpret_cast<int*>(w2s + (TR ? 3 : 2) * SE * H);
  float* qarr = sm + (size_t)BW * PW;           // [BW][32]
  float* aarr = qarr + BW * 32;                 // [BW][NA*CPL*32]

  int hc[CPL];
  bool cv[CPL];
  float acc2[CPL], acc1[CPL];
#pragma unroll
  for (int c = 0; c < CPL; ++c) {
    const int ci = col_of<PK>(lane, c);
    cv[c] = ci < HF;
    hc[c] = cv[c] ? ci / Fp : 0;
    acc2[c] = 0.f;
    acc1[c] = 0.f;
  }
  // constants of this row, per head, for the lane-per-edge phase
  float c0r[HT ? HT : 1], c1r[HT ? HT : 1], c2r[HT ? HT : 1];
  const float* rs_own = a.rowstat + r * 4 * H;
  if (HT) {
#pragma unroll
    for (int h = 0; h < (HT ? HT : 1); ++h) {
      if (TR) {
        c0r[h] = __ldg(a.t + r * H + h);
      } else {
        c0r[h] = __ldg(rs_own + h);
        c1r[h] = __ldg(rs_own + H + h);
        c2r[h] = __ldg(rs_own + 2 * H + h);
      }
    }
  }
  const bool vec4 = HT && (HT % 4 == 0) && aligned_to_dev(TR ? (const void*)a.rowstat : (const void*)a.t, 16);
  const bool seeded = a.keep == nullptr && a.keep_prob > 0.f;
  uint64_t dseed = seeded ? drop_seed_of(a) : 0;
  if (RB && seeded && a.slot_shift) dseed += (uint64_t)__ldg(a.slot_shift + gm) * (uint64_t)a.H * 0x9E3779B97F4A7C15ULL;
  const uint32_t thresh24 = (uint32_t)(a.keep_prob * 16777216.f);
  const int ngrp = 32 / Hp;
  const int hsub = lane % Hp, g = lane / Hp;
  float qsum = 0.f;

  for (int64_t c0 = (int64_t)wsub * SE; c0 < d; c0 += (int64_t)W * SE) {
    const int ne = (int)((d - c0) < SE ? (d - c0) : SE);
    // A: one lane per edge: attention weight, slope, the two FMA weights and the correction term, per head
    for (int k = lane; k < ne; k += 32) {
      const int64_t e = e0 + c0 + k;
      const int o = __ldg(a.col + e);
      cols[k] = o - (int)joff;  // node id within its graph (feature-row gathers); o itself indexes t / rowstat
      const float* ot = TR ? a.rowstat + (int64_t)o * 4 * H : a.t + (int64_t)o * H;
      const int64_t kslot = (TR && a.perm && (a.keep || seeded)) ? __ldg(a.perm + e) : e;  // forward edge slot
      if (HT) {
        float v0[HT ? HT : 1], v1[HT ? HT : 1], v2[HT ? HT : 1], v3[HT ? HT : 1];
        if (vec4) {
#pragma unroll
          for (int q = 0; q < (HT ? HT : 1) / 4; ++q) {
            const float4 x0 = __ldg(reinterpret_cast<const float4*>(ot) + q);
            v0[4 * q] = x0.x; v0[4 * q + 1] = x0.y; v0[4 * q + 2] = x0.z; v0[4 * q + 3] = x0.w;
            if (TR) {
              const float4 x1 = __ldg(reinterpret_cast<const float4*>(ot + H) + q);
              const float4 x2 = __ldg(reinterpret_cast<const float4*>(ot + 2 * H) + q);
              const float4 x3 = __ldg(reinterpret_cast<const float4*>(ot + 3 * H) + q);
              v1[4 * q] = x1.x; v1[4 * q + 1] = x1.y; v1[4 * q + 2] = x1.z; v1[4 * q + 3] = x1.w;
              v2[4 * q] = x2.x; v2[4 * q + 1] = x2.y; v2[4 * q + 2] = x2.z; v2[4 * q + 3] = x2.w;
              v3[4 * q] = x3.x; v3[4 * q + 1] = x3.y; v3[4 * q + 2] = x3.z; v3[4 * q + 3] = x3.w;
            }
          }
        } else {
#pragma unroll
          for (int h = 0; h < (HT ? HT : 1); ++h) {
            v0[h] = __ldg(ot + h);
            if (TR) {
              v1[h] = __ldg(ot + H + h);
              v2[h] = __ldg(ot + 2 * H + h);
              v3[h] = __ldg(ot + 3 * H + h);
            }
          }
        }
#pragma unroll
        for (int h = 0; h < (HT ? HT : 1); ++h) {
          const float z = c0r[h] + v0[h];  // s_i + t_j either way
          const float m = TR ? v1[h] : c1r[h];
          const float li = TR ? v2[h] : c2r[h];
          float slope = z > 0.f ? 1.f : a.alpha;
          float ee = z * slope;
          if (a.mode == GNN_GAT_EXPNEG) {
            ee = -ee;
            slope = -slope;
          }
          const float al = __expf(ee - m) * li;
          const float kp = a.keep ? __ldg(a.keep + kslot * H + h)
                                  : (seeded ? keep_factor(dseed, kslot, h, H, thresh24, a.drop_scale) : 1.f);
          const float w1 = kp * al;
          w2s[k * H + h] = w1 * slope;
          if (TR) w1s[k * H + h] = w1;
          qs[k * H + h] = TR ? al * slope * v3[h] : al * slope;
        }
      } else {
        for (int h = 0; h < H; ++h) {
          const float z = TR ? __ldg(ot + h) + __ldg(a.t + r * H + h) : __ldg(rs_own + h) + __ldg(ot + h);
          const float m = TR ? __ldg(ot + H + h) : __ldg(rs_own + H + h);
          const float li = TR ? __ldg(ot + 2 * H + h) : __ldg(rs_own + 2 * H + h);
          float slope = z > 0.f ? 1.f : a.alpha;
          float ee = z * slope;
          if (a.mode == GNN_GAT_EXPNEG) {
            ee = -ee;
            slope = -slope;
          }
          const float al = __expf(ee - m) * li;
          const float kp = a.keep ? __ldg(a.keep + kslot * H + h)
                                  : (seeded ? keep_factor(dseed, kslot, h, H, thresh24, a.drop_scale) : 1.f);
          const float w1 = kp * al;
          w2s[k * H + h] = w1 * slope;
          if (TR) w1s[k * H + h] = w1;
          qs[k * H + h] = TR ? al * slope * __ldg(ot + 3 * H + h) : al * slope;
        }
      }
    }
    __syncwarp();
    // Q: per-head sum of the correction terms of this chunk (fixed lane -> edge assignment: deterministic)
    if (hsub < H)
      for (int k = g; k < ne; k += ngrp) qsum += qs[k * H + hsub];
    // C: one lane per column, 8 row gathers in flight
    const T* base = reinterpret_cast<const T*>(TR ? a.d_out : a.Wh) + coff;
    const int64_t ldb = TR ? a.ldo : a.ldw;
    for (int k0 = 0; k0 < ne; k0 += 8) {
      typename RawOf<T>::type x[8][CPL / PK];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const bool ok = k0 + u < ne;
        const T* xr = base + (int64_t)(ok ? cols[k0 + u] : 0) * ldb;
#pragma unroll
        for (int q = 0; q < CPL / PK; ++q) x[u][q] = (ok && cv[q * PK]) ? ld_stage<T, PK>(xr, lane, q) : 0;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        if (k0 + u < ne) {
#pragma unroll
          for (int c = 0; c < CPL; ++c)
            if (cv[c]) {
              const float xv = stage_elem<T, PK>(x[u][c / PK], c);
              acc2[c] = fmaf(w2s[(k0 + u) * H + hc[c]], xv, acc2[c]);
              if (TR) acc1[c] = fmaf(w1s[(k0 + u) * H + hc[c]], xv, acc1[c]);
            }
        }
      }
    }
    __syncwarp();
  }
  for (int o = Hp; o < 32; o <<= 1) qsum += __shfl_xor_sync(0xffffffffu, qsum, o);

  if (W > 1) {
    // merge the warps' partials in warp order
    if (lane < Hp) qarr[warp * 32 + lane] = qsum;
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
      aarr[(warp * NA * CPL + c) * 32 + lane] = acc2[c];
      if (TR) aarr[(warp * NA * CPL + CPL + c) * 32 + lane] = acc1[c];
    }
    __syncthreads();
    if (warp != 0) return;
    qsum = 0.f;
    if (lane < Hp)
      for (int w = 0; w < BW; ++w) qsum += qarr[w * 32 + lane];
#pragma unroll
    for (int c = 0; c < CPL; ++c) {
      float t2 = 0.f, t1 = 0.f;
      for (int w = 0; w < BW; ++w) {
        t2 += aarr[(w * NA * CPL + c) * 32 + lane];
        if (TR) t1 += aarr[(w * NA * CPL + CPL + c) * 32 + lane];
      }
      acc2[c] = t2;
      acc1[c] = t1;
    }
  }
  // finalize (one warp): the head-wise contraction of the accumulated vector with this row's own vector
  float* buf = w2s;  // [HF] scratch (this warp's staging area is free now)
  __syncwarp();
  const T* own = reinterpret_cast<const T*>(TR ? a.Wh : a.d_out) + (r - roff) * (TR ? a.ldw : a.ldo) + coff;
#pragma unroll
  for (int c = 0; c < CPL; ++c)
    if (cv[c]) {
      const int ci = col_of<PK>(lane, c);
      buf[ci] = acc2[c] * ldv<T>(own + ci);
      if (TR) stv(reinterpret_cast<T*>(a.d_Wh) + (r - roff) * a.ld_dwh + coff + ci, acc1[c]);
    }
  __syncwarp();
  if (lane < H) {
    float tot = 0.f;
    for (int f = 0; f < Fp; ++f) tot += buf[lane * Fp + f];
    if (TR) a.d_t[r * H + lane] = tot - qsum;
    else a.d_s[r * H + lane] = tot - __ldg(rs_own + 3 * H + lane) * qsum;
  }
}

inline int next_pow2(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

int check_common(int64_t n, int H, int Fp) {
  GNN_REQUIRE(n >= 0 && H > 0 && Fp > 0, GNN_ERR_BAD_ARG, "bad size (n=%lld H=%d Fp=%d)", (long long)n, H, Fp);
  GNN_REQUIRE(H <= 32, GNN_ERR_UNSUPPORTED, "more than 32 heads per call (H=%d): split the heads", H);
  GNN_REQUIRE(H * Fp <= 256, GNN_ERR_UNSUPPORTED, "H*Fp=%d exceeds 256 columns per call: split the heads", H * Fp);
  GNN_REQUIRE(n < 0x7fffffffLL, GNN_ERR_UNSUPPORTED, "n does not fit int32");
  return GNN_OK;
}

int stage_edges(int H) {
  int se = tuning("gat.stage_edges", 128);
  while (se > 32 && se * H > 1024) se >>= 1;
  return se < 32 ? 32 : se;
}

// one CTA per row for every row when rows are long on average (dense metapath adjacencies);
// otherwise one warp per row, and only the rows of the caller's long-row list get a CTA
bool cooperative(int64_t n, int64_t nnz) {
  const int thr = tuning("gat.coop_min_avg_deg", 256);
  return n > 0 && nnz > 0 && nnz / n >= thr;
}

template <int W>
size_t gat_smem_bytes(int SE, int H, int HF, int cpl) {
  constexpr int BW = GatBlock<W>::kWarps;
  size_t f = (size_t)BW * gat_warp_floats(SE, H, HF);
  if (W > 1) f += (size_t)BW * 32 + 2 * (size_t)BW * cpl * 32;
  return f * sizeof(float);
}

// forward launch: picks the compile-time head count when there is one
template <typename T, int CPL, int W, bool RB>
int gat_fwd_launch(const GatArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
  constexpr int thr = GatBlock<W>::kWarps * 32;
#define GNN_GAT_FWD_PK(HT, PKV)                                                                                 \
  do {                                                                                                          \
    if (smem > 48 * 1024)                                                                                       \
      GNN_CUDA(cudaFuncSetAttribute(gat_fwd_kernel<T, CPL, W, HT, PKV, RB>,                                     \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                   \
    gat_fwd_kernel<T, CPL, W, HT, PKV, RB><<<grid, thr, smem, st>>>(a);                                         \
  } while (0)
#define GNN_GAT_FWD(HT)                                              \
  do {                                                               \
    if constexpr (sizeof(T) == 2 && CPL >= 2) {                      \
      if (a.packed) GNN_GAT_FWD_PK(HT, 2);                           \
      else GNN_GAT_FWD_PK(HT, 1);                                    \
    } else {                                                         \
      GNN_GAT_FWD_PK(HT, 1);                                         \
    }                                                                \
  } while (0)
  if (a.H == 8) GNN_GAT_FWD(8);
  else if (a.H == 1) GNN_GAT_FWD(1);
  else GNN_GAT_FWD(0);
#undef GNN_GAT_FWD
#undef GNN_GAT_FWD_PK
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

template <typename T, int W, bool RB>
int gat_fwd_dispatch(const GatArgs& a, int cpl, unsigned grid, cudaStream_t st) {
  int cplr = cpl <= 1 ? 1 : cpl <= 2 ? 2 : cpl <= 4 ? 4 : 8;
  if (a.packed && cplr < 2) cplr = 2;  // a packed lane owns column pairs
  const size_t smem = gat_smem_bytes<W>(a.SE, a.H, a.HF, cplr);
  switch (cplr) {
    case 1: return gat_fwd_launch<T, 1, W, RB>(a, grid, smem, st);
    case 2: return gat_fwd_launch<T, 2, W, RB>(a, grid, smem, st);
    case 4: return gat_fwd_launch<T, 4, W, RB>(a, grid, smem, st);
    default: return gat_fwd_launch<T, 8, W, RB>(a, grid, smem, st);
  }
}

// struct_size is the version of gnn_gat_dropout: the current size, or the size before edge_slot_base was appended
// (read as base 0); any other size is refused.  a.H must be set.
inline int set_dropout(GatArgs& a, const float* edge_keep, const gnn_gat_dropout* d) {
  a.keep = edge_keep;
  if (d && d->p > 0.f) {
    const bool cur = d->struct_size == (int32_t)sizeof(gnn_gat_dropout);
    GNN_REQUIRE(cur || d->struct_size == (int32_t)offsetof(gnn_gat_dropout, edge_slot_base), GNN_ERR_BAD_ARG,
                "gnn_gat_dropout struct_size mismatch (header/library version skew)");
    const int64_t base = cur ? d->edge_slot_base : 0;
    GNN_REQUIRE(base >= 0, GNN_ERR_BAD_ARG, "negative edge_slot_base");
    GNN_REQUIRE(base == 0 || !d->seed_dev, GNN_ERR_UNSUPPORTED,
                "edge_slot_base needs the whole seed on the host (seed_dev = NULL)");
    GNN_REQUIRE(d->p < 1.f, GNN_ERR_BAD_ARG, "dropout probability must be below 1");
    GNN_REQUIRE(!edge_keep, GNN_ERR_BAD_ARG, "give either an explicit keep mask or a seeded dropout, not both");
    a.keep_prob = 1.f - d->p;
    a.drop_scale = 1.f / a.keep_prob;
    // keep_factor hashes seed + (e*H + h + 1)*golden: slot e + base is slot e under seed + base*H*golden (mod 2^64),
    // so the base is folded into the seed here and the kernels are unchanged
    a.drop_seed = d->seed + (uint64_t)base * (uint64_t)a.H * 0x9E3779B97F4A7C15ULL;
    a.drop_seed_dev = d->seed_dev;
  }
  return GNN_OK;
}

// cooperative, or the listed hub rows first and then one warp per row
template <typename T, bool RB>
int gat_fwd_schedule(GatArgs& a, int cpl, int64_t n, int64_t nnz, const int64_t* long_rows, int64_t n_long,
                     int64_t long_threshold, cudaStream_t st) {
  if (cooperative(n, nnz)) return gat_fwd_dispatch<T, kGatWarps, RB>(a, cpl, (unsigned)n, st);
  if (n_long > 0) {  // hub rows: one 16-warp CTA each, launched first so the short rows fill in behind
    a.row_list = long_rows;
    int rc = gat_fwd_dispatch<T, 16, RB>(a, cpl, (unsigned)n_long, st);
    if (rc != GNN_OK) return rc;
    a.row_list = nullptr;
    a.skip_deg_gt = long_threshold;
  }
  return gat_fwd_dispatch<T, 1, RB>(a, cpl, (unsigned)((n + kGatWarps - 1) / kGatWarps), st);
}

template <typename T>
int gat_fwd_impl(const int64_t* rowptr, const int32_t* col, const T* Wh, int64_t ldw, const float* s, const float* t,
                 int64_t n, int64_t nnz, int32_t H, int32_t Fp, float alpha, int mode, int apply_elu,
                 const float* col_mean, const float* edge_keep, T* out, int64_t ldo, float* row_max, float* row_sum,
                 const int64_t* long_rows, int64_t n_long, int64_t long_threshold, cudaStream_t st,
                 T* out_act = nullptr, const gnn_gat_dropout* drop = nullptr, int64_t batch_nodes = 0,
                 const gnn_gat_batch* rb = nullptr) {
  int rc = check_common(n, H, Fp);
  if (rc != GNN_OK) return rc;
  if (n == 0) return GNN_OK;
  GNN_REQUIRE(rowptr && Wh && s && t && out, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(mode == GNN_GAT_SOFTMAX || mode == GNN_GAT_EXPNEG, GNN_ERR_BAD_ARG, "unknown mode %d", mode);
  GNN_REQUIRE(apply_elu >= 0 && apply_elu <= 2, GNN_ERR_BAD_ARG, "apply_elu must be 0, 1 or 2");
  const int HF = H * Fp;
  GNN_REQUIRE(batch_nodes >= 0 && (batch_nodes == 0 || n % batch_nodes == 0), GNN_ERR_BAD_ARG,
              "batch_nodes must divide the batched row count");
  const int64_t n_graphs = batch_nodes ? n / batch_nodes : 1;
  GNN_REQUIRE(ldw >= n_graphs * HF && ldo >= n_graphs * HF, GNN_ERR_BAD_ARG,
              "leading dimension smaller than (graphs x) H*Fp");
  GatArgs a{};
  a.batch_n = batch_nodes;
  a.rowptr = rowptr;
  a.col = col;
  a.Wh = Wh;
  a.ldw = ldw;
  a.s = s;
  a.t = t;
  a.n = n;
  a.H = H;
  a.Hp = next_pow2(H);
  a.Fp = Fp;
  a.HF = HF;
  a.alpha = alpha;
  a.mode = mode;
  a.elu = apply_elu;
  a.col_mean = col_mean;
  rc = set_dropout(a, edge_keep, drop);
  if (rc != GNN_OK) return rc;
  a.out = out;
  a.out_act = out_act;
  a.ldo = ldo;
  a.row_max = row_max;
  a.row_sum = row_sum;
  a.SE = stage_edges(H);
  a.packed = sizeof(T) == 2 && Fp % 2 == 0 && ldw % 2 == 0 && aligned_to(Wh, 4);
  const int cpl = (HF + 31) / 32;
  GNN_REQUIRE(n_long == 0 || (long_rows && long_threshold > 0), GNN_ERR_BAD_ARG, "inconsistent long-row list");
  if (rb) {
    // packed bf16 (PK = 2): graph gm's columns start at gm * HF (even, since Fp is) and its rows move by whole
    // rows of even ldw / ldo, so every staged 32-bit word stays 4-byte aligned under the RB offsets
    a.col_stride = rb->cols_per_graph;
    a.slot_shift = rb->slot_shift;
    return gat_fwd_schedule<T, true>(a, cpl, n, nnz, long_rows, n_long, long_threshold, st);
  }
  return gat_fwd_schedule<T, false>(a, cpl, n, nnz, long_rows, n_long, long_threshold, st);
}

template <typename T, int CPLV, int WV, bool TR, bool RB>
int gat_bwd2_launch(const GatArgs& a, unsigned grid, cudaStream_t st) {
  constexpr int BW = GatBlock<WV>::kWarps;
  size_t f = (size_t)BW * gat_bwd_warp_floats(a.SE, a.H, a.HF, TR);
  if (WV > 1) f += (size_t)BW * 32 + (size_t)BW * (TR ? 2 : 1) * CPLV * 32;
  const size_t smem = f * sizeof(float);
  constexpr int thrv = BW * 32;
#define GNN_BWD2_PK(HTV, PKV)                                                                                  \
  do {                                                                                                         \
    if (smem > 48 * 1024)                                                                                      \
      GNN_CUDA(cudaFuncSetAttribute(gat_bwd2_kernel<T, CPLV, WV, HTV, TR, PKV, RB>,                            \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                  \
    gat_bwd2_kernel<T, CPLV, WV, HTV, TR, PKV, RB><<<grid, thrv, smem, st>>>(a);                               \
  } while (0)
#define GNN_BWD2(HTV)                                                \
  do {                                                               \
    if constexpr (sizeof(T) == 2 && CPLV >= 2) {                     \
      if (a.packed) GNN_BWD2_PK(HTV, 2);                             \
      else GNN_BWD2_PK(HTV, 1);                                      \
    } else {                                                         \
      GNN_BWD2_PK(HTV, 1);                                           \
    }                                                                \
  } while (0)
  if (a.H == 8) GNN_BWD2(8);
  else if (a.H == 1) GNN_BWD2(1);
  else GNN_BWD2(0);
#undef GNN_BWD2
#undef GNN_BWD2_PK
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

template <typename T, int WV, bool TR, bool RB>
int gat_bwd2_dispatch(const GatArgs& a, int cplr, unsigned grid, cudaStream_t st) {
  switch (cplr) {
    case 1: return gat_bwd2_launch<T, 1, WV, TR, RB>(a, grid, st);
    case 2: return gat_bwd2_launch<T, 2, WV, TR, RB>(a, grid, st);
    case 4: return gat_bwd2_launch<T, 4, WV, TR, RB>(a, grid, st);
    default: return gat_bwd2_launch<T, 8, WV, TR, RB>(a, grid, st);
  }
}

// pass 1 over the forward CSR (d_s), then pass 2 over the transposed CSR (d_Wh, d_t).  W: 1 warp per row, 4 = every
// row a CTA (dense graphs), 16 = listed hub rows.  a.rowptr / a.col hold the forward CSR on entry.
template <typename T, bool RB>
int gat_bwd_passes(GatArgs& a, int cplr, int64_t n, int64_t n_cols, int64_t nnz, const int64_t* rowptr_t,
                   const int32_t* col_t, const int64_t* perm_t, const int64_t* long_rows, int64_t n_long,
                   const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold, cudaStream_t st) {
  int rc;
  // the row-record kernel and pass 1 walk the n forward rows; pass 2 the n_cols table rows (its own schedule)
  const bool coop = cooperative(n, nnz), coop_t = cooperative(n_cols, nnz);
  const unsigned grid1 = (unsigned)((n + kGatWarps - 1) / kGatWarps);
  const unsigned grid1_t = (unsigned)((n_cols + kGatWarps - 1) / kGatWarps);
  if (n == 0) {
    // no forward row: the table rows get zero gradients from pass 2 (every transposed row is empty)
  } else if (coop) {
    rc = gat_bwd2_dispatch<T, 4, false, RB>(a, cplr, (unsigned)n, st);
    if (rc != GNN_OK) return rc;
  } else {
    if (n_long > 0) {
      a.row_list = long_rows;
      rc = gat_bwd2_dispatch<T, 16, false, RB>(a, cplr, (unsigned)n_long, st);
      if (rc != GNN_OK) return rc;
      a.row_list = nullptr;
      a.skip_deg_gt = long_threshold;
    }
    rc = gat_bwd2_dispatch<T, 1, false, RB>(a, cplr, grid1, st);
    if (rc != GNN_OK) return rc;
  }
  a.rowptr = rowptr_t;
  a.col = col_t;
  a.perm = perm_t;
  a.n = n_cols;
  a.row_list = nullptr;
  a.skip_deg_gt = 0;
  if (RB) {  // transposed rows are table rows (per graph: col_stride of them); their ids are forward rows
    const int64_t rows = a.batch_n;
    a.batch_n = a.col_stride;
    a.col_stride = rows;
  }
  if (coop_t) return gat_bwd2_dispatch<T, 4, true, RB>(a, cplr, (unsigned)n_cols, st);
  if (n_long_t > 0) {
    a.row_list = long_rows_t;
    rc = gat_bwd2_dispatch<T, 16, true, RB>(a, cplr, (unsigned)n_long_t, st);
    if (rc != GNN_OK) return rc;
    a.row_list = nullptr;
    a.skip_deg_gt = long_threshold;
  }
  return gat_bwd2_dispatch<T, 1, true, RB>(a, cplr, grid1_t, st);
}

template <typename T>
int gat_bwd_impl(const int64_t* rowptr, const int32_t* col, const int64_t* rowptr_t, const int32_t* col_t,
                 const int64_t* perm_t, const T* Wh, int64_t ldw, const float* s, const float* t, const float* row_max,
                 const float* row_sum, const T* out_pre, const T* d_out, int64_t ldo, int64_t n, int64_t n_cols,
                 int32_t H, int32_t Fp,
                 float alpha, int mode, const float* edge_keep, T* d_Wh, int64_t ld_dwh, float* d_s, float* d_t,
                 float* row_scratch, int64_t nnz, const int64_t* long_rows, int64_t n_long, const int64_t* long_rows_t,
                 int64_t n_long_t, int64_t long_threshold, cudaStream_t st, int apply_elu = 0, T* d_pre = nullptr,
                 const gnn_gat_dropout* drop = nullptr, int64_t batch_nodes = 0,
                 const gnn_gat_batch* rb = nullptr) {
  int rc = check_common(n, H, Fp);
  if (rc != GNN_OK) return rc;
  rc = check_common(n_cols, H, Fp);
  if (rc != GNN_OK) return rc;
  GNN_REQUIRE(n_cols >= n, GNN_ERR_BAD_ARG, "n_cols (%lld) below the forward row count (%lld)", (long long)n_cols,
              (long long)n);
  GNN_REQUIRE(n_cols == n || batch_nodes == 0 || rb, GNN_ERR_UNSUPPORTED, "batched graphs are square (n_cols == n)");
  if (n == 0 && n_cols == 0) return GNN_OK;
  GNN_REQUIRE(rowptr && rowptr_t && Wh && s && t && row_max && row_sum && out_pre && d_out && d_Wh && d_s && d_t &&
                  row_scratch,
              GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(nnz >= 0 && (nnz == 0 || (col && col_t)), GNN_ERR_BAD_ARG, "null edge pointer (col/col_t)");
  GNN_REQUIRE(!(edge_keep || (drop && drop->p > 0.f)) || perm_t || nnz == 0, GNN_ERR_BAD_ARG,
              "attention dropout needs perm_t (transposed slot -> forward edge slot)");
  GNN_REQUIRE(apply_elu >= 0 && apply_elu <= 2 && (apply_elu == 0 || d_pre), GNN_ERR_BAD_ARG,
              "apply_elu must be 0..2 and needs the d_pre scratch when > 0");
  GNN_REQUIRE(mode == GNN_GAT_SOFTMAX || mode == GNN_GAT_EXPNEG, GNN_ERR_BAD_ARG, "unknown mode %d", mode);
  const int HF = H * Fp;
  GNN_REQUIRE(batch_nodes >= 0 && (batch_nodes == 0 || n % batch_nodes == 0), GNN_ERR_BAD_ARG,
              "batch_nodes must divide the batched row count");
  const int64_t n_graphs = batch_nodes ? n / batch_nodes : 1;
  GNN_REQUIRE(ldw >= n_graphs * HF && ldo >= n_graphs * HF && ld_dwh >= n_graphs * HF, GNN_ERR_BAD_ARG,
              "leading dimension smaller than (graphs x) H*Fp");
  GatArgs a{};
  a.batch_n = batch_nodes;
  a.Wh = Wh;
  a.ldw = ldw;
  a.s = s;
  a.t = t;
  a.n = n;
  a.H = H;
  a.Hp = next_pow2(H);
  a.Fp = Fp;
  a.HF = HF;
  a.alpha = alpha;
  a.mode = mode;
  rc = set_dropout(a, edge_keep, drop);
  if (rc != GNN_OK) return rc;
  a.ldo = ldo;
  a.SE = tuning("gat.bwd_stage_edges", 64);
  while (a.SE > 32 && a.SE * H > 1024) a.SE >>= 1;
  a.out_pre = out_pre;
  a.d_out = apply_elu > 0 ? d_pre : d_out;  // the passes gather the PRE-activation gradient
  a.rowstat = row_scratch;
  a.d_Wh = d_Wh;
  a.ld_dwh = ld_dwh;
  a.d_s = d_s;
  a.d_t = d_t;
  if (n > 0) {
    int64_t grid = (n * H + 255) / 256;
    const int64_t cap = (int64_t)num_sms() * 16;
    grid = grid > cap ? cap : grid;
    gat_rowstat_kernel<T><<<(unsigned)grid, 256, 0, st>>>(d_out, out_pre, ldo, s, row_max, row_sum, n, H, Fp,
                                                         row_scratch, apply_elu, d_pre, batch_nodes);
    GNN_LAUNCH_CHECK();
  }
  a.packed = sizeof(T) == 2 && Fp % 2 == 0 && ldw % 2 == 0 && ldo % 2 == 0 && aligned_to(Wh, 4) &&
             aligned_to(a.d_out, 4);
  const int cpl = (HF + 31) / 32;
  int cplr = cpl <= 1 ? 1 : cpl <= 2 ? 2 : cpl <= 4 ? 4 : 8;
  if (a.packed && cplr < 2) cplr = 2;
  GNN_REQUIRE((n_long == 0 || long_rows) && (n_long_t == 0 || long_rows_t) &&
                  ((n_long == 0 && n_long_t == 0) || long_threshold > 0),
              GNN_ERR_BAD_ARG, "inconsistent long-row lists");
  a.rowptr = rowptr;
  a.col = col;
  if (rb) {
    a.col_stride = rb->cols_per_graph;
    a.slot_shift = rb->slot_shift;
    return gat_bwd_passes<T, true>(a, cplr, n, n_cols, nnz, rowptr_t, col_t, perm_t, long_rows, n_long, long_rows_t,
                                   n_long_t, long_threshold, st);
  }
  return gat_bwd_passes<T, false>(a, cplr, n, n_cols, nnz, rowptr_t, col_t, perm_t, long_rows, n_long, long_rows_t,
                                  n_long_t, long_threshold, st);
}

// the batched-rectangular description: n_rows / n_cols are the launch's forward rows and table rows
int check_batch(const gnn_gat_batch* b, int64_t* n_rows, int64_t* n_cols) {
  GNN_REQUIRE(b, GNN_ERR_BAD_ARG, "null gnn_gat_batch");
  GNN_REQUIRE(b->struct_size == (int32_t)sizeof(gnn_gat_batch), GNN_ERR_BAD_ARG,
              "gnn_gat_batch struct_size mismatch (header/library version skew)");
  GNN_REQUIRE(b->n_graphs >= 1 && b->n_graphs <= 32, GNN_ERR_UNSUPPORTED, "n_graphs=%d outside 1..32", b->n_graphs);
  GNN_REQUIRE(b->rows_per_graph >= 0 && b->cols_per_graph >= b->rows_per_graph, GNN_ERR_BAD_ARG,
              "need 0 <= rows_per_graph <= cols_per_graph (got %lld, %lld)", (long long)b->rows_per_graph,
              (long long)b->cols_per_graph);
  GNN_REQUIRE(b->cols_per_graph * b->n_graphs < 0x7fffffffLL, GNN_ERR_UNSUPPORTED, "column ids do not fit int32");
  *n_rows = b->rows_per_graph * b->n_graphs;
  *n_cols = b->cols_per_graph * b->n_graphs;
  return GNN_OK;
}

}  // namespace

extern "C" {

int gnn_gat_scores_f32(const float* Wh, int64_t ldw, const float* a_src, const float* a_dst, int64_t n, int32_t H,
                       int32_t Fp, float* s, float* t, gnn_stream_t stream) {
  int rc = check_common(n, H, Fp);
  if (rc != GNN_OK) return rc;
  if (n == 0) return GNN_OK;
  GNN_REQUIRE(Wh && a_src && a_dst && s && t, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(ldw >= (int64_t)H * Fp, GNN_ERR_BAD_ARG, "ldw smaller than H*Fp");
  int64_t grid = (n * H + 255) / 256;
  const int64_t cap = (int64_t)num_sms() * 16;
  grid = grid > cap ? cap : grid;
  gat_scores_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(Wh, ldw, a_src, a_dst, n, H, Fp, s, t);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_gat_fused_fwd_f32(const int64_t* rowptr, const int32_t* col, const float* Wh, int64_t ldw, const float* s,
                          const float* t, int64_t n, int64_t nnz, int32_t H, int32_t Fp, float alpha, int mode,
                          int apply_elu, const float* col_mean, const float* edge_keep, float* out, int64_t ldo,
                          float* row_max, float* row_sum, const int64_t* long_rows, int64_t n_long,
                          int64_t long_threshold, int64_t batch_nodes, gnn_stream_t stream) {
  return gat_fwd_impl<float>(rowptr, col, Wh, ldw, s, t, n, nnz, H, Fp, alpha, mode, apply_elu, col_mean, edge_keep, out,
                             ldo, row_max, row_sum, long_rows, n_long, long_threshold, (cudaStream_t)stream, nullptr,
                             nullptr, batch_nodes);
}

int gnn_gat_fused_fwd_bf16(const int64_t* rowptr, const int32_t* col, const void* Wh, int64_t ldw, const float* s,
                           const float* t, int64_t n, int64_t nnz, int32_t H, int32_t Fp, float alpha, int mode,
                           int apply_elu, const float* col_mean, const float* edge_keep, void* out, int64_t ldo,
                           float* row_max, float* row_sum, const int64_t* long_rows, int64_t n_long,
                           int64_t long_threshold, int64_t batch_nodes, gnn_stream_t stream) {
  return gat_fwd_impl<__nv_bfloat16>(rowptr, col, (const __nv_bfloat16*)Wh, ldw, s, t, n, nnz, H, Fp, alpha, mode,
                                     apply_elu, col_mean, edge_keep, (__nv_bfloat16*)out, ldo, row_max, row_sum,
                                     long_rows, n_long, long_threshold, (cudaStream_t)stream, nullptr, nullptr,
                                     batch_nodes);
}

int gnn_gat_fused_fwd_train_f32(const int64_t* rowptr, const int32_t* col, const float* Wh, int64_t ldw,
                                const float* s, const float* t, int64_t n, int64_t nnz, int32_t H, int32_t Fp,
                                float alpha, int mode, int apply_elu, const float* col_mean, const float* edge_keep,
                                const gnn_gat_dropout* dropout, float* out_pre, float* out_act, int64_t ldo,
                                float* row_max, float* row_sum, const int64_t* long_rows, int64_t n_long,
                                int64_t long_threshold, int64_t batch_nodes, gnn_stream_t stream) {
  GNN_REQUIRE(out_act || apply_elu == 0, GNN_ERR_BAD_ARG, "apply_elu > 0 needs out_act");
  return gat_fwd_impl<float>(rowptr, col, Wh, ldw, s, t, n, nnz, H, Fp, alpha, mode, apply_elu, col_mean, edge_keep,
                             out_pre, ldo, row_max, row_sum, long_rows, n_long, long_threshold, (cudaStream_t)stream,
                             apply_elu > 0 ? out_act : nullptr, dropout, batch_nodes);
}

int gnn_gat_fused_fwd_train_bf16(const int64_t* rowptr, const int32_t* col, const void* Wh, int64_t ldw,
                                 const float* s, const float* t, int64_t n, int64_t nnz, int32_t H, int32_t Fp,
                                 float alpha, int mode, int apply_elu, const float* col_mean, const float* edge_keep,
                                 const gnn_gat_dropout* dropout, void* out_pre, void* out_act, int64_t ldo,
                                 float* row_max, float* row_sum, const int64_t* long_rows, int64_t n_long,
                                 int64_t long_threshold, int64_t batch_nodes, gnn_stream_t stream) {
  GNN_REQUIRE(out_act || apply_elu == 0, GNN_ERR_BAD_ARG, "apply_elu > 0 needs out_act");
  return gat_fwd_impl<__nv_bfloat16>(rowptr, col, (const __nv_bfloat16*)Wh, ldw, s, t, n, nnz, H, Fp, alpha, mode,
                                     apply_elu, col_mean, edge_keep, (__nv_bfloat16*)out_pre, ldo, row_max, row_sum,
                                     long_rows, n_long, long_threshold, (cudaStream_t)stream,
                                     apply_elu > 0 ? (__nv_bfloat16*)out_act : nullptr, dropout, batch_nodes);
}

int gnn_gat_fused_bwd_f32(const int64_t* rowptr, const int32_t* col, const int64_t* rowptr_t, const int32_t* col_t,
                          const int64_t* perm_t, const float* Wh, int64_t ldw, const float* s, const float* t,
                          const float* row_max, const float* row_sum, const float* out_pre, const float* d_out,
                          int64_t ldo, int64_t n, int32_t H, int32_t Fp, float alpha, int mode,
                          const float* edge_keep, float* d_Wh, int64_t ld_dwh, float* d_s, float* d_t,
                          float* row_scratch, int64_t nnz, const int64_t* long_rows, int64_t n_long,
                          const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold, int apply_elu,
                          float* d_pre, const gnn_gat_dropout* dropout, int64_t batch_nodes, gnn_stream_t stream) {
  return gat_bwd_impl<float>(rowptr, col, rowptr_t, col_t, perm_t, Wh, ldw, s, t, row_max, row_sum, out_pre, d_out, ldo,
                             n, n, H, Fp, alpha, mode, edge_keep, d_Wh, ld_dwh, d_s, d_t, row_scratch, nnz, long_rows,
                             n_long, long_rows_t, n_long_t, long_threshold, (cudaStream_t)stream, apply_elu, d_pre,
                             dropout, batch_nodes);
}

int gnn_gat_fused_bwd_bf16(const int64_t* rowptr, const int32_t* col, const int64_t* rowptr_t, const int32_t* col_t,
                           const int64_t* perm_t, const void* Wh, int64_t ldw, const float* s, const float* t,
                           const float* row_max, const float* row_sum, const void* out_pre, const void* d_out,
                           int64_t ldo, int64_t n, int32_t H, int32_t Fp, float alpha, int mode,
                           const float* edge_keep, void* d_Wh, int64_t ld_dwh, float* d_s, float* d_t,
                           float* row_scratch, int64_t nnz, const int64_t* long_rows, int64_t n_long,
                           const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold, int apply_elu,
                           void* d_pre, const gnn_gat_dropout* dropout, int64_t batch_nodes, gnn_stream_t stream) {
  return gat_bwd_impl<__nv_bfloat16>(rowptr, col, rowptr_t, col_t, perm_t, (const __nv_bfloat16*)Wh, ldw, s, t, row_max,
                                     row_sum, (const __nv_bfloat16*)out_pre, (const __nv_bfloat16*)d_out, ldo, n, n, H, Fp,
                                     alpha, mode, edge_keep, (__nv_bfloat16*)d_Wh, ld_dwh, d_s, d_t, row_scratch, nnz,
                                     long_rows, n_long, long_rows_t, n_long_t, long_threshold, (cudaStream_t)stream,
                                     apply_elu, (__nv_bfloat16*)d_pre, dropout, batch_nodes);
}

int gnn_gat_fused_bwd_ex_f32(const int64_t* rowptr, const int32_t* col, const int64_t* rowptr_t, const int32_t* col_t,
                             const int64_t* perm_t, const float* Wh, int64_t ldw, const float* s, const float* t,
                             const float* row_max, const float* row_sum, const float* out_pre, const float* d_out,
                             int64_t ldo, int64_t n_rows, int64_t n_cols, int32_t H, int32_t Fp, float alpha, int mode,
                             const float* edge_keep, float* d_Wh, int64_t ld_dwh, float* d_s, float* d_t,
                             float* row_scratch, int64_t nnz, const int64_t* long_rows, int64_t n_long,
                             const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold, int apply_elu,
                             float* d_pre, const gnn_gat_dropout* dropout, gnn_stream_t stream) {
  return gat_bwd_impl<float>(rowptr, col, rowptr_t, col_t, perm_t, Wh, ldw, s, t, row_max, row_sum, out_pre, d_out, ldo,
                             n_rows, n_cols, H, Fp, alpha, mode, edge_keep, d_Wh, ld_dwh, d_s, d_t, row_scratch, nnz,
                             long_rows, n_long, long_rows_t, n_long_t, long_threshold, (cudaStream_t)stream, apply_elu,
                             d_pre, dropout, 0);
}

int gnn_gat_fused_bwd_ex_bf16(const int64_t* rowptr, const int32_t* col, const int64_t* rowptr_t, const int32_t* col_t,
                              const int64_t* perm_t, const void* Wh, int64_t ldw, const float* s, const float* t,
                              const float* row_max, const float* row_sum, const void* out_pre, const void* d_out,
                              int64_t ldo, int64_t n_rows, int64_t n_cols, int32_t H, int32_t Fp, float alpha, int mode,
                              const float* edge_keep, void* d_Wh, int64_t ld_dwh, float* d_s, float* d_t,
                              float* row_scratch, int64_t nnz, const int64_t* long_rows, int64_t n_long,
                              const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold, int apply_elu,
                              void* d_pre, const gnn_gat_dropout* dropout, gnn_stream_t stream) {
  return gat_bwd_impl<__nv_bfloat16>(rowptr, col, rowptr_t, col_t, perm_t, (const __nv_bfloat16*)Wh, ldw, s, t, row_max,
                                     row_sum, (const __nv_bfloat16*)out_pre, (const __nv_bfloat16*)d_out, ldo, n_rows,
                                     n_cols, H, Fp, alpha, mode, edge_keep, (__nv_bfloat16*)d_Wh, ld_dwh, d_s, d_t,
                                     row_scratch, nnz, long_rows, n_long, long_rows_t, n_long_t, long_threshold,
                                     (cudaStream_t)stream, apply_elu, (__nv_bfloat16*)d_pre, dropout, 0);
}

int gnn_gat_fused_fwd_batch_f32(const int64_t* rowptr, const int32_t* col, const float* Wh, int64_t ldw,
                                const float* s, const float* t, int64_t nnz, int32_t H, int32_t Fp, float alpha,
                                int mode, int apply_elu, const float* edge_keep, const gnn_gat_dropout* dropout,
                                float* out_pre, float* out_act, int64_t ldo, float* row_max, float* row_sum,
                                const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                                const gnn_gat_batch* batch, gnn_stream_t stream) {
  int64_t n = 0, n_cols = 0;
  int rc = check_batch(batch, &n, &n_cols);
  if (rc != GNN_OK) return rc;
  GNN_REQUIRE(out_act || apply_elu == 0, GNN_ERR_BAD_ARG, "apply_elu > 0 needs out_act");
  if (n == 0) return GNN_OK;
  return gat_fwd_impl<float>(rowptr, col, Wh, ldw, s, t, n, nnz, H, Fp, alpha, mode, apply_elu, nullptr, edge_keep,
                             out_pre, ldo, row_max, row_sum, long_rows, n_long, long_threshold, (cudaStream_t)stream,
                             apply_elu > 0 ? out_act : nullptr, dropout, batch->rows_per_graph, batch);
}

int gnn_gat_fused_bwd_batch_f32(const int64_t* rowptr, const int32_t* col, const int64_t* rowptr_t, const int32_t* col_t,
                                const int64_t* perm_t, const float* Wh, int64_t ldw, const float* s, const float* t,
                                const float* row_max, const float* row_sum, const float* out_pre, const float* d_out,
                                int64_t ldo, int32_t H, int32_t Fp, float alpha, int mode, const float* edge_keep,
                                float* d_Wh, int64_t ld_dwh, float* d_s, float* d_t, float* row_scratch, int64_t nnz,
                                const int64_t* long_rows, int64_t n_long, const int64_t* long_rows_t, int64_t n_long_t,
                                int64_t long_threshold, int apply_elu, float* d_pre, const gnn_gat_dropout* dropout,
                                const gnn_gat_batch* batch, gnn_stream_t stream) {
  int64_t n = 0, n_cols = 0;
  int rc = check_batch(batch, &n, &n_cols);
  if (rc != GNN_OK) return rc;
  return gat_bwd_impl<float>(rowptr, col, rowptr_t, col_t, perm_t, Wh, ldw, s, t, row_max, row_sum, out_pre, d_out, ldo,
                             n, n_cols, H, Fp, alpha, mode, edge_keep, d_Wh, ld_dwh, d_s, d_t, row_scratch, nnz,
                             long_rows, n_long, long_rows_t, n_long_t, long_threshold, (cudaStream_t)stream, apply_elu,
                             d_pre, dropout, batch->rows_per_graph, batch);
}

int gnn_gat_fused_fwd_batch_bf16(const int64_t* rowptr, const int32_t* col, const void* Wh, int64_t ldw,
                                 const float* s, const float* t, int64_t nnz, int32_t H, int32_t Fp, float alpha,
                                 int mode, int apply_elu, const float* edge_keep, const gnn_gat_dropout* dropout,
                                 void* out_pre, void* out_act, int64_t ldo, float* row_max, float* row_sum,
                                 const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                                 const gnn_gat_batch* batch, gnn_stream_t stream) {
  int64_t n = 0, n_cols = 0;
  int rc = check_batch(batch, &n, &n_cols);
  if (rc != GNN_OK) return rc;
  GNN_REQUIRE(out_act || apply_elu == 0, GNN_ERR_BAD_ARG, "apply_elu > 0 needs out_act");
  if (n == 0) return GNN_OK;
  return gat_fwd_impl<__nv_bfloat16>(rowptr, col, (const __nv_bfloat16*)Wh, ldw, s, t, n, nnz, H, Fp, alpha, mode,
                                     apply_elu, nullptr, edge_keep, (__nv_bfloat16*)out_pre, ldo, row_max, row_sum,
                                     long_rows, n_long, long_threshold, (cudaStream_t)stream,
                                     apply_elu > 0 ? (__nv_bfloat16*)out_act : nullptr, dropout, batch->rows_per_graph,
                                     batch);
}

int gnn_gat_fused_bwd_batch_bf16(const int64_t* rowptr, const int32_t* col, const int64_t* rowptr_t,
                                 const int32_t* col_t, const int64_t* perm_t, const void* Wh, int64_t ldw,
                                 const float* s, const float* t, const float* row_max, const float* row_sum,
                                 const void* out_pre, const void* d_out, int64_t ldo, int32_t H, int32_t Fp,
                                 float alpha, int mode, const float* edge_keep, void* d_Wh, int64_t ld_dwh, float* d_s,
                                 float* d_t, float* row_scratch, int64_t nnz, const int64_t* long_rows, int64_t n_long,
                                 const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold, int apply_elu,
                                 void* d_pre, const gnn_gat_dropout* dropout, const gnn_gat_batch* batch,
                                 gnn_stream_t stream) {
  int64_t n = 0, n_cols = 0;
  int rc = check_batch(batch, &n, &n_cols);
  if (rc != GNN_OK) return rc;
  return gat_bwd_impl<__nv_bfloat16>(rowptr, col, rowptr_t, col_t, perm_t, (const __nv_bfloat16*)Wh, ldw, s, t, row_max,
                                     row_sum, (const __nv_bfloat16*)out_pre, (const __nv_bfloat16*)d_out, ldo, n, n_cols,
                                     H, Fp, alpha, mode, edge_keep, (__nv_bfloat16*)d_Wh, ld_dwh, d_s, d_t,
                                     row_scratch, nnz, long_rows, n_long, long_rows_t, n_long_t, long_threshold,
                                     (cudaStream_t)stream, apply_elu, (__nv_bfloat16*)d_pre, dropout,
                                     batch->rows_per_graph, batch);
}

}  // extern "C"
