// GraphSAGE fixed-fanout neighbour gather + reduce, fused.
// Replaces, at /root/reference:
//   GraphSAGE_Pytorch/data_utils.py:64          CPU feature gather of the sampled ids
//   GraphSAGE_Pytorch/models/Aggregator.py:19-24 mean / sum / max over the fanout axis
//   GraphSAGE/graph_utils.py:6 + GraphSAGE.py:47-49  torch.embedding + torch.mean
//
// TMA path (sm_100a): persistent CTAs (4 per SM) take source nodes blockIdx.x, +grid, ...;
// one producer warp reads the sampled ids (next chunk prefetched) and issues one
// cp.async.bulk (TMA 1-D bulk copy, SASS UBLKCP) per gathered feature row into a
// shared-memory ring, completing on an mbarrier; five consumer warps add the staged rows from
// shared memory (LDS.128) in fanout order and write the reduced row once.  No feature row
// touches a register before it is reduced.  Up to 4 index blocks with different fanouts (the
// hops of one minibatch: GraphSage.py:24-27 runs every hop through the same layer) share ONE
// launch, so the short hop-1 block rides in the shadow of the long hop-2 block.
// Vector-load path: the row-parallel kernel of rowreduce.cuh with an implicit CSR
// (rowptr = i*fanout), used when rows are not 16-byte aligned or too short for TMA.
#include "rowreduce.cuh"

using namespace gnn;

namespace {

constexpr int kConsumerWarps = 5;
constexpr int kConsumerThreads = kConsumerWarps * 32;
constexpr int kSageThreads = 32 + kConsumerThreads;
constexpr int kMaxBlocks = 4;
constexpr int kIdDepth = 4;  // chunks of sampled ids the producer keeps in flight

template <typename T>
struct SageArgs {
  const T* table;
  int64_t ld;
  int32_t F;
  int32_t n_blocks;
  const int32_t* idx32[kMaxBlocks];
  const int64_t* idx64[kMaxBlocks];
  int64_t src_off[kMaxBlocks + 1];  // cumulative source counts; a CTA strides over the union
  int32_t fanout[kMaxBlocks];
  int32_t kc[kMaxBlocks];            // rows per ring stage for this block
  float scale[kMaxBlocks];
  T* out[kMaxBlocks];
  int64_t ldo[kMaxBlocks];
  int32_t* argmax[kMaxBlocks];
  int32_t out_vec16[kMaxBlocks];     // output rows can take 16-byte stores
  int32_t row_bytes;                 // bytes copied per row (multiple of 16)
  int32_t stage_rows;                // ring stage capacity in rows (max kc)
  int32_t stages;
  int32_t nvec;                      // 16-byte vectors per row
  int64_t n_table_rows;              // ids outside [0, n_table_rows) are skipped like negative (padding) ids
  // fp32 tables only: write every reduced value x as TWO fp16 planes, hi = fp16(x) at out[...] and
  // lo = fp16(x - hi) lo_off[b] fp16 elements further (out / ldo then count fp16 elements).  hi + lo carries 22
  // mantissa bits (x - hi is exact in fp32; a lo below fp16's normal range only costs < 3e-8 ABSOLUTE): the operand
  // form of a 3-product fp16 tensor-core GEMM with fp32 accumulation that stands in for the fp32 X.W product at
  // fp32-level accuracy.  The caller guarantees |x| < 65504 (fp16 range).
  int32_t split[kMaxBlocks];
  int64_t lo_off[kMaxBlocks];
};

// Sharded table (gnn_sharded_table): global row r of shard s = the largest s with row_begin[s] <= r lives at
// base[s] + (r - row_begin[s]) * ld = origin[s] + r * ld, origin[s] the byte address base[s] - row_begin[s] * ld
// (integer arithmetic: it may lie outside any allocation; only origin + r * ld is ever dereferenced).  Bounds fit
// int32 (n_table_rows < 2^31).  `table` is unused; n_table_rows = row_begin[n_shards].
template <typename T>
struct SageShardedArgs : SageArgs<T> {
  uint64_t origin[GNN_MAX_SHARDS];
  int32_t row_begin[GNN_MAX_SHARDS];
  int32_t n_shards;
};
template <typename T, bool SH>
struct SageArgsOf {
  using type = SageArgs<T>;
};
template <typename T>
struct SageArgsOf<T, true> {
  using type = SageShardedArgs<T>;
};

// Two fp32 adds in one instruction (SASS FADD2, sm_100): same round-to-nearest result as two
// FADDs at half the issue slots.  The bf16 consumer loop was issue-bound (ncu r01: 195 warp
// instructions per 1.2 KB row, 64 % issue-active with one scheduler idle).
__device__ __forceinline__ void add2(float& a0, float& a1, float x0, float x1) {
  asm("{\n\t.reg .b64 ra, rx;\n\tmov.b64 ra, {%0, %1};\n\tmov.b64 rx, {%2, %3};\n\t"
      "add.rn.f32x2 ra, ra, rx;\n\tmov.b64 {%0, %1}, ra;\n\t}"
      : "+f"(a0), "+f"(a1)
      : "f"(x0), "f"(x1));
}

template <typename T>
struct Vec16;
template <>
struct Vec16<float> {
  static constexpr int E = 4;
  static __device__ __forceinline__ void unpack(const uint4& w, float (&o)[4]) {
    o[0] = __uint_as_float(w.x); o[1] = __uint_as_float(w.y); o[2] = __uint_as_float(w.z); o[3] = __uint_as_float(w.w);
  }
  static __device__ __forceinline__ void add(const uint4& w, float (&acc)[4]) {
    add2(acc[0], acc[1], __uint_as_float(w.x), __uint_as_float(w.y));
    add2(acc[2], acc[3], __uint_as_float(w.z), __uint_as_float(w.w));
  }
};
template <>
struct Vec16<__nv_bfloat16> {
  static constexpr int E = 8;
  static __device__ __forceinline__ void unpack(const uint4& w, float (&o)[8]) {
    bf16x2_to_f32(w.x, o[0], o[1]); bf16x2_to_f32(w.y, o[2], o[3]);
    bf16x2_to_f32(w.z, o[4], o[5]); bf16x2_to_f32(w.w, o[6], o[7]);
  }
  static __device__ __forceinline__ void add(const uint4& w, float (&acc)[8]) {
    float x[8];
    unpack(w, x);
#pragma unroll
    for (int i = 0; i < 8; i += 2) add2(acc[i], acc[i + 1], x[i], x[i + 1]);
  }
};

// position of a CTA in its work list: (global source g -> block b, source within block, chunk)
struct Cursor {
  int64_t g;
  int64_t src;
  int b, fan, kc, c0;
};
template <typename T>
__device__ __forceinline__ void cursor_set(Cursor& c, const SageArgs<T>& a, int64_t g) {
  c.g = g;
  c.c0 = 0;
  if (g < a.src_off[a.n_blocks]) {
    int b = 0;
    while (b + 1 < a.n_blocks && g >= a.src_off[b + 1]) ++b;
    c.b = b;
    c.src = g - a.src_off[b];
    c.fan = a.fanout[b];
    c.kc = a.kc[b];
  }
}
template <typename T>
__device__ __forceinline__ void cursor_next(Cursor& c, const SageArgs<T>& a) {
  c.c0 += c.kc;
  if (c.c0 >= c.fan) cursor_set(c, a, c.g + gridDim.x);
}

// CTAs per SM the register allocation of the sharded kernel is held to (0: ptxas chooses, as for the unsharded
// kernel).  4 x 192 threads caps it at 80 registers, what the unsharded twin uses or less; without the bound ptxas
// spilled a few bytes in some sharded twins of spill-free kernels.  The bf16 max kernels with 3-4 vectors per thread
// need 114-121 registers unsharded, so they keep ptxas's choice.
template <typename T, int NV, int OP, bool SH>
constexpr int sage_min_ctas() {
  return (SH && !(sizeof(T) == 2 && OP == GNN_REDUCE_MAX && NV >= 3)) ? 4 : 0;
}

// SH: the table is sharded (SageShardedArgs); only the producer's source address depends on it.
template <typename T, int NV, int OP, bool PK = true, bool SH = false>
__global__ void __launch_bounds__(kSageThreads, (sage_min_ctas<T, NV, OP, SH>()))
    sage_tma_kernel(const typename SageArgsOf<T, SH>::type a) {
  constexpr int E = Vec16<T>::E;
  extern __shared__ __align__(128) unsigned char smem[];
  const int S = a.stages;
  const int stage_bytes = a.stage_rows * a.row_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)S * stage_bytes);
  uint64_t* empty = full + S;
  uint32_t* mask = reinterpret_cast<uint32_t*>(empty + S);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < S; ++i) {
      mbar_init(full + i, 1);
      mbar_init(empty + i, kConsumerWarps);
    }
    mbar_fence_init();
  }
  __syncthreads();
  const int64_t total_src = a.src_off[a.n_blocks];

  if (warp == 0) {
    // ===== producer: sampled ids -> one bulk copy per gathered row =====
    auto load_id = [&](const Cursor& c) -> int64_t {
      if (c.g >= total_src) return -1;
      const int rows = min(c.kc, c.fan - c.c0);
      if (lane >= rows) return -1;
      const int64_t p = c.src * c.fan + c.c0 + lane;
      if (a.idx32[c.b]) return (int64_t)__ldg(a.idx32[c.b] + p);
      if (a.idx64[c.b]) return __ldg(a.idx64[c.b] + p);
      return p;  // identity block
    };
    // The ids of the next kIdDepth chunks are always in flight: with a single chunk of lookahead
    // the producer paid one DRAM round trip per ring stage whenever a source's ids sat in a
    // sector of their own (fanout 10 = 40 bytes), which capped the 1.2 KB bf16 rows at 0.61.
    Cursor cur, look;
    cursor_set(cur, a, blockIdx.x);
    look = cur;
    int64_t rq[kIdDepth];
#pragma unroll
    for (int d = 0; d < kIdDepth; ++d) {
      rq[d] = load_id(look);
      if (look.g < total_src) cursor_next(look, a);
    }
    int stage = 0;
    uint32_t par = 0;
    while (cur.g < total_src) {
#pragma unroll
      for (int d = 0; d < kIdDepth; ++d) {
        if (cur.g >= total_src) break;
        const int64_t r = rq[d];
        rq[d] = load_id(look);
        if (look.g < total_src) cursor_next(look, a);
        mbar_wait(empty + stage, par ^ 1u);
        const bool valid = r >= 0 && r < a.n_table_rows;
        const unsigned m = __ballot_sync(0xffffffffu, valid);
        if (lane == 0) {
          mask[stage] = m;
          mbar_arrive_expect_tx(full + stage, (uint32_t)__popc(m) * (uint32_t)a.row_bytes);
        }
        __syncwarp();
        if (valid) {
          const T* src;
          if constexpr (SH) {
            // unrolled scan of the (uniform) shard bounds: no per-lane indexing into the parameter space
            uint64_t origin = a.origin[0];
#pragma unroll
            for (int s = 1; s < GNN_MAX_SHARDS; ++s)
              if (s < a.n_shards && (int32_t)r >= a.row_begin[s]) origin = a.origin[s];
            src = reinterpret_cast<const T*>(origin + (uint64_t)(r * a.ld) * sizeof(T));
          } else {
            src = a.table + r * a.ld;
          }
          bulk_g2s(smem + (size_t)stage * stage_bytes + (size_t)lane * a.row_bytes, src, (uint32_t)a.row_bytes,
                   full + stage);
        }
        cursor_next(cur, a);
        if (++stage == S) {
          stage = 0;
          par ^= 1u;
        }
      }
    }
  } else {
    // ===== consumers: reduce the staged rows in fanout order =====
    const int t = threadIdx.x - 32;
    float acc[NV][E];
    int best[NV][E];
    auto reset = [&]() {
#pragma unroll
      for (int v = 0; v < NV; ++v)
#pragma unroll
        for (int i = 0; i < E; ++i) {
          acc[v][i] = (OP == GNN_REDUCE_MAX) ? -INFINITY : 0.f;
          best[v][i] = 0;
        }
    };
    reset();
    Cursor cur;
    cursor_set(cur, a, blockIdx.x);
    int stage = 0;
    uint32_t par = 0;
    for (; cur.g < total_src; cursor_next(cur, a)) {
      const int c0 = cur.c0;
      const int rows = min(cur.kc, cur.fan - c0);
      mbar_wait(full + stage, par);
      const unsigned m = mask[stage];
      const unsigned char* sb = smem + (size_t)stage * stage_bytes;
      const unsigned all_rows = rows >= 32 ? 0xffffffffu : ((1u << rows) - 1u);
      if (OP != GNN_REDUCE_MAX && m == all_rows) {
        // every id of the chunk is valid (the sampled blocks of GraphSAGE_Pytorch always are):
        // no per-row mask test, packed adds
#pragma unroll 5
        for (int k = 0; k < rows; ++k) {
#pragma unroll
          for (int v = 0; v < NV; ++v) {
            const int vi = t + v * kConsumerThreads;
            if (vi < a.nvec) {
              const uint4 w = *reinterpret_cast<const uint4*>(sb + (size_t)k * a.row_bytes + (size_t)vi * 16);
              if (PK) {
                Vec16<T>::add(w, acc[v]);
              } else {
                float x[E];
                Vec16<T>::unpack(w, x);
#pragma unroll
                for (int i = 0; i < E; ++i) acc[v][i] += x[i];
              }
            }
          }
        }
      } else {
#pragma unroll 4
        for (int k = 0; k < rows; ++k) {
          if (!((m >> k) & 1u)) continue;
#pragma unroll
          for (int v = 0; v < NV; ++v) {
            const int vi = t + v * kConsumerThreads;
            if (vi < a.nvec) {
              const uint4 w = *reinterpret_cast<const uint4*>(sb + (size_t)k * a.row_bytes + (size_t)vi * 16);
              float x[E];
              Vec16<T>::unpack(w, x);
#pragma unroll
              for (int i = 0; i < E; ++i) {
                if (OP == GNN_REDUCE_MAX) {
                  if (x[i] > acc[v][i]) {
                    acc[v][i] = x[i];
                    best[v][i] = c0 + k;
                  }
                } else {
                  acc[v][i] += x[i];
                }
              }
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty + stage);
      if (c0 + cur.kc >= cur.fan) {  // last chunk of this source: write the reduced row
        const int b = cur.b;
        T* orow = a.out[b] + cur.src * a.ldo[b];
        const float scale = a.scale[b];
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int vi = t + v * kConsumerThreads;
          if (vi < a.nvec) {
            float o[E];
#pragma unroll
            for (int i = 0; i < E; ++i) o[i] = (OP == GNN_REDUCE_MAX) ? acc[v][i] : acc[v][i] * scale;
            const int col0 = vi * E;
            if (sizeof(T) == 4 && a.split[b]) {
              // E == 4 floats -> 4 + 4 fp16 (two 8-byte stores); columns >= F are padding and stay untouched
              __half* hrow = reinterpret_cast<__half*>(a.out[b]) + cur.src * a.ldo[b] + col0;
              uint32_t hw[2], lw[2];
#pragma unroll
              for (int i = 0; i < 2; ++i) {
                const __half h0 = __float2half_rn(o[2 * i]), h1 = __float2half_rn(o[2 * i + 1]);
                const __half l0 = __float2half_rn(o[2 * i] - __half2float(h0));
                const __half l1 = __float2half_rn(o[2 * i + 1] - __half2float(h1));
                hw[i] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
                lw[i] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
              }
              if (col0 + 3 < a.F) {
                *reinterpret_cast<uint2*>(hrow) = make_uint2(hw[0], hw[1]);
                *reinterpret_cast<uint2*>(hrow + a.lo_off[b]) = make_uint2(lw[0], lw[1]);
              } else {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                  if (col0 + i < a.F) {
                    const __half h = __float2half_rn(o[i]);
                    hrow[i] = h;
                    hrow[a.lo_off[b] + i] = __float2half_rn(o[i] - __half2float(h));
                  }
              }
            } else if (a.out_vec16[b]) {
              store_cols<T, E>(orow + col0, o, a.F - col0);  // columns >= F stay untouched
            } else {
#pragma unroll
              for (int i = 0; i < E; ++i)
                if (col0 + i < a.F) {
                  float o1[1] = {o[i]};
                  VecIO<T, 1>::store(orow + col0 + i, o1);
                }
            }
            if (OP == GNN_REDUCE_MAX && a.argmax[b]) {
#pragma unroll
              for (int i = 0; i < E; ++i)
                if (col0 + i < a.F) a.argmax[b][cur.src * a.ldo[b] + col0 + i] = best[v][i];
            }
          }
        }
        reset();
      }
      if (++stage == S) {
        stage = 0;
        par ^= 1u;
      }
    }
  }
}

template <typename T, int NV, int OP, bool PK, bool SH>
int launch_tma_pk(const typename SageArgsOf<T, SH>::type& a, size_t smem_bytes, int grid, cudaStream_t st) {
  // function attributes belong to a device's context: remember the largest size set PER DEVICE (a process driving
  // several GPUs must not skip the call on the second one); benign race: setting the attribute is idempotent
  static size_t configured[64] = {};
  int dev = 0;
  const bool cached = cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64;
  if (!cached || smem_bytes > configured[dev]) {
    GNN_CUDA(cudaFuncSetAttribute(sage_tma_kernel<T, NV, OP, PK, SH>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem_bytes));
    if (cached) configured[dev] = smem_bytes;
  }
  sage_tma_kernel<T, NV, OP, PK, SH><<<grid, kSageThreads, smem_bytes, st>>>(a);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

template <typename T, int NV, int OP, bool SH>
int launch_tma_inst(const typename SageArgsOf<T, SH>::type& a, size_t smem_bytes, int grid, cudaStream_t st) {
  // packed adds pay where the consumers are issue-bound (bf16: 8 unpack + 8 add per 16 bytes);
  // "sage.packed_add": -1 = by dtype, 0 / 1 = force
  const int knob = tuning("sage.packed_add", -1);
  const bool pk = (OP != GNN_REDUCE_MAX) && (knob < 0 ? sizeof(T) == 2 : knob != 0);
  if (pk) return launch_tma_pk<T, NV, OP, true, SH>(a, smem_bytes, grid, st);
  return launch_tma_pk<T, NV, OP, false, SH>(a, smem_bytes, grid, st);
}

template <typename T, int OP, bool SH>
int launch_tma(const typename SageArgsOf<T, SH>::type& a, size_t smem_bytes, int grid, cudaStream_t st) {
  const int nv = (a.nvec + kConsumerThreads - 1) / kConsumerThreads;
  switch (nv) {
    case 1: return launch_tma_inst<T, 1, OP, SH>(a, smem_bytes, grid, st);
    case 2: return launch_tma_inst<T, 2, OP, SH>(a, smem_bytes, grid, st);
    case 3: return launch_tma_inst<T, 3, OP, SH>(a, smem_bytes, grid, st);
    case 4: return launch_tma_inst<T, 4, OP, SH>(a, smem_bytes, grid, st);
    default: break;
  }
  set_error("TMA gather: row too wide (nvec=%d)", a.nvec);
  return GNN_ERR_UNSUPPORTED;
}

template <typename T>
struct GatherBlock {
  const void* idx;
  int idx_bits;
  int64_t n_src;
  int32_t fanout;
  T* out;
  int64_t ldo;
  int32_t* argmax;
  int32_t split = 0;     // fp32 only: out is an fp16 buffer, hi/lo planes (see SageArgs::split)
  int64_t lo_off = 0;
};

// Every field of a gnn_sharded_table, before anything is launched.
int check_sharded_table(const gnn_sharded_table* sh, int64_t ld, int32_t F, int esz) {
  GNN_REQUIRE(sh, GNN_ERR_BAD_ARG, "null sharded table");
  GNN_REQUIRE(sh->struct_size == (int32_t)sizeof(gnn_sharded_table), GNN_ERR_BAD_ARG,
              "gnn_sharded_table.struct_size %d, expected %d", sh->struct_size, (int)sizeof(gnn_sharded_table));
  GNN_REQUIRE(sh->n_shards >= 1 && sh->n_shards <= GNN_MAX_SHARDS, GNN_ERR_BAD_ARG, "n_shards %d outside [1, %d]",
              sh->n_shards, GNN_MAX_SHARDS);
  GNN_REQUIRE(sh->row_begin[0] == 0, GNN_ERR_BAD_ARG, "row_begin[0] must be 0");
  for (int s = 0; s < sh->n_shards; ++s) {
    GNN_REQUIRE(sh->row_begin[s + 1] >= sh->row_begin[s], GNN_ERR_BAD_ARG, "row_begin decreases at shard %d", s);
    if (sh->row_begin[s + 1] > sh->row_begin[s])
      GNN_REQUIRE(sh->base[s] && aligned_to(sh->base[s], 16), GNN_ERR_MISALIGNED,
                  "shard %d: base must be non-null and 16-byte aligned", s);
  }
  GNN_REQUIRE(ld >= F && F >= 0, GNN_ERR_BAD_ARG, "leading dimension smaller than F");
  GNN_REQUIRE(ld * esz % 16 == 0, GNN_ERR_MISALIGNED, "sharded table: ld_table * elem must be a multiple of 16");
  return GNN_OK;
}

template <typename T>
int gather_reduce_impl(const T* table, int64_t ld, int64_t n_table_rows, int32_t F, int reduce,
                       const GatherBlock<T>* blocks, int n_blocks, cudaStream_t st,
                       const gnn_sharded_table* sh = nullptr) {
  if (sh) {
    const int rc = check_sharded_table(sh, ld, F, (int)sizeof(T));
    if (rc != GNN_OK) return rc;
    const size_t rb = round_up((size_t)F * sizeof(T), 16);
    GNN_REQUIRE(F == 0 || (rb >= 256 && rb / 16 <= 4 * (size_t)kConsumerThreads), GNN_ERR_UNSUPPORTED,
                "sharded table: TMA path only, rows of 256 to %d bytes (F=%d gives %d)", 64 * kConsumerThreads, F,
                (int)rb);
    n_table_rows = sh->row_begin[sh->n_shards];
  }
  GNN_REQUIRE(F >= 0 && n_blocks >= 0 && n_blocks <= kMaxBlocks, GNN_ERR_BAD_ARG, "bad size (F=%d, blocks=%d, max %d)",
              F, n_blocks, kMaxBlocks);
  GNN_REQUIRE(reduce == GNN_REDUCE_MEAN || reduce == GNN_REDUCE_SUM || reduce == GNN_REDUCE_MAX, GNN_ERR_BAD_ARG,
              "unknown reduce %d (GraphSAGE_Pytorch/models/Aggregator.py:26 raises ValueError)", reduce);
  GNN_REQUIRE(n_table_rows < 0x7fffffffLL, GNN_ERR_UNSUPPORTED, "table rows do not fit int32");
  int64_t total_src = 0;
  for (int b = 0; b < n_blocks; ++b) {
    const GatherBlock<T>& k = blocks[b];
    GNN_REQUIRE(k.n_src >= 0 && k.fanout >= 0, GNN_ERR_BAD_ARG, "negative size");
    if (k.n_src == 0 || F == 0) continue;
    GNN_REQUIRE(k.fanout > 0, GNN_ERR_BAD_ARG, "fanout must be positive");
    GNN_REQUIRE((table || sh) && k.out, GNN_ERR_BAD_ARG, "null table/out");
    GNN_REQUIRE(k.idx == nullptr || k.idx_bits == 32 || k.idx_bits == 64, GNN_ERR_BAD_ARG, "idx_bits must be 32 or 64");
    GNN_REQUIRE(ld >= F && k.ldo >= F, GNN_ERR_BAD_ARG, "leading dimension smaller than F");
    GNN_REQUIRE(!k.split || (sizeof(T) == 4 && reduce != GNN_REDUCE_MAX && k.lo_off >= F && k.ldo % 4 == 0 &&
                             k.lo_off % 4 == 0 && aligned_to(k.out, 8)),
                GNN_ERR_BAD_ARG, "hi/lo fp16 output needs an fp32 table, mean/sum, 8-byte aligned planes");
    GNN_REQUIRE(k.idx != nullptr || k.n_src * (int64_t)k.fanout <= n_table_rows, GNN_ERR_BAD_ARG,
                "identity block needs n_src*fanout <= n_table_rows");
    total_src += k.n_src;
  }
  if (total_src == 0 || F == 0) return GNN_OK;

  const int esz = (int)sizeof(T);
  const int row_bytes = (int)round_up((size_t)F * esz, 16);
  // a sharded table has no vector-load form: its rows were checked for the TMA path above
  const bool tma_ok = sh || (!tuning("sage.force_ldg", 0) && aligned_to(table, 16) && ((ld * esz) % 16 == 0) &&
                             (int64_t)row_bytes <= ld * esz && row_bytes >= 256 && (row_bytes / 16) <= 4 * kConsumerThreads);
  if (tma_ok) {
    SageShardedArgs<T> a{};
    if (sh) {
      for (int s = 0; s < sh->n_shards; ++s) {
        a.origin[s] = (uint64_t)(uintptr_t)sh->base[s] - (uint64_t)(sh->row_begin[s] * ld) * sizeof(T);
        a.row_begin[s] = (int32_t)sh->row_begin[s];
      }
      a.n_shards = sh->n_shards;
    }
    a.table = table;
    a.ld = ld;
    a.F = F;
    a.n_table_rows = n_table_rows;
    a.row_bytes = row_bytes;
    a.nvec = row_bytes / 16;
    const int E = 16 / esz;
    int kc0 = tuning("sage.chunk_bytes", 12288) / row_bytes;
    kc0 = kc0 < 1 ? 1 : kc0;
    kc0 = kc0 > 32 ? 32 : kc0;
    const size_t budget = (size_t)tuning("sage.smem_kb", 48) * 1024;
    while (kc0 > 1 && budget / ((size_t)kc0 * row_bytes) < 2) kc0 = (kc0 + 1) / 2;
    int nb = 0, stage_rows = 1;
    a.src_off[0] = 0;
    for (int b = 0; b < n_blocks; ++b) {
      const GatherBlock<T>& k = blocks[b];
      if (k.n_src == 0) continue;
      a.idx32[nb] = (k.idx && k.idx_bits == 32) ? (const int32_t*)k.idx : nullptr;
      a.idx64[nb] = (k.idx && k.idx_bits == 64) ? (const int64_t*)k.idx : nullptr;
      a.fanout[nb] = k.fanout;
      int kc = kc0 > k.fanout ? k.fanout : kc0;
      const int nchunk = (k.fanout + kc - 1) / kc;
      kc = (k.fanout + nchunk - 1) / nchunk;  // balance the chunks of one source
      a.kc[nb] = kc;
      stage_rows = kc > stage_rows ? kc : stage_rows;
      a.scale[nb] = (reduce == GNN_REDUCE_MEAN) ? 1.0f / (float)k.fanout : 1.0f;
      a.out[nb] = k.out;
      a.ldo[nb] = k.ldo;
      a.argmax[nb] = (reduce == GNN_REDUCE_MAX) ? k.argmax : nullptr;
      a.out_vec16[nb] = aligned_to(k.out, 16) && ((k.ldo * esz) % 16 == 0) && ((int64_t)a.nvec * E <= k.ldo);
      a.split[nb] = k.split;
      a.lo_off[nb] = k.lo_off;
      a.src_off[nb + 1] = a.src_off[nb] + k.n_src;
      ++nb;
    }
    a.n_blocks = nb;
    a.stage_rows = stage_rows;
    int stages = (int)(budget / ((size_t)stage_rows * row_bytes));
    stages = stages > 8 ? 8 : stages;
    GNN_REQUIRE(stages >= 2, GNN_ERR_UNSUPPORTED, "row of %d bytes does not fit the shared-memory ring", row_bytes);
    a.stages = stages;
    const size_t smem_bytes = (size_t)stages * stage_rows * row_bytes + (size_t)stages * (16 + 4) + 16;
    int64_t grid = (int64_t)num_sms() * tuning("sage.ctas_per_sm", 4);
    grid = grid > total_src ? total_src : grid;
    const SageArgs<T>& flat = a;  // the unsharded kernels take the base part only
    switch (reduce) {
      case GNN_REDUCE_MAX:
        return sh ? launch_tma<T, GNN_REDUCE_MAX, true>(a, smem_bytes, (int)grid, st)
                  : launch_tma<T, GNN_REDUCE_MAX, false>(flat, smem_bytes, (int)grid, st);
      default:
        return sh ? launch_tma<T, GNN_REDUCE_SUM, true>(a, smem_bytes, (int)grid, st)
                  : launch_tma<T, GNN_REDUCE_SUM, false>(flat, smem_bytes, (int)grid, st);
    }
  }

  for (int b = 0; b < n_blocks; ++b)
    GNN_REQUIRE(!blocks[b].split, GNN_ERR_UNSUPPORTED,
                "hi/lo fp16 output is implemented on the TMA path only (16-byte aligned rows of >= 256 bytes)");
  for (int b = 0; b < n_blocks; ++b) {
    const GatherBlock<T>& k = blocks[b];
    if (k.n_src == 0) continue;
    RowArgs<T> r{};
    r.rowptr = nullptr;
    r.fanout = k.fanout;
    r.col32 = (k.idx && k.idx_bits == 32) ? (const int32_t*)k.idx : nullptr;
    r.col64 = (k.idx && k.idx_bits == 64) ? (const int64_t*)k.idx : nullptr;
    r.val = nullptr;
    r.src_div = 0;
    r.scale = (reduce == GNN_REDUCE_MEAN) ? 1.0f / (float)k.fanout : 1.0f;
    r.n_src_rows = (int32_t)n_table_rows;
    r.X = table;
    r.ldx = ld;
    r.Y = k.out;
    r.ldy = k.ldo;
    r.n_rows = k.n_src;
    r.F = F;
    r.skip_deg_gt = 0;
    r.argmax = (reduce == GNN_REDUCE_MAX) ? k.argmax : nullptr;
    const int rc = (reduce == GNN_REDUCE_MAX) ? launch_row_reduce<T, 1>(r, st) : launch_row_reduce<T, 0>(r, st);
    if (rc != GNN_OK) return rc;
  }
  return GNN_OK;
}

template <typename T>
int gather_reduce_multi(const T* table, int64_t ld, int64_t n_table_rows, int32_t F, int reduce, int32_t n_blocks,
                        const void* const* idx, int idx_bits, const int64_t* n_src, const int32_t* fanout,
                        void* const* out, const int64_t* ld_out, cudaStream_t st,
                        const gnn_sharded_table* sh = nullptr) {
  GNN_REQUIRE(n_blocks >= 0 && n_blocks <= kMaxBlocks, GNN_ERR_UNSUPPORTED, "at most %d blocks per launch", kMaxBlocks);
  GNN_REQUIRE(n_blocks == 0 || (idx && n_src && fanout && out && ld_out), GNN_ERR_BAD_ARG, "null block array");
  GatherBlock<T> blocks[kMaxBlocks];
  for (int b = 0; b < n_blocks; ++b)
    blocks[b] = GatherBlock<T>{idx[b], idx_bits, n_src[b], fanout[b], (T*)out[b], ld_out[b], nullptr};
  return gather_reduce_impl<T>(table, ld, n_table_rows, F, reduce, blocks, n_blocks, st, sh);
}

int gather_reduce_multi_split(const float* table, int64_t ld_table, int64_t n_table_rows, int32_t F, int reduce,
                              int32_t n_blocks, const void* const* idx_host, int idx_bits, const int64_t* n_src_host,
                              const int32_t* fanout_host, void* const* out_hi_host, const int64_t* ld_out_host,
                              const int64_t* lo_off_host, cudaStream_t st, const gnn_sharded_table* sh = nullptr) {
  GNN_REQUIRE(n_blocks >= 0 && n_blocks <= kMaxBlocks, GNN_ERR_UNSUPPORTED, "at most %d blocks per launch", kMaxBlocks);
  GNN_REQUIRE(n_blocks == 0 || (idx_host && n_src_host && fanout_host && out_hi_host && ld_out_host && lo_off_host),
              GNN_ERR_BAD_ARG, "null block array");
  GatherBlock<float> blocks[kMaxBlocks];
  for (int b = 0; b < n_blocks; ++b) {
    blocks[b] = GatherBlock<float>{idx_host[b], idx_bits, n_src_host[b], fanout_host[b], (float*)out_hi_host[b],
                                   ld_out_host[b], nullptr};
    blocks[b].split = 1;
    blocks[b].lo_off = lo_off_host[b];
  }
  return gather_reduce_impl<float>(table, ld_table, n_table_rows, F, reduce, blocks, n_blocks, st, sh);
}

__global__ void __launch_bounds__(256) bwd_dense_kernel(const float* __restrict__ d_out, int64_t ld,
                                                        const int32_t* __restrict__ argmax, int64_t n_src, int fanout,
                                                        int F, float scale, float* __restrict__ d_neigh) {
  const int64_t total = n_src * (int64_t)fanout * F;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
    const int f = (int)(p % F);
    const int64_t ik = p / F;
    const int k = (int)(ik % fanout);
    const int64_t i = ik / fanout;
    const float g = __ldg(d_out + i * ld + f);
    float v;
    if (argmax) v = (__ldg(argmax + i * ld + f) == k) ? g : 0.f;
    else v = g * scale;
    d_neigh[p] = v;
  }
}

}  // namespace

extern "C" {

int gnn_gather_reduce_f32(const float* table, int64_t ld_table, int64_t n_table_rows, const void* idx, int idx_bits,
                          int64_t n_src, int32_t fanout, int32_t F, int reduce, float* out, int64_t ld_out,
                          int32_t* argmax, gnn_stream_t stream) {
  GatherBlock<float> blk{idx, idx_bits, n_src, fanout, out, ld_out, argmax};
  return gather_reduce_impl<float>(table, ld_table, n_table_rows, F, reduce, &blk, 1, (cudaStream_t)stream);
}

int gnn_gather_reduce_bf16(const void* table, int64_t ld_table, int64_t n_table_rows, const void* idx, int idx_bits,
                           int64_t n_src, int32_t fanout, int32_t F, int reduce, void* out, int64_t ld_out,
                           int32_t* argmax, gnn_stream_t stream) {
  GatherBlock<__nv_bfloat16> blk{idx, idx_bits, n_src, fanout, (__nv_bfloat16*)out, ld_out, argmax};
  return gather_reduce_impl<__nv_bfloat16>((const __nv_bfloat16*)table, ld_table, n_table_rows, F, reduce, &blk, 1,
                                           (cudaStream_t)stream);
}

int gnn_gather_reduce_multi_f32(const float* table, int64_t ld_table, int64_t n_table_rows, int32_t F, int reduce,
                                int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                const int64_t* n_src_host, const int32_t* fanout_host, void* const* out_host,
                                const int64_t* ld_out_host, gnn_stream_t stream) {
  return gather_reduce_multi<float>(table, ld_table, n_table_rows, F, reduce, n_blocks, idx_host, idx_bits, n_src_host,
                                    fanout_host, out_host, ld_out_host, (cudaStream_t)stream);
}

int gnn_gather_reduce_multi_f32_split(const float* table, int64_t ld_table, int64_t n_table_rows, int32_t F, int reduce,
                                      int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                      const int64_t* n_src_host, const int32_t* fanout_host, void* const* out_hi_host,
                                      const int64_t* ld_out_host, const int64_t* lo_off_host, gnn_stream_t stream) {
  return gather_reduce_multi_split(table, ld_table, n_table_rows, F, reduce, n_blocks, idx_host, idx_bits, n_src_host,
                                   fanout_host, out_hi_host, ld_out_host, lo_off_host, (cudaStream_t)stream);
}

int gnn_gather_reduce_multi_sharded_f32(const gnn_sharded_table* table, int64_t ld_table, int32_t F, int reduce,
                                        int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                        const int64_t* n_src_host, const int32_t* fanout_host, void* const* out_host,
                                        const int64_t* ld_out_host, gnn_stream_t stream) {
  GNN_REQUIRE(table, GNN_ERR_BAD_ARG, "null sharded table");
  return gather_reduce_multi<float>(nullptr, ld_table, 0, F, reduce, n_blocks, idx_host, idx_bits, n_src_host,
                                    fanout_host, out_host, ld_out_host, (cudaStream_t)stream, table);
}

int gnn_gather_reduce_multi_sharded_bf16(const gnn_sharded_table* table, int64_t ld_table, int32_t F, int reduce,
                                         int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                         const int64_t* n_src_host, const int32_t* fanout_host, void* const* out_host,
                                         const int64_t* ld_out_host, gnn_stream_t stream) {
  GNN_REQUIRE(table, GNN_ERR_BAD_ARG, "null sharded table");
  return gather_reduce_multi<__nv_bfloat16>(nullptr, ld_table, 0, F, reduce, n_blocks, idx_host, idx_bits, n_src_host,
                                            fanout_host, out_host, ld_out_host, (cudaStream_t)stream, table);
}

int gnn_gather_reduce_multi_sharded_f32_split(const gnn_sharded_table* table, int64_t ld_table, int32_t F, int reduce,
                                              int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                              const int64_t* n_src_host, const int32_t* fanout_host,
                                              void* const* out_hi_host, const int64_t* ld_out_host,
                                              const int64_t* lo_off_host, gnn_stream_t stream) {
  GNN_REQUIRE(table, GNN_ERR_BAD_ARG, "null sharded table");
  return gather_reduce_multi_split(nullptr, ld_table, 0, F, reduce, n_blocks, idx_host, idx_bits, n_src_host,
                                   fanout_host, out_hi_host, ld_out_host, lo_off_host, (cudaStream_t)stream, table);
}

int gnn_gather_reduce_multi_bf16(const void* table, int64_t ld_table, int64_t n_table_rows, int32_t F, int reduce,
                                 int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                 const int64_t* n_src_host, const int32_t* fanout_host, void* const* out_host,
                                 const int64_t* ld_out_host, gnn_stream_t stream) {
  return gather_reduce_multi<__nv_bfloat16>((const __nv_bfloat16*)table, ld_table, n_table_rows, F, reduce, n_blocks,
                                            idx_host, idx_bits, n_src_host, fanout_host, out_host, ld_out_host,
                                            (cudaStream_t)stream);
}

int gnn_gather_reduce_typed_f32(const float* table, int64_t ld_row, int64_t n_nodes, int32_t n_types, const void* idx,
                                int idx_bits, int64_t n_src, int32_t fanout, int32_t F, int reduce, float* out,
                                int64_t ld_out, gnn_stream_t stream) {
  GNN_REQUIRE(n_src >= 0 && n_nodes >= 0 && F >= 0, GNN_ERR_BAD_ARG, "negative size");
  GNN_REQUIRE(n_types > 0 && fanout > 0, GNN_ERR_BAD_ARG, "n_types and fanout must be positive");
  GNN_REQUIRE(reduce == GNN_REDUCE_MEAN || reduce == GNN_REDUCE_SUM, GNN_ERR_BAD_ARG,
              "typed gather supports sum and mean (GATNE_Pytorch/models/GATNE.py:72-77 raises otherwise)");
  if (n_src == 0 || F == 0) return GNN_OK;
  GNN_REQUIRE(table && idx && out, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(idx_bits == 32 || idx_bits == 64, GNN_ERR_BAD_ARG, "idx_bits must be 32 or 64");
  GNN_REQUIRE(ld_row >= F && ld_out >= F, GNN_ERR_BAD_ARG, "leading dimension smaller than F");
  GNN_REQUIRE(n_nodes * (int64_t)n_types < 0x7fffffffLL, GNN_ERR_UNSUPPORTED, "n_nodes * n_types does not fit int32");
  RowArgs<float> r{};
  r.rowptr = nullptr;
  r.fanout = fanout;
  r.col32 = idx_bits == 32 ? (const int32_t*)idx : nullptr;
  r.col64 = idx_bits == 64 ? (const int64_t*)idx : nullptr;
  r.val = nullptr;
  r.src_div = 0;
  r.src_mul = n_types;
  r.scale = (reduce == GNN_REDUCE_MEAN) ? 1.0f / (float)fanout : 1.0f;
  r.n_src_rows = (int32_t)(n_nodes * (int64_t)n_types);
  r.X = table;
  r.ldx = ld_row;
  r.Y = out;
  r.ldy = ld_out;
  r.n_rows = n_src * (int64_t)n_types;
  r.F = F;
  r.skip_deg_gt = 0;
  r.argmax = nullptr;
  return launch_row_reduce<float, 0>(r, (cudaStream_t)stream);
}

int gnn_gather_reduce_bwd_f32(const int64_t* rowptr_t, const int32_t* pos_t, int64_t n_table_rows, int32_t fanout,
                              float scale, const float* d_out, int64_t ld_dout, float* d_table, int64_t ld_dtable,
                              int32_t F, gnn_stream_t stream) {
  GNN_REQUIRE(n_table_rows >= 0 && F >= 0 && fanout > 0, GNN_ERR_BAD_ARG, "bad size");
  if (n_table_rows == 0 || F == 0) return GNN_OK;
  GNN_REQUIRE(rowptr_t && pos_t && d_out && d_table, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(ld_dout >= F && ld_dtable >= F, GNN_ERR_BAD_ARG, "leading dimension smaller than F");
  RowArgs<float> r{};
  r.rowptr = rowptr_t;
  r.fanout = 0;
  r.col32 = pos_t;
  r.col64 = nullptr;
  r.val = nullptr;
  r.src_div = fanout;
  r.scale = scale;
  r.X = d_out;
  r.ldx = ld_dout;
  r.Y = d_table;
  r.ldy = ld_dtable;
  r.n_rows = n_table_rows;
  r.F = F;
  r.skip_deg_gt = 0;
  r.argmax = nullptr;
  return launch_row_reduce<float, 0>(r, (cudaStream_t)stream);
}

int gnn_gather_reduce_bwd_dense_f32(const float* d_out, int64_t ld_dout, const int32_t* argmax, int64_t n_src,
                                    int32_t fanout, int32_t F, float scale, float* d_neigh, gnn_stream_t stream) {
  GNN_REQUIRE(n_src >= 0 && fanout > 0 && F >= 0, GNN_ERR_BAD_ARG, "bad size");
  if (n_src == 0 || F == 0) return GNN_OK;
  GNN_REQUIRE(d_out && d_neigh, GNN_ERR_BAD_ARG, "null pointer");
  const int64_t total = n_src * (int64_t)fanout * F;
  int64_t grid = (total + 255) / 256;
  const int64_t cap = (int64_t)num_sms() * 16;
  grid = grid > cap ? cap : grid;
  bwd_dense_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(d_out, ld_dout, argmax, n_src, fanout, F, scale,
                                                                   d_neigh);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

}  // extern "C"
