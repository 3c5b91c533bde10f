// Multi-GPU halo exchange over NVLink peer memory (SURVEY.md §8e).
// One process per GPU.  Halo buffers and arrival flags are plain cudaMalloc allocations exported
// with CUDA IPC so that every rank can map every peer's buffer.  The reference has no multi-GPU path
// for message passing (only nn.DataParallel, HAN/train_utils/train_eval.py:46); this is new.
//
//   gnn_halo_push    fused pack + transfer: feature rows of the local X go straight into the owning
//                    peers' halo buffers, no staging buffer.  Two movers:
//       TMA mover    (halo_move_tma_kernel) every warp is an independent mover with a ring of
//                    shared-memory stages; lanes issue one bulk gather (cp.async.bulk global->shared,
//                    SASS UBLKCP.S.G) per row, and when the stage's mbarrier completes ONE lane issues
//                    ONE bulk store (shared -> peer global, UBLKCP.G.S) for the whole stage — rows a
//                    peer receives are consecutive in its halo, so a stage leaves as one NVLink write.
//                    No row passes through registers or the load/store unit, so the mover can sit on
//                    every SM next to the SpMM CTAs without competing for the LSU.
//       vector mover (halo_push_kernel) warp per row, 128-bit loads/stores; the fallback for rows that
//                    are not 16-byte multiples or non-contiguous destination rows.
//                    Measured (r02, 2 GPUs, papers100M-shaped, exchange alone): both movers are bound
//                    by remote-write issue per SM — 22 GB/s (vector) / 26 GB/s (TMA) per SM — so NVLink
//                    rate needs >= 30 SMs' worth of issue either way; the TMA mover gets it from one
//                    warp on EVERY SM instead of taking 32 SMs away from the HBM-bound SpMM.
//   gnn_peer_signal / gnn_peer_wait   per-peer arrival flags (monotonic counters in peer memory):
//                    a rank signals each peer after its wave of rows has been pushed (stream order:
//                    the mover kernel has completed), and the consumer of a wave waits only for that
//                    wave's flags — no collective barrier on the data path.
//   gnn_peer_reduce_rows_f32   out[r] = relu?(src[0][row_lo + r] + ... + src[P-1][row_lo + r]): the ordered
//                    cross-rank sum of P row buffers (this rank's and the peers' mappings), read over NVLink,
//                    added left to right in fp32 — every rank that reduces a row gets the same bits.
#include "common.cuh"

using namespace gnn;

namespace {

constexpr int kMaxPeers = 16;

struct MoveArgs {
  const unsigned char* X;
  int64_t ldx_bytes;
  int32_t row_bytes;              // bytes moved per row
  int32_t rows_per_stage;         // TMA mover: rows per ring stage (<= 32)
  const int32_t* send_rows;       // nullable: identity (row k of the segment is local row seg_begin + k)
  int64_t seg_begin[kMaxPeers];   // slot s: first entry of send_rows (or first local row) of the segment
  int64_t seg_rows[kMaxPeers];    // slot s: rows to send
  int64_t cum[kMaxPeers + 1];     // slot s: TMA mover: first chunk id; vector mover: first row position
  unsigned char* dst[kMaxPeers];  // slot s: first destination row (peer halo base + dst_row * ld_dst)
  int64_t ld_dst_bytes;
  int32_t n_slots;
};

// ---- vector mover: one warp per sent row, UNROLL rows in flight per warp --------------------
// The sent-row ids of the NEXT iteration are loaded before the rows of this one are stored: without
// this prefetch every iteration was a chain of two dependent DRAM round trips (id, then row).
template <typename V, int UNROLL>
__global__ void halo_push_kernel(const MoveArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t total = a.cum[a.n_slots];
  const int nv = a.row_bytes / (int)sizeof(V);
  auto src_row = [&](int64_t k, int& slot) -> int64_t {
    slot = 0;
    while (slot + 1 < a.n_slots && k >= a.cum[slot + 1]) ++slot;
    const int64_t i = a.seg_begin[slot] + (k - a.cum[slot]);
    return a.send_rows ? (int64_t)__ldg(a.send_rows + i) : i;
  };
  int64_t rid[UNROLL], rid_next[UNROLL];
  int sl[UNROLL], sl_next[UNROLL];
#pragma unroll
  for (int u = 0; u < UNROLL; ++u) {
    const int64_t k = w * UNROLL + u;
    sl[u] = 0;
    rid[u] = (k < total) ? src_row(k, sl[u]) : -1;
  }
  for (int64_t k0 = w * UNROLL; k0 < total; k0 += nw * UNROLL) {
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const int64_t kn = k0 + nw * UNROLL + u;
      sl_next[u] = 0;
      rid_next[u] = (kn < total) ? src_row(kn, sl_next[u]) : -1;
    }
    const V* src[UNROLL];
    V* dst[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const int64_t k = k0 + u;
      src[u] = nullptr;
      dst[u] = nullptr;
      if (k < total) {
        src[u] = reinterpret_cast<const V*>(a.X + rid[u] * a.ldx_bytes);
        dst[u] = reinterpret_cast<V*>(a.dst[sl[u]] + (k - a.cum[sl[u]]) * a.ld_dst_bytes);
      }
    }
    for (int c = lane; c < nv; c += 32) {
      V v[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u)
        if (src[u]) v[u] = __ldg(src[u] + c);
#pragma unroll
      for (int u = 0; u < UNROLL; ++u)
        if (dst[u]) dst[u][c] = v[u];
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      rid[u] = rid_next[u];
      sl[u] = sl_next[u];
    }
  }
}

// ---- TMA mover ----------------------------------------------------------------------------------
constexpr int kTmaStages = 3;

__global__ void halo_move_tma_kernel(const MoveArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_warps = blockDim.x >> 5;
  const int R = a.rows_per_stage;
  const int stage_bytes = R * a.row_bytes;
  unsigned char* ring = smem + (size_t)warp * kTmaStages * stage_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)n_warps * kTmaStages * stage_bytes) + warp * kTmaStages;
  if (lane == 0) {
    for (int s = 0; s < kTmaStages; ++s) mbar_init(full + s, 1);
    mbar_fence_init();
  }
  __syncwarp();
  const int64_t n_chunks = a.cum[a.n_slots];
  const int64_t w = (int64_t)blockIdx.x * n_warps + warp;
  const int64_t nw = (int64_t)gridDim.x * n_warps;
  // chunk id -> (slot, first row of the chunk within the slot's segment)
  auto locate = [&](int64_t c, int& slot, int64_t& row0) {
    slot = 0;
    while (slot + 1 < a.n_slots && c >= a.cum[slot + 1]) ++slot;
    row0 = (c - a.cum[slot]) * R;
  };
  auto load_id = [&](int64_t c) -> int64_t {
    if (c >= n_chunks) return -1;
    int slot;
    int64_t row0;
    locate(c, slot, row0);
    const int64_t r = row0 + lane;
    if (lane >= R || r >= a.seg_rows[slot]) return -1;
    const int64_t i = a.seg_begin[slot] + r;
    return a.send_rows ? (int64_t)__ldg(a.send_rows + i) : i;
  };
  // gathers of chunk c into ring stage `stg` (ids already in `rid_c`)
  auto issue = [&](int64_t c, int64_t rid_c, int stg) {
    int slot;
    int64_t row0;
    locate(c, slot, row0);
    const int64_t left = a.seg_rows[slot] - row0;
    const int rows = (int)(left < R ? left : R);
    if (lane == 0) mbar_arrive_expect_tx(full + stg, (uint32_t)rows * (uint32_t)a.row_bytes);
    __syncwarp();
    if (lane < rows)
      bulk_g2s(ring + (size_t)stg * stage_bytes + (size_t)lane * a.row_bytes, a.X + rid_c * a.ldx_bytes,
               (uint32_t)a.row_bytes, full + stg);
  };
  // Software pipeline: the gathers of the next kTmaStages-1 chunks are in flight while chunk k is stored.
  constexpr int P = kTmaStages - 1;
  int64_t rid_ahead = load_id(w);
  int fill_stage = 0;
#pragma unroll
  for (int k = 0; k < P; ++k) {
    const int64_t c = w + (int64_t)k * nw;
    if (c < n_chunks) issue(c, rid_ahead, fill_stage);
    rid_ahead = load_id(c + nw);
    fill_stage = (fill_stage + 1 == kTmaStages) ? 0 : fill_stage + 1;
  }
  int stage = 0;
  uint32_t parity = 0;
  for (int64_t c = w; c < n_chunks; c += nw) {
    int slot;
    int64_t row0;
    locate(c, slot, row0);
    const int64_t left = a.seg_rows[slot] - row0;
    const int rows = (int)(left < R ? left : R);
    mbar_wait(full + stage, parity);
    if (lane == 0) {
      fence_proxy_async_smem();
      bulk_s2g(a.dst[slot] + row0 * a.ld_dst_bytes, ring + (size_t)stage * stage_bytes,
               (uint32_t)rows * (uint32_t)a.row_bytes);
      bulk_commit_group();
    }
    // refill the stage chunk c - nw was stored from: that store must have read it (at most the store just
    // committed may still be reading)
    const int64_t cf = c + (int64_t)P * nw;
    if (cf < n_chunks) {
      if (lane == 0) bulk_wait_group_read<1>();
      __syncwarp();
      issue(cf, rid_ahead, fill_stage);
    }
    rid_ahead = load_id(cf + nw);
    fill_stage = (fill_stage + 1 == kTmaStages) ? 0 : fill_stage + 1;
    if (++stage == kTmaStages) {
      stage = 0;
      parity ^= 1u;
    }
  }
  if (lane == 0) bulk_wait_group<0>();  // every store performed before the kernel (and the signal after it) ends
  __syncwarp();
}

// ---- TMA mover, all waves in ONE launch, arrival flags raised from inside ------------------------
// The per-wave launches of the mover leave a tail (the last chunks of a wave drain while most warps
// idle) and a launch + signal gap between waves: measured at 8 GPUs the exchange alone ran at 506 GB/s
// in 4 waves against 575 GB/s in one.  Here every warp walks the chunks of ALL waves in order (segments
// sorted by wave, then rotated peer); when a warp crosses from wave w to a later wave (or runs out of
// chunks) it waits for its own bulk stores, fences and counts itself on wave_done[w]; the LAST warp of
// the grid to do so raises wave w's flag on every peer.  Warps never wait for each other.
struct WaveMoveArgs {
  const unsigned char* X;
  int64_t ldx_bytes;
  int32_t row_bytes;
  int32_t rows_per_stage;
  const int32_t* send_rows;
  const int64_t* seg;   // [n_segs][5] device table: src_begin, rows, destination address, first chunk id, wave
  int32_t n_segs;
  int32_t n_waves;
  int64_t n_chunks;
  uint32_t* wave_done;  // [n_waves], zeroed before the launch
  uint32_t* flag[kMaxPeers];
  int32_t n_peers;
  int32_t my_slot;
  uint32_t flag_base;   // wave w announces flag_base + w + 1
};

__global__ void halo_move_tma_waves_kernel(const WaveMoveArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_warps = blockDim.x >> 5;
  const int R = a.rows_per_stage;
  const int stage_bytes = R * a.row_bytes;
  unsigned char* ring = smem + (size_t)warp * kTmaStages * stage_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)n_warps * kTmaStages * stage_bytes) + warp * kTmaStages;
  if (lane == 0) {
    for (int s = 0; s < kTmaStages; ++s) mbar_init(full + s, 1);
    mbar_fence_init();
  }
  __syncwarp();
  const int64_t n_chunks = a.n_chunks;
  const int64_t w = (int64_t)blockIdx.x * n_warps + warp;
  const int64_t nw = (int64_t)gridDim.x * n_warps;
  // segment of chunk c: chunk ids only grow along a warp's walk, so a galloping step from the previous segment
  // and a binary search inside the bracket (an interleaved table has tens of thousands of short segments and a
  // warp skips gridDim * warps chunks per step)
  auto seek = [&](int& slot, int64_t c) {
    int lo = slot, step = 1;
    int hi = lo + 1;
    while (hi < a.n_segs && c >= __ldg(a.seg + hi * 5 + 3)) {
      lo = hi;
      hi += step;
      step <<= 1;
    }
    if (hi > a.n_segs) hi = a.n_segs;
    // invariant: first chunk of lo <= c, and (hi == n_segs or first chunk of hi > c)
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (c >= __ldg(a.seg + mid * 5 + 3)) lo = mid; else hi = mid;
    }
    slot = lo;
  };
  int slot_l = 0, slot_i = 0, slot_s = 0;
  auto load_id = [&](int64_t c) -> int64_t {
    if (c >= n_chunks) return -1;
    seek(slot_l, c);
    const int64_t r = (c - __ldg(a.seg + slot_l * 5 + 3)) * R + lane;
    if (lane >= R || r >= __ldg(a.seg + slot_l * 5 + 1)) return -1;
    const int64_t i = __ldg(a.seg + slot_l * 5) + r;
    return a.send_rows ? (int64_t)__ldg(a.send_rows + i) : i;
  };
  auto issue = [&](int64_t c, int64_t rid_c, int stg) {
    seek(slot_i, c);
    const int64_t left = __ldg(a.seg + slot_i * 5 + 1) - (c - __ldg(a.seg + slot_i * 5 + 3)) * R;
    const int rows = (int)(left < R ? left : R);
    if (lane == 0) mbar_arrive_expect_tx(full + stg, (uint32_t)rows * (uint32_t)a.row_bytes);
    __syncwarp();
    if (lane < rows)
      bulk_g2s(ring + (size_t)stg * stage_bytes + (size_t)lane * a.row_bytes, a.X + rid_c * a.ldx_bytes,
               (uint32_t)a.row_bytes, full + stg);
  };
  // this warp is done with wave wv: its stores have been performed; the last warp of the grid signals
  auto arrive = [&](int wv) {
    if (lane == 0) {
      bulk_wait_group<0>();
      asm volatile("fence.proxy.async;" ::: "memory");
      __threadfence_system();
      const uint32_t old = atomicAdd(a.wave_done + wv, 1u);
      if (old == (uint32_t)(nw - 1)) {
        __threadfence_system();
        for (int q = 0; q < a.n_peers; ++q)
          if (q != a.my_slot && a.flag[q])
            asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(a.flag[q] + a.my_slot),
                         "r"(a.flag_base + (uint32_t)wv + 1u)
                         : "memory");
      }
    }
    __syncwarp();
  };
  constexpr int P = kTmaStages - 1;
  int64_t rid_ahead = load_id(w);
  int fill_stage = 0;
#pragma unroll
  for (int k = 0; k < P; ++k) {
    const int64_t c = w + (int64_t)k * nw;
    if (c < n_chunks) issue(c, rid_ahead, fill_stage);
    rid_ahead = load_id(c + nw);
    fill_stage = (fill_stage + 1 == kTmaStages) ? 0 : fill_stage + 1;
  }
  int stage = 0, cur_wave = 0;
  uint32_t parity = 0;
  for (int64_t c = w; c < n_chunks; c += nw) {
    seek(slot_s, c);
    const int wave_c = (int)__ldg(a.seg + slot_s * 5 + 4);
    for (; cur_wave < wave_c; ++cur_wave) arrive(cur_wave);
    const int64_t row0 = (c - __ldg(a.seg + slot_s * 5 + 3)) * R;
    const int64_t left = __ldg(a.seg + slot_s * 5 + 1) - row0;
    const int rows = (int)(left < R ? left : R);
    mbar_wait(full + stage, parity);
    if (lane == 0) {
      fence_proxy_async_smem();
      bulk_s2g(reinterpret_cast<unsigned char*>(__ldg(a.seg + slot_s * 5 + 2)) + row0 * a.row_bytes,
               ring + (size_t)stage * stage_bytes, (uint32_t)rows * (uint32_t)a.row_bytes);
      bulk_commit_group();
    }
    const int64_t cf = c + (int64_t)P * nw;
    if (cf < n_chunks) {
      if (lane == 0) bulk_wait_group_read<1>();
      __syncwarp();
      issue(cf, rid_ahead, fill_stage);
    }
    rid_ahead = load_id(cf + nw);
    fill_stage = (fill_stage + 1 == kTmaStages) ? 0 : fill_stage + 1;
    if (++stage == kTmaStages) {
      stage = 0;
      parity ^= 1u;
    }
  }
  for (; cur_wave < a.n_waves; ++cur_wave) arrive(cur_wave);
}

// ---- arrival flags ------------------------------------------------------------------------------
struct SignalArgs {
  uint32_t* flag[kMaxPeers];  // peer q's flag array (mapped peer memory); slot written = my_slot
  int32_t n_peers;
  int32_t my_slot;
  int32_t skip;
  uint32_t value;
};

__global__ void peer_signal_kernel(const SignalArgs a) {
  const int q = threadIdx.x;
  if (q >= a.n_peers || q == a.skip || a.flag[q] == nullptr) return;
  // stream order: the mover kernel that wrote the rows has completed; the fence orders this store
  // behind every write this GPU has made visible so far
  __threadfence_system();
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(a.flag[q] + a.my_slot), "r"(a.value) : "memory");
}

__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// One thread per peer slot spins until flags[q] has reached `value` (wrap-safe).  Bounded: after
// timeout_ns the kernel gives up and sets *status = 1 + q (the caller checks it after the step) —
// a lost peer must not hang the GPU.
__global__ void peer_wait_kernel(const uint32_t* flags, int n_slots, int skip, uint32_t value, uint32_t* status,
                                 uint64_t timeout_ns) {
  const int q = threadIdx.x;
  if (q >= n_slots || q == skip) return;
  const uint64_t t0 = globaltimer_ns();
  for (;;) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + q) : "memory");
    if ((int32_t)(v - value) >= 0) break;
    if (globaltimer_ns() - t0 > timeout_ns) {
      if (status) atomicMax(status, 1u + (uint32_t)q);
      break;
    }
    __nanosleep(200);
  }
}

// ---- ordered row reduction over P sources -------------------------------------------------------
struct ReduceArgs {
  const float* src[kMaxPeers];
  int32_t n_src;
  int64_t ld_src;
  int64_t row_lo;
  int64_t n_rows;
  int32_t F;
  int32_t n_vec;   // float4 columns per row (0 on the scalar path)
  int32_t per_row; // work items per row: n_vec + (F - 4 * n_vec) scalar tail columns
  float* out;
  int64_t ld_out;
  int32_t relu;
};

// One thread per (row, float4 column) or (row, tail column).  The P sources are added in slot order, starting from
// src[0]: ((s0 + s1) + s2) + ..., with no reassociation (plain adds, nothing to contract).
__global__ void peer_reduce_rows_kernel(const ReduceArgs a) {
  const int64_t total = a.n_rows * a.per_row;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / a.per_row;
    const int c = (int)(i - r * a.per_row);
    const int64_t s_off = (a.row_lo + r) * a.ld_src;
    float* o = a.out + r * a.ld_out;
    if (c < a.n_vec) {
      float4 acc = __ldcg(reinterpret_cast<const float4*>(a.src[0] + s_off) + c);
      for (int q = 1; q < a.n_src; ++q) {
        const float4 v = __ldcg(reinterpret_cast<const float4*>(a.src[q] + s_off) + c);
        acc.x += v.x;
        acc.y += v.y;
        acc.z += v.z;
        acc.w += v.w;
      }
      if (a.relu) {
        acc.x = acc.x < 0.f ? 0.f : acc.x;
        acc.y = acc.y < 0.f ? 0.f : acc.y;
        acc.z = acc.z < 0.f ? 0.f : acc.z;
        acc.w = acc.w < 0.f ? 0.f : acc.w;
      }
      reinterpret_cast<float4*>(o)[c] = acc;
    } else {
      const int col = 4 * a.n_vec + (c - a.n_vec);
      float acc = __ldcg(a.src[0] + s_off + col);
      for (int q = 1; q < a.n_src; ++q) acc += __ldcg(a.src[q] + s_off + col);
      if (a.relu) acc = acc < 0.f ? 0.f : acc;
      o[col] = acc;
    }
  }
}

}  // namespace

extern "C" {

int gnn_peer_alloc(size_t bytes, void** dev_ptr, void* ipc_handle_64B_host) {
  GNN_REQUIRE(dev_ptr && ipc_handle_64B_host && bytes > 0, GNN_ERR_BAD_ARG, "bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
  GNN_CUDA(cudaMalloc(dev_ptr, bytes));
  cudaError_t e = cudaMemset(*dev_ptr, 0, bytes);  // arrival flags start at 0
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, *dev_ptr);
  if (e != cudaSuccess) {
    cudaFree(*dev_ptr);
    *dev_ptr = nullptr;
    set_error("cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    return GNN_ERR_CUDA;
  }
  memcpy(ipc_handle_64B_host, &h, 64);
  return GNN_OK;
}

int gnn_peer_open(const void* ipc_handle_64B_host, void** dev_ptr) {
  GNN_REQUIRE(dev_ptr && ipc_handle_64B_host, GNN_ERR_BAD_ARG, "bad argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle_64B_host, 64);
  GNN_CUDA(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return GNN_OK;
}

int gnn_peer_close(void* dev_ptr) {
  if (!dev_ptr) return GNN_OK;
  GNN_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return GNN_OK;
}

int gnn_peer_free(void* dev_ptr) {
  if (!dev_ptr) return GNN_OK;
  GNN_CUDA(cudaFree(dev_ptr));
  return GNN_OK;
}

int gnn_peer_copy_async(void* dst, const void* src, size_t bytes, gnn_stream_t stream) {
  if (bytes == 0) return GNN_OK;
  GNN_REQUIRE(dst && src, GNN_ERR_BAD_ARG, "null pointer");
  GNN_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return GNN_OK;
}

int gnn_peer_signal(uint32_t* const* peer_flags_host, int32_t n_peers, int32_t my_slot, int32_t skip_peer,
                    uint32_t value, gnn_stream_t stream) {
  GNN_REQUIRE(peer_flags_host && n_peers > 0 && n_peers <= kMaxPeers && my_slot >= 0, GNN_ERR_BAD_ARG, "bad argument");
  SignalArgs a{};
  for (int q = 0; q < n_peers; ++q) a.flag[q] = peer_flags_host[q];
  a.n_peers = n_peers;
  a.my_slot = my_slot;
  a.skip = skip_peer;
  a.value = value;
  peer_signal_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(a);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_peer_wait(const uint32_t* flags, int32_t n_slots, int32_t skip_slot, uint32_t value, uint32_t* status,
                  int64_t timeout_ms, gnn_stream_t stream) {
  GNN_REQUIRE(flags && n_slots > 0 && n_slots <= 32, GNN_ERR_BAD_ARG, "bad argument");
  const uint64_t ns = (uint64_t)(timeout_ms > 0 ? timeout_ms : 10000) * 1000000ull;
  peer_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(flags, n_slots, skip_slot, value, status, ns);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_halo_rows_per_stage(int32_t row_bytes) {
  if (row_bytes <= 0 || row_bytes % 16 != 0 || row_bytes > 16384) return 0;
  const int r = 16384 / row_bytes;
  return r > 32 ? 32 : r;
}

int gnn_halo_push_waves(const void* X, int64_t ldx, int32_t F, int32_t elem_size, const int32_t* send_rows,
                        const int64_t* seg_table_dev, int32_t n_segs, int32_t n_waves, int64_t n_chunks,
                        uint32_t* wave_done_dev, uint32_t* const* peer_flags_host, int32_t n_peers, int32_t my_slot,
                        uint32_t flag_base, const gnn_halo_opts* opts, gnn_stream_t stream) {
  GNN_REQUIRE(n_peers > 0 && n_peers <= kMaxPeers && my_slot >= 0 && my_slot < n_peers, GNN_ERR_BAD_ARG, "bad peers");
  GNN_REQUIRE(!opts || opts->struct_size == (int32_t)sizeof(gnn_halo_opts), GNN_ERR_BAD_ARG,
              "gnn_halo_opts struct_size mismatch (header/library version skew)");
  GNN_REQUIRE(X && wave_done_dev && peer_flags_host && n_waves > 0 && n_waves <= 64 && n_segs >= 0 && n_chunks >= 0,
              GNN_ERR_BAD_ARG, "bad argument");
  GNN_REQUIRE(n_segs == 0 || seg_table_dev, GNN_ERR_BAD_ARG, "null segment table");
  GNN_REQUIRE(elem_size == 2 || elem_size == 4, GNN_ERR_UNSUPPORTED, "elem_size must be 2 or 4");
  GNN_REQUIRE(F > 0 && ldx >= F, GNN_ERR_BAD_ARG, "bad feature width / leading dimension");
  WaveMoveArgs a{};
  a.X = (const unsigned char*)X;
  a.ldx_bytes = ldx * elem_size;
  a.row_bytes = F * elem_size;
  a.rows_per_stage = gnn_halo_rows_per_stage(a.row_bytes);
  GNN_REQUIRE(a.rows_per_stage > 0 && aligned_to(X, 16) && a.ldx_bytes % 16 == 0, GNN_ERR_UNSUPPORTED,
              "the wave mover needs 16-byte-multiple rows (<= 16 KB) and a 16-byte aligned table");
  a.send_rows = send_rows;
  a.seg = seg_table_dev;
  a.n_segs = n_segs;
  a.n_waves = n_waves;
  a.n_chunks = n_segs > 0 ? n_chunks : 0;
  a.wave_done = wave_done_dev;
  for (int q = 0; q < n_peers; ++q) a.flag[q] = peer_flags_host[q];
  a.n_peers = n_peers;
  a.my_slot = my_slot;
  a.flag_base = flag_base;
  cudaStream_t st = (cudaStream_t)stream;
  GNN_CUDA(cudaMemsetAsync(wave_done_dev, 0, (size_t)n_waves * sizeof(uint32_t), st));
  int warps = (opts && opts->warps_per_cta > 0) ? opts->warps_per_cta : 1;
  const size_t per_warp = (size_t)kTmaStages * a.rows_per_stage * a.row_bytes + kTmaStages * 8;
  const int max_warps = (int)((200 * 1024) / per_warp);
  warps = warps > max_warps ? max_warps : warps;
  warps = warps > 32 ? 32 : warps;
  const size_t smem = (size_t)warps * per_warp;
  GNN_CUDA(cudaFuncSetAttribute(halo_move_tma_waves_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t grid = (opts && opts->ctas > 0) ? opts->ctas : num_sms();
  halo_move_tma_waves_kernel<<<(unsigned)(grid < 1 ? 1 : grid), warps * 32, smem, st>>>(a);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_halo_push(const void* X, int64_t ldx, int32_t F, int32_t elem_size, const int32_t* send_rows,
                  const int64_t* seg_begin_host, const int64_t* seg_rows_host, void* const* peer_dst_host,
                  const int64_t* dst_row_host, int64_t ld_dst, int32_t n_peers, const gnn_halo_opts* opts,
                  gnn_stream_t stream) {
  GNN_REQUIRE(n_peers >= 0 && n_peers <= kMaxPeers, GNN_ERR_UNSUPPORTED, "n_peers=%d exceeds %d", n_peers, kMaxPeers);
  if (n_peers == 0) return GNN_OK;
  GNN_REQUIRE(!opts || opts->struct_size == (int32_t)sizeof(gnn_halo_opts), GNN_ERR_BAD_ARG,
              "gnn_halo_opts struct_size mismatch (header/library version skew)");
  GNN_REQUIRE(X && seg_begin_host && seg_rows_host && peer_dst_host && dst_row_host, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(elem_size == 2 || elem_size == 4, GNN_ERR_UNSUPPORTED, "elem_size must be 2 or 4");
  GNN_REQUIRE(F > 0 && ldx >= F && ld_dst >= F, GNN_ERR_BAD_ARG, "bad feature width / leading dimension");
  const int first = opts ? opts->first_peer : 0;
  GNN_REQUIRE(first >= 0 && first < n_peers, GNN_ERR_BAD_ARG, "first_peer out of range");
  MoveArgs a{};
  a.X = (const unsigned char*)X;
  a.ldx_bytes = ldx * elem_size;
  a.row_bytes = F * elem_size;
  a.send_rows = send_rows;
  a.ld_dst_bytes = ld_dst * elem_size;
  bool v16 = aligned_to(X, 16) && a.ldx_bytes % 16 == 0 && a.ld_dst_bytes % 16 == 0 && a.row_bytes % 16 == 0;
  // segments in rotated order (rank r starts with peer r+1: no receiver is hit by every sender at once)
  int ns = 0;
  int64_t total_rows = 0;
  for (int s = 0; s < n_peers; ++s) {
    const int q = (first + s) % n_peers;
    const int64_t rows = seg_rows_host[q];
    GNN_REQUIRE(rows >= 0 && seg_begin_host[q] >= 0 && dst_row_host[q] >= 0, GNN_ERR_BAD_ARG, "negative segment");
    if (rows == 0) continue;
    GNN_REQUIRE(peer_dst_host[q] != nullptr, GNN_ERR_BAD_ARG, "null peer destination %d", q);
    a.seg_begin[ns] = seg_begin_host[q];
    a.seg_rows[ns] = rows;
    a.dst[ns] = (unsigned char*)peer_dst_host[q] + dst_row_host[q] * a.ld_dst_bytes;
    v16 = v16 && aligned_to(a.dst[ns], 16);
    total_rows += rows;
    ++ns;
  }
  a.n_slots = ns;
  if (total_rows == 0) return GNN_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int mover = opts ? opts->mover : 0;
  const bool contiguous = a.ld_dst_bytes == a.row_bytes;
  const bool tma_ok = v16 && contiguous && a.row_bytes <= 16384;
  GNN_REQUIRE(mover != 2 || tma_ok, GNN_ERR_UNSUPPORTED,
              "TMA mover needs 16-byte-multiple rows (<= 16 KB) and contiguous destination rows");
  if ((mover == 0 || mover == 2) && tma_ok) {
    int R = 16384 / a.row_bytes;
    R = R > 32 ? 32 : R;
    a.rows_per_stage = R;
    a.cum[0] = 0;
    for (int s = 0; s < ns; ++s) a.cum[s + 1] = a.cum[s] + (a.seg_rows[s] + R - 1) / R;
    int warps = (opts && opts->warps_per_cta > 0) ? opts->warps_per_cta : 1;
    const size_t per_warp = (size_t)kTmaStages * R * a.row_bytes + kTmaStages * 8;
    const int max_warps = (int)((200 * 1024) / per_warp);
    warps = warps > max_warps ? max_warps : warps;
    warps = warps > 32 ? 32 : warps;
    const size_t smem = (size_t)warps * per_warp;
    // per-device opt-in for > 48 KB of dynamic shared memory (idempotent, cheap)
    GNN_CUDA(cudaFuncSetAttribute(halo_move_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t grid = (opts && opts->ctas > 0) ? opts->ctas : num_sms();
    const int64_t need = (a.cum[ns] + warps - 1) / warps;
    grid = grid > need ? need : grid;
    halo_move_tma_kernel<<<(unsigned)(grid < 1 ? 1 : grid), warps * 32, smem, st>>>(a);
  } else {
    a.cum[0] = 0;
    for (int s = 0; s < ns; ++s) a.cum[s + 1] = a.cum[s] + a.seg_rows[s];
    const int warps = (opts && opts->warps_per_cta > 0) ? (opts->warps_per_cta > 32 ? 32 : opts->warps_per_cta) : 8;
    const size_t smem = (opts && opts->claim_smem_bytes > 0) ? (size_t)opts->claim_smem_bytes : 0;
    int64_t grid = (opts && opts->ctas > 0) ? opts->ctas : num_sms();
    const int64_t need = (total_rows + (int64_t)warps * 4 - 1) / ((int64_t)warps * 4);
    grid = grid > need ? need : grid;
    grid = grid < 1 ? 1 : grid;
    const bool v4 = aligned_to(X, 4) && a.ldx_bytes % 4 == 0 && a.ld_dst_bytes % 4 == 0 && a.row_bytes % 4 == 0;
    if (v16) {
      if (smem > 48 * 1024)
        GNN_CUDA(cudaFuncSetAttribute(halo_push_kernel<uint4, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      halo_push_kernel<uint4, 4><<<(unsigned)grid, warps * 32, smem, st>>>(a);
    } else if (v4) {
      halo_push_kernel<uint32_t, 4><<<(unsigned)grid, warps * 32, smem > 48 * 1024 ? 0 : smem, st>>>(a);
    } else {
      halo_push_kernel<uint16_t, 4><<<(unsigned)grid, warps * 32, smem > 48 * 1024 ? 0 : smem, st>>>(a);
    }
  }
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_peer_reduce_rows_f32(const float* const* src_host, int32_t n_src, int64_t ld_src, int32_t F, int64_t row_lo,
                             int64_t row_hi, float* out, int64_t ld_out, int32_t relu, gnn_stream_t stream) {
  GNN_REQUIRE(src_host && out, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(n_src >= 1 && n_src <= kMaxPeers, GNN_ERR_BAD_ARG, "n_src=%d outside [1, %d]", n_src, kMaxPeers);
  GNN_REQUIRE(F > 0 && ld_src >= F && ld_out >= F, GNN_ERR_BAD_ARG, "bad width / leading dimension");
  GNN_REQUIRE(row_lo >= 0 && row_hi >= row_lo, GNN_ERR_BAD_ARG, "bad row range [%lld, %lld)", (long long)row_lo,
              (long long)row_hi);
  ReduceArgs a{};
  bool v16 = ld_src % 4 == 0 && ld_out % 4 == 0 && aligned_to(out, 16);
  for (int q = 0; q < n_src; ++q) {
    GNN_REQUIRE(src_host[q] != nullptr, GNN_ERR_BAD_ARG, "null pointer (source %d)", q);
    a.src[q] = src_host[q];
    v16 = v16 && aligned_to(src_host[q], 16);
  }
  if (row_hi == row_lo) return GNN_OK;
  a.n_src = n_src;
  a.ld_src = ld_src;
  a.row_lo = row_lo;
  a.n_rows = row_hi - row_lo;
  a.F = F;
  a.n_vec = v16 ? F / 4 : 0;
  a.per_row = a.n_vec + (F - 4 * a.n_vec);
  a.out = out;
  a.ld_out = ld_out;
  a.relu = relu ? 1 : 0;
  const int64_t total = a.n_rows * a.per_row;
  int64_t grid = (total + 255) / 256;
  const int64_t cap = (int64_t)num_sms() * 8;
  grid = grid > cap ? cap : grid;
  peer_reduce_rows_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(a);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

}  // extern "C"
