// Shared device/host helpers for the sm_100a message-passing kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>
#include "../../include/gnn_b200.h"

namespace gnn {

// ---- error reporting across the C ABI (never throw, never abort) -------------
void set_error(const char* fmt, ...);
int num_sms();
int tuning(const char* key, int dflt);
extern std::atomic<int64_t> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

#define GNN_REQUIRE(cond, status, ...)            \
  do {                                            \
    if (!(cond)) {                                \
      ::gnn::set_error(__VA_ARGS__);              \
      return (status);                            \
    }                                             \
  } while (0)

#define GNN_CUDA(call)                                                                   \
  do {                                                                                   \
    cudaError_t e__ = (call);                                                            \
    if (e__ != cudaSuccess) {                                                            \
      ::gnn::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return GNN_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

#define GNN_LAUNCH_CHECK()                                                               \
  do {                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                \
    if (e__ != cudaSuccess) {                                                            \
      ::gnn::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), __FILE__, __LINE__); \
      return GNN_ERR_CUDA;                                                               \
    }                                                                                    \
    ::gnn::count_launch();                                                               \
  } while (0)

inline bool aligned_to(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }
inline size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- vector loads: VEC elements of T -> VEC floats ----------------------------
template <typename T, int VEC>
struct VecIO;

template <>
struct VecIO<float, 1> {
  static __device__ __forceinline__ void load(const float* p, float (&o)[1]) { o[0] = __ldg(p); }
  static __device__ __forceinline__ void store(float* p, const float (&v)[1]) { p[0] = v[0]; }
};
template <>
struct VecIO<float, 2> {
  static __device__ __forceinline__ void load(const float* p, float (&o)[2]) {
    float2 v = __ldg(reinterpret_cast<const float2*>(p));
    o[0] = v.x; o[1] = v.y;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[2]) {
    *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
  }
};
template <>
struct VecIO<float, 4> {
  static __device__ __forceinline__ void load(const float* p, float (&o)[4]) {
    float4 v = __ldg(reinterpret_cast<const float4*>(p));
    o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};

__device__ __forceinline__ void bf16x2_to_f32(uint32_t w, float& a, float& b) {
  a = __uint_as_float(w << 16);
  b = __uint_as_float(w & 0xffff0000u);
}
__device__ __forceinline__ uint32_t f32_to_bf16x2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
template <>
struct VecIO<__nv_bfloat16, 1> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&o)[1]) {
    unsigned short u = __ldg(reinterpret_cast<const unsigned short*>(p));
    o[0] = __uint_as_float(((uint32_t)u) << 16);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[1]) { p[0] = __float2bfloat16_rn(v[0]); }
};
template <>
struct VecIO<__nv_bfloat16, 2> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&o)[2]) {
    uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p));
    bf16x2_to_f32(w, o[0], o[1]);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[2]) {
    *reinterpret_cast<uint32_t*>(p) = f32_to_bf16x2(v[0], v[1]);
  }
};
template <>
struct VecIO<__nv_bfloat16, 4> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&o)[4]) {
    uint2 w = __ldg(reinterpret_cast<const uint2*>(p));
    bf16x2_to_f32(w.x, o[0], o[1]);
    bf16x2_to_f32(w.y, o[2], o[3]);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[4]) {
    *reinterpret_cast<uint2*>(p) = make_uint2(f32_to_bf16x2(v[0], v[1]), f32_to_bf16x2(v[2], v[3]));
  }
};
template <>
struct VecIO<__nv_bfloat16, 8> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&o)[8]) {
    uint4 w = __ldg(reinterpret_cast<const uint4*>(p));
    bf16x2_to_f32(w.x, o[0], o[1]);
    bf16x2_to_f32(w.y, o[2], o[3]);
    bf16x2_to_f32(w.z, o[4], o[5]);
    bf16x2_to_f32(w.w, o[6], o[7]);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[8]) {
    *reinterpret_cast<uint4*>(p) = make_uint4(f32_to_bf16x2(v[0], v[1]), f32_to_bf16x2(v[2], v[3]),
                                              f32_to_bf16x2(v[4], v[5]), f32_to_bf16x2(v[6], v[7]));
  }
};

// The first n columns of a VEC-wide vector of a row (n counts from p to the row's F): a whole vector when it lies
// inside the F columns, else element by element.  A row's last, partial vector thus never touches the caller's
// columns past F (a padded or sliced output's neighbours), and the accumulate load reads none of them.
template <typename T, int VEC>
__device__ __forceinline__ void store_cols(T* p, const float (&v)[VEC], int n) {
  if (n >= VEC) {
    VecIO<T, VEC>::store(p, v);
    return;
  }
#pragma unroll
  for (int i = 0; i < VEC; ++i)
    if (i < n) {
      const float o[1] = {v[i]};
      VecIO<T, 1>::store(p + i, o);
    }
}
template <typename T, int VEC>
__device__ __forceinline__ void load_cols(const T* p, float (&v)[VEC], int n) {
  if (n >= VEC) {
    VecIO<T, VEC>::load(p, v);
    return;
  }
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    float o[1] = {0.f};
    if (i < n) VecIO<T, 1>::load(p + i, o);
    v[i] = o[0];
  }
}

// ---- raw (still packed) vector staging: keeps bf16 rows at half the registers while the
// gathers are in flight; unpacked only when they are consumed --------------------------------
template <typename T, int VEC>
struct VecRaw {
  static constexpr int W = (sizeof(T) * VEC + 3) / 4;  // 32-bit words
  uint32_t w[W];
};
template <typename T, int VEC>
__device__ __forceinline__ VecRaw<T, VEC> load_raw(const T* p) {
  VecRaw<T, VEC> r;
  constexpr int B = (int)sizeof(T) * VEC;
  if constexpr (B == 16) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
    r.w[0] = v.x; r.w[1] = v.y; r.w[2] = v.z; r.w[3] = v.w;
  } else if constexpr (B == 8) {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
    r.w[0] = v.x; r.w[1] = v.y;
  } else if constexpr (B == 4) {
    r.w[0] = __ldg(reinterpret_cast<const uint32_t*>(p));
  } else {
    r.w[0] = __ldg(reinterpret_cast<const unsigned short*>(p));
  }
  return r;
}
template <typename T, int VEC>
__device__ __forceinline__ VecRaw<T, VEC> zero_raw() {
  VecRaw<T, VEC> r;
#pragma unroll
  for (int i = 0; i < VecRaw<T, VEC>::W; ++i) r.w[i] = 0u;
  return r;
}
template <typename T, int VEC>
__device__ __forceinline__ void unpack_raw(const VecRaw<T, VEC>& r, float (&o)[VEC]) {
  if constexpr (sizeof(T) == 4) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) o[i] = __uint_as_float(r.w[i]);
  } else if constexpr (VEC == 1) {
    o[0] = __uint_as_float(r.w[0] << 16);
  } else {
#pragma unroll
    for (int i = 0; i < VEC / 2; ++i) bf16x2_to_f32(r.w[i], o[2 * i], o[2 * i + 1]);
  }
}

// ---- mbarrier + 1-D TMA bulk copy (cp.async.bulk -> SASS UBLKCP) -------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// global -> shared bulk copy; size and both addresses must be multiples of 16 bytes.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// shared -> global bulk copy (TMA store, completes through the bulk async-group mechanism);
// size and both addresses must be multiples of 16 bytes.  The destination may be peer memory.
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N of this thread's bulk groups still READ their shared-memory source
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// wait until at most N of this thread's bulk groups are incomplete (writes performed)
template <int N>
__device__ __forceinline__ void bulk_wait_group() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ float elu1(float x) { return x > 0.f ? x : expm1f(x); }

}  // namespace gnn
