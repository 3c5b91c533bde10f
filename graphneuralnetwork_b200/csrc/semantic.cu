// HAN semantic attention (SURVEY.md §8 rows a12 / f2), the part around its one GEMM:
//   /root/reference HAN/models/SemanticAttention.py:15-20
//       w    = self.project(z).mean(0)          project = Linear(D,K) -> Tanh -> Linear(K,1,bias=False)
//       beta = softmax(w, dim=0)                over the M metapaths
//       out  = (beta.expand(N,M,1) * z).sum(1)
// The reference materialises tanh(.) [N,M,K], the [N,M,1] projection, beta expanded to [N,M,1] and beta*z [N,M,D].
// Here P = z·W1ᵀ stays a library GEMM and everything after it is two launches forward and two backward:
//   scores      : scores[m] = 1/N Σ_n Σ_k q_k tanh(P[n,m,k] + b_k), and beta = softmax_M(scores) by the last CTA;
//   combine     : out[n,:] = Σ_m beta_m z[n,m,:];
//   combine_bwd : dz[n,m,:] = beta_m dOut[n,:] (the direct term), dbeta_m = Σ_n <dOut_n, z[n,m]>, and the softmax
//                 backward d_scores_m / N by the last CTA;
//   scores_bwd  : dP = d_scores_m/N · q_k (1 - tanh²), dq_k = Σ d_scores_m/N · tanh, db_k = Σ dP — column sums.
// All sums are ordered (per-warp grid-stride order, warps in order inside a CTA, CTAs in order by the last CTA to
// take a ticket): deterministic, no floating-point atomics.  The ticket counter lives in the caller's workspace
// (zero before the first use; every kernel leaves it zero again).
#include "common.cuh"

using namespace gnn;

namespace {

constexpr int kSemThreads = 256;
constexpr int kSemWarps = kSemThreads / 32;
constexpr int kSemMaxM = 32;
constexpr int kSemMaxK = 256;

// every reduction kernel gives a CTA >= 64 nodes (or 64 row steps) of work before a second CTA is used: on small graphs
// (ACM: 3,025 nodes) the serial tail — the last CTA adding the others' partials — stays a few microseconds
int sem_grid_cap() { return num_sms() * 2; }

__device__ inline float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// true in every thread of the LAST CTA to arrive (the partials of all CTAs are then visible)
__device__ inline bool last_cta(unsigned int* counter) {
  __shared__ bool is_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(counter, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}

// per-warp accumulators acc (lane m holds metapath m) -> CTA partial -> (last CTA) tot[m] in shared memory
__device__ inline bool reduce_over_grid_m(float acc, int M, float* partial, unsigned int* counter, float* tot_sm) {
  __shared__ float wacc[kSemWarps][32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  wacc[warp][lane] = acc;
  __syncthreads();
  if (threadIdx.x < M) {
    float s = 0.f;
    for (int w = 0; w < kSemWarps; ++w) s += wacc[w][threadIdx.x];
    partial[(size_t)blockIdx.x * M + threadIdx.x] = s;
  }
  if (!last_cta(counter)) return false;
  // the last CTA adds the CTAs' partials: warp w owns metapaths w, w + 8, ...; lane-strided over the CTAs, then a
  // fixed shuffle tree (the grid is a function of N alone, so the order is the same on every call)
  for (int m = warp; m < M; m += kSemWarps) {
    float s = 0.f;
    for (unsigned g = lane; g < gridDim.x; g += 32) s += __ldcg(partial + (size_t)g * M + m);
    s = warp_sum(s);
    if (lane == 0) tot_sm[m] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) *counter = 0u;
  return true;
}

// this thread's warp's share of sum_n sum_k q_k tanh(P[n,m,k] + b_k), metapath m in lane m
__device__ __forceinline__ float scores_warp_acc(const float* __restrict__ P, int64_t ldp, const float* __restrict__ b,
                                                 const float* __restrict__ q, int64_t N, int M, int K) {
  const int lane = threadIdx.x & 31;
  const int64_t gw = ((int64_t)blockIdx.x * kSemThreads + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * kSemThreads) >> 5;
  float acc = 0.f;
  for (int64_t n = gw; n < N; n += nw) {
    for (int m = 0; m < M; ++m) {
      const float* row = P + (n * M + m) * ldp;
      float v = 0.f;
      for (int k = lane; k < K; k += 32) v = fmaf(__ldg(q + k), tanhf(__ldg(row + k) + (b ? __ldg(b + k) : 0.f)), v);
      v = warp_sum(v);
      if (lane == m) acc += v;
    }
  }
  return acc;
}

// one thread: tot (the node sums, overwritten) -> scores = tot / N, beta = softmax_M(scores)
__device__ __forceinline__ void scores_finalize(float* tot, int64_t N, int M, float* scores, float* beta) {
  float mx = -INFINITY;
  for (int m = 0; m < M; ++m) {
    tot[m] = tot[m] / (float)N;
    scores[m] = tot[m];
    mx = fmaxf(mx, tot[m]);
  }
  float sum = 0.f;
  for (int m = 0; m < M; ++m) {
    tot[m] = expf(tot[m] - mx);
    sum += tot[m];
  }
  for (int m = 0; m < M; ++m) beta[m] = tot[m] / sum;
}

__global__ void __launch_bounds__(kSemThreads) semantic_scores_kernel(const float* __restrict__ P, int64_t ldp,
                                                                      const float* __restrict__ b,
                                                                      const float* __restrict__ q, int64_t N, int M,
                                                                      int K, float* scores, float* beta, float* partial,
                                                                      unsigned int* counter) {
  __shared__ float tot[32];
  const float acc = scores_warp_acc(P, ldp, b, q, N, M, K);
  if (!reduce_over_grid_m(acc, M, partial, counter, tot)) return;
  if (threadIdx.x == 0) scores_finalize(tot, N, M, scores, beta);
}

// the node sums of semantic_scores_kernel over this part's rows, before the division by N
__global__ void __launch_bounds__(kSemThreads) semantic_scores_partial_kernel(const float* __restrict__ P, int64_t ldp,
                                                                              const float* __restrict__ b,
                                                                              const float* __restrict__ q, int64_t N,
                                                                              int M, int K, float* sums, float* partial,
                                                                              unsigned int* counter) {
  __shared__ float tot[32];
  const float acc = scores_warp_acc(P, ldp, b, q, N, M, K);
  if (!reduce_over_grid_m(acc, M, partial, counter, tot)) return;
  if (threadIdx.x < M) sums[threadIdx.x] = tot[threadIdx.x];
}

__global__ void semantic_scores_finalize_kernel(const float* __restrict__ sums, int64_t n_total, int M, float* scores,
                                                float* beta) {
  __shared__ float tot[32];
  for (int m = 0; m < M; ++m) tot[m] = sums[m];
  scores_finalize(tot, n_total, M, scores, beta);
}

__global__ void __launch_bounds__(kSemThreads) semantic_combine_kernel(const float* __restrict__ beta,
                                                                       const float* __restrict__ z, int64_t N, int M,
                                                                       int D, float* __restrict__ out) {
  const int64_t total = N * D;
  for (int64_t i = (int64_t)blockIdx.x * kSemThreads + threadIdx.x; i < total; i += (int64_t)gridDim.x * kSemThreads) {
    const int64_t n = i / D;
    const int d = (int)(i - n * D);
    const float* zr = z + n * M * D + d;
    float s = 0.f;
    for (int m = 0; m < M; ++m) s = fmaf(__ldg(beta + m), __ldg(zr + (int64_t)m * D), s);
    out[i] = s;
  }
}

// writes the direct term dz = beta_m dOut of this thread's rows; returns its warp's share of
// dbeta_m = sum_n <dOut_n, z_nm>, metapath m in lane m
__device__ __forceinline__ float combine_bwd_warp_acc(const float* __restrict__ d_out, const float* __restrict__ z,
                                                      const float* __restrict__ beta, int64_t N, int M, int D,
                                                      float* __restrict__ dz) {
  const int lane = threadIdx.x & 31;
  const int64_t gw = ((int64_t)blockIdx.x * kSemThreads + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * kSemThreads) >> 5;
  float acc = 0.f;
  for (int64_t n = gw; n < N; n += nw) {
    const float* g = d_out + n * D;
    for (int m = 0; m < M; ++m) {
      const float bm = __ldg(beta + m);
      const float* zr = z + (n * M + m) * D;
      float* dzr = dz + (n * M + m) * D;
      float v = 0.f;
      for (int d = lane; d < D; d += 32) {
        const float gd = __ldg(g + d);
        v = fmaf(gd, __ldg(zr + d), v);
        dzr[d] = bm * gd;
      }
      v = warp_sum(v);
      if (lane == m) acc += v;
    }
  }
  return acc;
}

// one thread: the softmax backward over M, divided by the node count N
__device__ __forceinline__ void combine_bwd_finalize(const float* tot, const float* beta, int64_t N, int M,
                                                     float* d_scores_over_n) {
  float dotp = 0.f;  // Σ_j beta_j dbeta_j
  for (int m = 0; m < M; ++m) dotp = fmaf(beta[m], tot[m], dotp);
  for (int m = 0; m < M; ++m) d_scores_over_n[m] = beta[m] * (tot[m] - dotp) / (float)N;
}

__global__ void __launch_bounds__(kSemThreads) semantic_combine_bwd_kernel(const float* __restrict__ d_out,
                                                                           const float* __restrict__ z,
                                                                           const float* __restrict__ beta, int64_t N,
                                                                           int M, int D, float* __restrict__ dz,
                                                                           float* d_scores_over_n, float* partial,
                                                                           unsigned int* counter) {
  __shared__ float tot[32];
  const float acc = combine_bwd_warp_acc(d_out, z, beta, N, M, D, dz);
  if (!reduce_over_grid_m(acc, M, partial, counter, tot)) return;
  if (threadIdx.x == 0) combine_bwd_finalize(tot, beta, N, M, d_scores_over_n);
}

__global__ void __launch_bounds__(kSemThreads) semantic_combine_bwd_partial_kernel(
    const float* __restrict__ d_out, const float* __restrict__ z, const float* __restrict__ beta, int64_t N, int M,
    int D, float* __restrict__ dz, float* dbeta, float* partial, unsigned int* counter) {
  __shared__ float tot[32];
  const float acc = combine_bwd_warp_acc(d_out, z, beta, N, M, D, dz);
  if (!reduce_over_grid_m(acc, M, partial, counter, tot)) return;
  if (threadIdx.x < M) dbeta[threadIdx.x] = tot[threadIdx.x];
}

__global__ void semantic_combine_bwd_finalize_kernel(const float* __restrict__ dbeta, const float* __restrict__ beta,
                                                     int64_t n_total, int M, float* d_scores_over_n) {
  combine_bwd_finalize(dbeta, beta, n_total, M, d_scores_over_n);
}

__global__ void __launch_bounds__(kSemThreads) semantic_scores_bwd_kernel(const float* __restrict__ P, int64_t ldp,
                                                                          const float* __restrict__ b,
                                                                          const float* __restrict__ q,
                                                                          const float* __restrict__ dsn, int64_t R,
                                                                          int M, int K, float* __restrict__ dP,
                                                                          int64_t lddp, float* dq, float* db,
                                                                          float* partial, unsigned int* counter) {
  __shared__ float sq[kSemThreads], sb[kSemThreads];
  const int rows_per_iter = kSemThreads / K;  // K <= 256
  const int k = threadIdx.x % K, ry = threadIdx.x / K;
  const bool active = ry < rows_per_iter;
  float aq = 0.f, ab = 0.f;
  if (active) {
    const float qk = __ldg(q + k), bk = b ? __ldg(b + k) : 0.f;
    for (int64_t r = (int64_t)blockIdx.x * rows_per_iter + ry; r < R; r += (int64_t)gridDim.x * rows_per_iter) {
      const float t = tanhf(__ldg(P + r * ldp + k) + bk);
      const float ds = __ldg(dsn + (int)(r % M));
      const float g = ds * qk * (1.f - t * t);
      dP[r * lddp + k] = g;
      aq = fmaf(ds, t, aq);
      ab += g;
    }
  }
  sq[threadIdx.x] = aq;
  sb[threadIdx.x] = ab;
  __syncthreads();
  if (threadIdx.x < K) {
    float s0 = 0.f, s1 = 0.f;
    for (int y = 0; y < rows_per_iter; ++y) {
      s0 += sq[y * K + threadIdx.x];
      s1 += sb[y * K + threadIdx.x];
    }
    partial[(size_t)blockIdx.x * 2 * K + threadIdx.x] = s0;
    partial[(size_t)blockIdx.x * 2 * K + K + threadIdx.x] = s1;
  }
  if (!last_cta(counter)) return;
  if (threadIdx.x < K) {
    float s0 = 0.f, s1 = 0.f;
#pragma unroll 8
    for (unsigned g = 0; g < gridDim.x; ++g) {  // 16 independent loads in flight per thread, added in CTA order
      s0 += __ldcg(partial + (size_t)g * 2 * K + threadIdx.x);
      s1 += __ldcg(partial + (size_t)g * 2 * K + K + threadIdx.x);
    }
    dq[threadIdx.x] = s0;
    if (db) db[threadIdx.x] = s1;
  }
  __syncthreads();
  if (threadIdx.x == 0) *counter = 0u;
}

int check_sem(int64_t N, int32_t M, int32_t KD, const char* what) {
  GNN_REQUIRE(N >= 0 && M >= 1 && KD >= 1, GNN_ERR_BAD_ARG, "negative or zero size");
  GNN_REQUIRE(M <= kSemMaxM, GNN_ERR_UNSUPPORTED, "%d metapaths exceed %d per call", M, kSemMaxM);
  (void)what;
  return GNN_OK;
}

int64_t sem_ws_bytes(int32_t K) {
  const int64_t per_cta = 2 * (int64_t)(K > kSemMaxM ? K : kSemMaxM);
  return (4 + (int64_t)sem_grid_cap() * per_cta) * (int64_t)sizeof(float);
}

unsigned grid_for(int64_t items_per_cta_step, int64_t items) {
  int64_t g = (items + items_per_cta_step - 1) / items_per_cta_step;
  const int64_t cap = sem_grid_cap();
  g = g < 1 ? 1 : (g > cap ? cap : g);
  return (unsigned)g;
}

}  // namespace

extern "C" {

int64_t gnn_semantic_workspace_size(int32_t K) { return K >= 1 && K <= kSemMaxK ? sem_ws_bytes(K) : -1; }

int gnn_semantic_scores_f32(const float* P, int64_t ldp, const float* bias, const float* q, int64_t N, int32_t M,
                            int32_t K, float* scores, float* beta, void* workspace, int64_t workspace_bytes,
                            void* stream) {
  int rc = check_sem(N, M, K, "gnn_semantic_scores");
  if (rc != GNN_OK) return rc;
  GNN_REQUIRE(K <= kSemMaxK, GNN_ERR_UNSUPPORTED, "hidden width %d exceeds %d", K, kSemMaxK);
  GNN_REQUIRE(N > 0, GNN_ERR_BAD_ARG, "semantic attention over zero nodes (mean over an empty axis)");
  GNN_REQUIRE(P && q && scores && beta && workspace, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(ldp >= K, GNN_ERR_BAD_ARG, "ldp smaller than K");
  GNN_REQUIRE(workspace_bytes >= sem_ws_bytes(K) && aligned_to(workspace, 16), GNN_ERR_BAD_ARG,
              "workspace too small or misaligned (gnn_semantic_workspace_size)");
  float* ws = static_cast<float*>(workspace);
  semantic_scores_kernel<<<grid_for(kSemWarps * 8, N), kSemThreads, 0, (cudaStream_t)stream>>>(
      P, ldp, bias, q, N, M, K, scores, beta, ws + 4, reinterpret_cast<unsigned int*>(ws));
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_semantic_combine_f32(const float* beta, const float* z, int64_t N, int32_t M, int32_t D, float* out,
                             void* stream) {
  int rc = check_sem(N, M, D, "gnn_semantic_combine");
  if (rc != GNN_OK) return rc;
  if (N == 0) return GNN_OK;
  GNN_REQUIRE(beta && z && out, GNN_ERR_BAD_ARG, "null pointer");
  semantic_combine_kernel<<<grid_for(kSemThreads, N * D), kSemThreads, 0, (cudaStream_t)stream>>>(beta, z, N, M, D,
                                                                                                  out);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_semantic_combine_bwd_f32(const float* d_out, const float* z, const float* beta, int64_t N, int32_t M,
                                 int32_t D, float* dz, float* d_scores_over_n, void* workspace,
                                 int64_t workspace_bytes, void* stream) {
  int rc = check_sem(N, M, D, "gnn_semantic_combine_bwd");
  if (rc != GNN_OK) return rc;
  GNN_REQUIRE(N > 0, GNN_ERR_BAD_ARG, "semantic attention over zero nodes");
  GNN_REQUIRE(d_out && z && beta && dz && d_scores_over_n && workspace, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(workspace_bytes >= sem_ws_bytes(kSemMaxM) && aligned_to(workspace, 16), GNN_ERR_BAD_ARG,
              "workspace too small or misaligned (gnn_semantic_workspace_size)");
  float* ws = static_cast<float*>(workspace);
  semantic_combine_bwd_kernel<<<grid_for(kSemWarps * 8, N), kSemThreads, 0, (cudaStream_t)stream>>>(
      d_out, z, beta, N, M, D, dz, d_scores_over_n, ws + 4, reinterpret_cast<unsigned int*>(ws));
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_semantic_scores_bwd_f32(const float* P, int64_t ldp, const float* bias, const float* q,
                                const float* d_scores_over_n, int64_t N, int32_t M, int32_t K, float* dP, int64_t lddp,
                                float* dq, float* dbias, void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = check_sem(N, M, K, "gnn_semantic_scores_bwd");
  if (rc != GNN_OK) return rc;
  GNN_REQUIRE(K <= kSemMaxK, GNN_ERR_UNSUPPORTED, "hidden width %d exceeds %d", K, kSemMaxK);
  GNN_REQUIRE(N > 0, GNN_ERR_BAD_ARG, "semantic attention over zero nodes");
  GNN_REQUIRE(P && q && d_scores_over_n && dP && dq && workspace, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(ldp >= K && lddp >= K, GNN_ERR_BAD_ARG, "leading dimension smaller than K");
  GNN_REQUIRE(workspace_bytes >= sem_ws_bytes(K) && aligned_to(workspace, 16), GNN_ERR_BAD_ARG,
              "workspace too small or misaligned (gnn_semantic_workspace_size)");
  float* ws = static_cast<float*>(workspace);
  const int rows_per_iter = kSemThreads / K;
  semantic_scores_bwd_kernel<<<grid_for(rows_per_iter * 64, N * M), kSemThreads, 0, (cudaStream_t)stream>>>(
      P, ldp, bias, q, d_scores_over_n, N * M, M, K, dP, lddp, dq, dbias, ws + 4,
      reinterpret_cast<unsigned int*>(ws));
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_semantic_scores_partial_f32(const float* P, int64_t ldp, const float* bias, const float* q, int64_t N,
                                    int32_t M, int32_t K, float* sums, void* workspace, int64_t workspace_bytes,
                                    void* stream) {
  int rc = check_sem(N, M, K, "gnn_semantic_scores_partial");
  if (rc != GNN_OK) return rc;
  GNN_REQUIRE(K <= kSemMaxK, GNN_ERR_UNSUPPORTED, "hidden width %d exceeds %d", K, kSemMaxK);
  GNN_REQUIRE((P || N == 0) && q && sums && workspace, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(ldp >= K, GNN_ERR_BAD_ARG, "ldp smaller than K");
  GNN_REQUIRE(workspace_bytes >= sem_ws_bytes(K) && aligned_to(workspace, 16), GNN_ERR_BAD_ARG,
              "workspace too small or misaligned (gnn_semantic_workspace_size)");
  float* ws = static_cast<float*>(workspace);
  semantic_scores_partial_kernel<<<grid_for(kSemWarps * 8, N), kSemThreads, 0, (cudaStream_t)stream>>>(
      P, ldp, bias, q, N, M, K, sums, ws + 4, reinterpret_cast<unsigned int*>(ws));
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_semantic_scores_finalize_f32(const float* sums, int64_t n_total, int32_t M, float* scores, float* beta,
                                     void* stream) {
  int rc = check_sem(n_total, M, 1, "gnn_semantic_scores_finalize");
  if (rc != GNN_OK) return rc;
  GNN_REQUIRE(n_total > 0, GNN_ERR_BAD_ARG, "semantic attention over zero nodes (mean over an empty axis)");
  GNN_REQUIRE(sums && scores && beta, GNN_ERR_BAD_ARG, "null pointer");
  semantic_scores_finalize_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(sums, n_total, M, scores, beta);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_semantic_combine_bwd_partial_f32(const float* d_out, const float* z, const float* beta, int64_t N, int32_t M,
                                         int32_t D, float* dz, float* dbeta, void* workspace, int64_t workspace_bytes,
                                         void* stream) {
  int rc = check_sem(N, M, D, "gnn_semantic_combine_bwd_partial");
  if (rc != GNN_OK) return rc;
  GNN_REQUIRE(((d_out && z && dz) || N == 0) && beta && dbeta && workspace, GNN_ERR_BAD_ARG, "null pointer");
  GNN_REQUIRE(workspace_bytes >= sem_ws_bytes(kSemMaxM) && aligned_to(workspace, 16), GNN_ERR_BAD_ARG,
              "workspace too small or misaligned (gnn_semantic_workspace_size)");
  float* ws = static_cast<float*>(workspace);
  semantic_combine_bwd_partial_kernel<<<grid_for(kSemWarps * 8, N), kSemThreads, 0, (cudaStream_t)stream>>>(
      d_out, z, beta, N, M, D, dz, dbeta, ws + 4, reinterpret_cast<unsigned int*>(ws));
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

int gnn_semantic_combine_bwd_finalize_f32(const float* dbeta, const float* beta, int64_t n_total, int32_t M,
                                          float* d_scores_over_n, void* stream) {
  int rc = check_sem(n_total, M, 1, "gnn_semantic_combine_bwd_finalize");
  if (rc != GNN_OK) return rc;
  GNN_REQUIRE(n_total > 0, GNN_ERR_BAD_ARG, "semantic attention over zero nodes");
  GNN_REQUIRE(dbeta && beta && d_scores_over_n, GNN_ERR_BAD_ARG, "null pointer");
  semantic_combine_bwd_finalize_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(dbeta, beta, n_total, M, d_scores_over_n);
  GNN_LAUNCH_CHECK();
  return GNN_OK;
}

}  // extern "C"
