// GCN aggregation Y = Â·X: C ABI over the CSR SpMM kernels of spmm_kernels.cuh.
// Replaces torch.spmm(adj, support) at /root/reference GCN/GCN.py:43 and, on the
// transposed CSR, its autograd backward Âᵀ·dY.
#include "spmm_kernels.cuh"

using namespace gnn;

namespace {

template <typename T>
int spmm_impl(const int64_t* rowptr, const int32_t* col, const float* val, const T* X, T* Y, int64_t n_rows,
              int64_t n_cols, int32_t F, int64_t ldx, int64_t ldy, const int64_t* long_rows, int64_t n_long,
              int64_t long_threshold, const int64_t* chunk_off, int64_t n_chunks, int32_t chunk_edges, int accumulate,
              int32_t rows_per_team, const float* bias, int32_t relu, void* workspace, size_t workspace_bytes,
              cudaStream_t st, const gnn_spmm_opts* ex = nullptr, int64_t epi_skip = 0) {
  GNN_REQUIRE(n_rows >= 0 && n_cols >= 0 && F >= 0, GNN_ERR_BAD_ARG, "negative size");
  if (n_rows == 0 || F == 0) return GNN_OK;
  // col may be null only for a graph without edges (nnz lives on the device; rowptr decides)
  GNN_REQUIRE(rowptr && X && Y, GNN_ERR_BAD_ARG, "null pointer (rowptr/X/Y)");
  GNN_REQUIRE(ldx >= F && ldy >= F, GNN_ERR_BAD_ARG, "leading dimension smaller than F (ldx=%lld ldy=%lld F=%d)",
              (long long)ldx, (long long)ldy, F);
  GNN_REQUIRE(n_cols < 0x7fffffffLL, GNN_ERR_UNSUPPORTED, "n_cols does not fit int32 column ids");
  GNN_REQUIRE(aligned_to(X, sizeof(T)) && aligned_to(Y, sizeof(T)), GNN_ERR_MISALIGNED, "X/Y not element aligned");
  SpmmArgs<T> a{};
  a.rowptr = rowptr;
  a.col = col;
  a.val = val;
  a.X = X;
  a.ldx = ldx;
  a.Y = Y;
  a.ldy = ldy;
  a.n_rows = n_rows;
  a.F = F;
  a.skip_deg_gt = 0;
  a.accumulate = accumulate ? 1 : 0;
  GNN_REQUIRE(rows_per_team >= 0, GNN_ERR_BAD_ARG, "rows_per_team must be >= 0");
  // the planned entry keeps the epilogue on overwriting launches; the extended one also fuses it into the
  // accumulating (last) pass of a two-pass row: y = relu?(y_prev + sum + b)
  GNN_REQUIRE(ex || !(accumulate && (bias || relu)), GNN_ERR_BAD_ARG, "the bias/ReLU epilogue belongs to the final pass");
  a.bias = bias;
  a.relu = relu ? 1 : 0;
  a.rows_per_team = tuning("spmm.rows_per_team", 0) > 0 ? tuning("spmm.rows_per_team", 0) : rows_per_team;
  a.split = 0x7fffffff;
  if (ex) {
    // row-subset / two-table form: the CSR is compact over the selected rows
    GNN_REQUIRE(ex->accumulate_prefix >= 0 && ex->accumulate_prefix <= n_rows, GNN_ERR_BAD_ARG,
                "accumulate_prefix out of range");
    GNN_REQUIRE(epi_skip >= 0 && epi_skip <= n_rows, GNN_ERR_BAD_ARG, "epilogue_skip_prefix out of range");
    GNN_REQUIRE(ex->exclusion_smem_bytes >= 0 && ex->exclusion_smem_bytes <= 48 * 1024, GNN_ERR_BAD_ARG,
                "exclusion_smem_bytes must be within [0, 48 KB]");
    a.row_map = ex->row_map;
    a.acc_prefix = ex->accumulate_prefix;
    a.excl_smem = ex->exclusion_smem_bytes;
    a.epi_skip = epi_skip;
    if (ex->X2) {
      GNN_REQUIRE(ex->split >= 0 && ex->split <= n_cols && ex->ldx2 >= F, GNN_ERR_BAD_ARG, "bad split / ldx2");
      GNN_REQUIRE(aligned_to(ex->X2, sizeof(T)), GNN_ERR_MISALIGNED, "X2 not element aligned");
      a.ldx2 = ex->ldx2;
      a.split = (int32_t)ex->split;
      a.X2 = (const T*)ex->X2 - ex->split * ex->ldx2;  // pre-offset: column c >= split reads X2 + c * ldx2
    }
  }
  if (n_long > 0) {
    GNN_REQUIRE(long_rows && chunk_off && long_threshold > 0 && chunk_edges > 0 && n_chunks >= n_long, GNN_ERR_BAD_ARG,
                "inconsistent long-row plan");
    GNN_REQUIRE(n_chunks < 0x7fffffffLL, GNN_ERR_UNSUPPORTED, "too many long-row chunks");
    GNN_REQUIRE(workspace && workspace_bytes >= spmm_long_workspace_bytes(n_chunks, (int)sizeof(T)), GNN_ERR_WORKSPACE,
                "workspace too small for %lld chunks", (long long)n_chunks);
    a.skip_deg_gt = long_threshold;
    // long rows first: their few, heavy CTAs start early and the short-row grid fills in behind
    int rc = spmm_long<T>(a, long_rows, n_long, chunk_off, n_chunks, chunk_edges, (float*)workspace, st);
    if (rc != GNN_OK) return rc;
  }
  return spmm_main<T>(a, st);
}

// struct_size is the version of gnn_spmm_opts: the current size, or the size before epilogue_skip_prefix was
// appended (read as 0).  -1: missing or unknown version (the caller's struct must not be read past its end).
int64_t spmm_opts_epilogue_skip(const gnn_spmm_opts* o) {
  if (!o) return -1;
  if (o->struct_size == (int32_t)sizeof(gnn_spmm_opts)) return o->epilogue_skip_prefix;
  if (o->struct_size == (int32_t)offsetof(gnn_spmm_opts, epilogue_skip_prefix)) return 0;
  return -1;
}

}  // namespace

extern "C" {

size_t gnn_spmm_csr_workspace_size(int64_t n_chunks, int32_t elem_size) {
  if (n_chunks <= 0 || (elem_size != 2 && elem_size != 4)) return 0;
  return spmm_long_workspace_bytes(n_chunks, elem_size);
}

int gnn_spmm_csr_f32(const int64_t* rowptr, const int32_t* col, const float* val, const float* X, float* Y,
                     int64_t n_rows, int64_t n_cols, int32_t F, int64_t ldx, int64_t ldy, gnn_stream_t stream) {
  return spmm_impl<float>(rowptr, col, val, X, Y, n_rows, n_cols, F, ldx, ldy, nullptr, 0, 0, nullptr, 0, 0, 0, 0,
                          nullptr, 0, nullptr, 0, (cudaStream_t)stream);
}

int gnn_spmm_csr_bf16(const int64_t* rowptr, const int32_t* col, const float* val, const void* X, void* Y,
                      int64_t n_rows, int64_t n_cols, int32_t F, int64_t ldx, int64_t ldy, gnn_stream_t stream) {
  return spmm_impl<__nv_bfloat16>(rowptr, col, val, (const __nv_bfloat16*)X, (__nv_bfloat16*)Y, n_rows, n_cols, F, ldx,
                                  ldy, nullptr, 0, 0, nullptr, 0, 0, 0, 0, nullptr, 0, nullptr, 0, (cudaStream_t)stream);
}

int gnn_spmm_csr_planned_f32(const int64_t* rowptr, const int32_t* col, const float* val, const float* X, float* Y,
                             int64_t n_rows, int64_t n_cols, int32_t F, int64_t ldx, int64_t ldy,
                             const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                             const int64_t* chunk_off, int64_t n_chunks, int32_t chunk_edges, int accumulate,
                             int32_t rows_per_team, const float* bias, int32_t relu, void* workspace,
                             size_t workspace_bytes, gnn_stream_t stream) {
  return spmm_impl<float>(rowptr, col, val, X, Y, n_rows, n_cols, F, ldx, ldy, long_rows, n_long, long_threshold,
                          chunk_off, n_chunks, chunk_edges, accumulate, rows_per_team, bias, relu, workspace, workspace_bytes,
                          (cudaStream_t)stream);
}

int gnn_spmm_csr_planned_bf16(const int64_t* rowptr, const int32_t* col, const float* val, const void* X, void* Y,
                              int64_t n_rows, int64_t n_cols, int32_t F, int64_t ldx, int64_t ldy,
                              const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                              const int64_t* chunk_off, int64_t n_chunks, int32_t chunk_edges, int accumulate,
                              int32_t rows_per_team, const float* bias, int32_t relu, void* workspace,
                              size_t workspace_bytes, gnn_stream_t stream) {
  return spmm_impl<__nv_bfloat16>(rowptr, col, val, (const __nv_bfloat16*)X, (__nv_bfloat16*)Y, n_rows, n_cols, F, ldx,
                                  ldy, long_rows, n_long, long_threshold, chunk_off, n_chunks, chunk_edges, accumulate,
                                  rows_per_team, bias, relu, workspace, workspace_bytes, (cudaStream_t)stream);
}

int gnn_spmm_csr_ex_f32(const int64_t* rowptr, const int32_t* col, const float* val, const float* X, float* Y,
                        int64_t n_rows, int64_t n_cols, int32_t F, int64_t ldx, int64_t ldy, const gnn_spmm_opts* o,
                        gnn_stream_t stream) {
  const int64_t epi_skip = spmm_opts_epilogue_skip(o);
  GNN_REQUIRE(epi_skip >= 0, GNN_ERR_BAD_ARG, "gnn_spmm_opts missing or struct_size mismatch (header/library version skew)");
  return spmm_impl<float>(rowptr, col, val, X, Y, n_rows, n_cols, F, ldx, ldy, o->long_rows, o->n_long,
                          o->long_threshold, o->chunk_off, o->n_chunks, o->chunk_edges, o->accumulate, o->rows_per_team,
                          o->bias, o->relu, o->workspace, o->workspace_bytes, (cudaStream_t)stream, o, epi_skip);
}

int gnn_spmm_csr_ex_bf16(const int64_t* rowptr, const int32_t* col, const float* val, const void* X, void* Y,
                         int64_t n_rows, int64_t n_cols, int32_t F, int64_t ldx, int64_t ldy, const gnn_spmm_opts* o,
                         gnn_stream_t stream) {
  const int64_t epi_skip = spmm_opts_epilogue_skip(o);
  GNN_REQUIRE(epi_skip >= 0, GNN_ERR_BAD_ARG, "gnn_spmm_opts missing or struct_size mismatch (header/library version skew)");
  return spmm_impl<__nv_bfloat16>(rowptr, col, val, (const __nv_bfloat16*)X, (__nv_bfloat16*)Y, n_rows, n_cols, F, ldx,
                                  ldy, o->long_rows, o->n_long, o->long_threshold, o->chunk_off, o->n_chunks,
                                  o->chunk_edges, o->accumulate, o->rows_per_team, o->bias, o->relu, o->workspace,
                                  o->workspace_bytes, (cudaStream_t)stream, o, epi_skip);
}

}  // extern "C"
