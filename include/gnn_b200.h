/*
 * gnn_b200.h — C ABI of the B200-native message-passing kernels.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference
 * (kaddly/GraphNeuralNetwork) has no FFI: its seam is the Python
 * nn.Module.forward of each layer, which bottoms out in ATen calls.  Every entry
 * point below replaces one of those ATen call sites; the citation after "replaces"
 * is the reference file:line whose arithmetic the entry point reproduces.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless the
 *    name ends in _host;
 *  - the caller owns every buffer; the library never allocates outputs; scratch is
 *    passed in as (workspace, workspace_bytes) after a *_workspace_size query;
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*), makes
 *    no hidden synchronisation, and is re-entrant;
 *  - return value: 0 = GNN_OK, otherwise a gnn_status; never throws, never aborts.
 *    gnn_last_error_string() returns a thread-local description of the last failure;
 *  - deterministic: no floating-point atomics anywhere; the same inputs give the
 *    same bits on every run.
 *  - index types: rowptr int64, col int32 (SURVEY.md §7 "Index width").
 */
#ifndef GNN_B200_H
#define GNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* gnn_stream_t; /* cudaStream_t */

typedef enum {
  GNN_OK = 0,
  GNN_ERR_BAD_ARG = 1,
  GNN_ERR_MISALIGNED = 2,
  GNN_ERR_UNSUPPORTED = 3,
  GNN_ERR_CUDA = 4,
  GNN_ERR_WORKSPACE = 5
} gnn_status;

/* reduce op of the fixed-fanout gather (GraphSAGE_Pytorch/models/Aggregator.py:19-24) */
typedef enum { GNN_REDUCE_MEAN = 0, GNN_REDUCE_SUM = 1, GNN_REDUCE_MAX = 2 } gnn_reduce;

/* edge-score mode of the fused attention kernel */
typedef enum {
  GNN_GAT_SOFTMAX = 0, /* GAT/models/layers.py:26-32: softmax_j(LeakyReLU(s_i+t_j)) */
  GNN_GAT_EXPNEG = 1   /* GAT/models/layers.py:108-122: exp(-LeakyReLU(.)) / rowsum  */
} gnn_gat_mode;

/* ---- library ---------------------------------------------------------- */
int gnn_version(void);
const char* gnn_last_error_string(void);
const char* gnn_status_string(int status);
/* number of kernels this library has launched in the calling process (bench.py's
 * gpu_launches claim is read from here). */
int64_t gnn_launch_count(void);
/* tuning knobs for measurement sweeps ("sage.smem_kb", "sage.chunk_rows",
 * "sage.force_ldg", "spmm.long_row", ...).  Returns GNN_ERR_BAD_ARG for unknown keys. */
int gnn_set_tuning(const char* key, int value);
int gnn_get_tuning(const char* key, int* value);

/* ---- graph construction (bit-exact index work) -------------------------- */

/* COO (as produced by GCN/data_utils.py:63-70 sparse_mx_to_torch_sparse_tensor:
 * int64 indices [2,nnz] row-major sorted, fp32 values) -> CSR.  The sort is stable
 * in (row), so the within-row order of the input is preserved; for the reference's
 * already row-major-sorted COO the result is the identity permutation.
 * perm_out (nullable, int64[nnz]) receives the input position of every output slot. */
size_t gnn_build_csr_from_coo_workspace_size(int64_t nnz, int64_t n_rows);
int gnn_build_csr_from_coo(const int64_t* coo_row, const int64_t* coo_col, const float* coo_val /*nullable*/,
                           int64_t nnz, int64_t n_rows, int64_t n_cols,
                           int64_t* rowptr /*[n_rows+1]*/, int32_t* col /*[nnz]*/, float* val /*nullable [nnz]*/,
                           int64_t* perm_out /*nullable [nnz]*/,
                           void* workspace, size_t workspace_bytes, gnn_stream_t stream);

/* Dense mask (GAT/models/layers.py:29 / HAN/models/NodeAttention.py:28: `adj > 0`)
 * -> CSR pattern, columns ascending, i.e. the order of `adj.nonzero()`
 * (GAT/models/layers.py:98).  Two steps because nnz is only known after the count.
 * adj_dtype: 0 = fp32 (GAT/data_utils.py:85), 1 = fp64 (HAN/utils/data_utils.py:85-89). */
size_t gnn_dense_mask_count_workspace_size(int64_t n_rows);
int gnn_dense_mask_count(const void* adj, int adj_dtype, int64_t n_rows, int64_t n_cols, int64_t ld,
                         int64_t* rowptr /*[n_rows+1], out*/,
                         void* workspace, size_t workspace_bytes, gnn_stream_t stream);
int gnn_dense_mask_fill(const void* adj, int adj_dtype, int64_t n_rows, int64_t n_cols, int64_t ld,
                        const int64_t* rowptr, int32_t* col /*[nnz]*/, gnn_stream_t stream);

/* Pattern product C = pattern(A·B) of two pattern CSRs, A [n_a x k] and B [k x n_b]
 * (replaces HeteroGraph.get_mate_path_graph, HAN/utils/data_utils.py:85-89: the metapath
 * adjacency (P·Pᵀ > 0) of a relation matrix P, there a dense float64 N x N array).  Values are
 * ignored; column ids within a row may be unsorted or repeated, and ids outside [0, k) of A or
 * [0, n_b) of B are skipped.  Rows [row_lo, row_hi) of A: output row r lists, once each and
 * ascending, every global column j with (row_lo+r, x) in A and (x, j) in B -- scipy's
 * ((A_bool @ B_bool) > 0) after sort_indices(), the adj.nonzero() order of the dense mask.
 * self_loops (only when n_a == n_b) adds column i to row i, as (P·Pᵀ + I) > 0.
 * Two steps because nnz is only known after the count.  Both take a workspace of
 * gnn_pattern_product_count_workspace_size(row_hi - row_lo) bytes and route each row by its
 * product count to one of three paths (tuning keys "metapath.small_max", "metapath.medium_max",
 * "metapath.tile_cols"); path_rows (nullable int64[3]) receives the rows each path took
 * (warp sort, CTA sort, shared-memory bitmap).  No floating point; the integer atomics of the
 * bitmap path produce an order-independent set, so the output is the same bits on every run. */
size_t gnn_pattern_product_count_workspace_size(int64_t n_rows);
int gnn_pattern_product_count(const int64_t* a_rowptr, const int32_t* a_col, int64_t n_a, int64_t k,
                              const int64_t* b_rowptr, const int32_t* b_col, int64_t n_b,
                              int64_t row_lo, int64_t row_hi, int self_loops,
                              int64_t* rowptr /*[row_hi-row_lo+1], out, starts at 0*/,
                              int64_t* path_rows /*nullable int64[3], out*/,
                              void* workspace, size_t workspace_bytes, gnn_stream_t stream);
int gnn_pattern_product_fill(const int64_t* a_rowptr, const int32_t* a_col, int64_t n_a, int64_t k,
                             const int64_t* b_rowptr, const int32_t* b_col, int64_t n_b,
                             int64_t row_lo, int64_t row_hi, int self_loops,
                             const int64_t* rowptr /*the count's*/, int32_t* col /*[rowptr[row_hi-row_lo]]*/,
                             void* workspace, size_t workspace_bytes, gnn_stream_t stream);

/* CSR -> CSR of the transpose (the structure the deterministic backward walks:
 * autograd of GCN/GCN.py:43 is Âᵀ·dY; GAT/models/layers.py:63 is aᵀ·dY).
 * Stable in the original row order, so each transposed row lists its sources in
 * ascending original-row order.  perm_t (nullable) = original edge slot per new slot. */
size_t gnn_csr_transpose_workspace_size(int64_t nnz, int64_t n_rows, int64_t n_cols);
int gnn_csr_transpose(const int64_t* rowptr, const int32_t* col, const float* val /*nullable*/,
                      int64_t n_rows, int64_t n_cols, int64_t nnz,
                      int64_t* rowptr_t /*[n_cols+1]*/, int32_t* col_t /*[nnz]*/, float* val_t /*nullable*/,
                      int64_t* perm_t /*nullable [nnz]*/,
                      void* workspace, size_t workspace_bytes, gnn_stream_t stream);

/* Fixed-fanout index block idx[n_src*fanout] (GraphSAGE_Pytorch/sample_utils.py:16
 * src-major layout; GraphSAGE/data_utils.py:105-116 [n,k] map) -> per-table-row list
 * of the flat positions that reference it (ascending): the transposed structure the
 * deterministic gather backward walks.  idx_bits is 32 or 64; negative ids are skipped. */
size_t gnn_index_block_transpose_workspace_size(int64_t n_idx, int64_t n_table_rows);
int gnn_index_block_transpose(const void* idx, int idx_bits, int64_t n_idx, int64_t n_table_rows,
                              int64_t* rowptr_t /*[n_table_rows+1]*/, int32_t* pos_t /*[n_idx]*/,
                              void* workspace, size_t workspace_bytes, gnn_stream_t stream);

/* ---- GCN: Y = Â·X (replaces torch.spmm, GCN/GCN.py:43) ------------------------------ */
/* Row-parallel CSR SpMM, sub-warp per row chosen from F, 128-bit feature loads,
 * sequential in-order accumulation per row (deterministic).  val == NULL => pattern
 * only (all ones).  X [n_cols, ldx], Y [n_rows, ldy], F <= ldx, ldy.
 * The bf16 variant reads/writes bf16 and accumulates in fp32.
 * Backward (dX = Âᵀ·dY) is the same call on the gnn_csr_transpose output. */
int gnn_spmm_csr_f32(const int64_t* rowptr, const int32_t* col, const float* val,
                     const float* X, float* Y, int64_t n_rows, int64_t n_cols, int32_t F,
                     int64_t ldx, int64_t ldy, gnn_stream_t stream);
int gnn_spmm_csr_bf16(const int64_t* rowptr, const int32_t* col, const float* val,
                      const void* X, void* Y, int64_t n_rows, int64_t n_cols, int32_t F,
                      int64_t ldx, int64_t ldy, gnn_stream_t stream);
/* Same, with a plan for power-law graphs: the rows whose nnz exceeds the caller's threshold
 * (long_rows[n_long], ascending row ids) are cut into chunks of chunk_edges edges, one CTA
 * per chunk; chunk_off[n_long+1] is the exclusive prefix sum of ceil(nnz_row/chunk_edges)
 * and n_chunks its last entry.  Per-chunk partial sums live in the workspace
 * (gnn_spmm_csr_workspace_size) and are added per row in chunk order: deterministic.
 * All other rows take the row-block streaming kernel.  n_long may be 0 (no plan arrays
 * needed); accumulate=1 adds into Y (the remote-column pass of the partitioned SpMM,
 * SURVEY.md §8e).  rows_per_team (0 = default) is how many consecutive rows one sub-warp
 * team streams: the default suits sparse rows (papers100M-shaped, 14 edges per row); the
 * host lowers it on dense graphs (Reddit-shaped, 490 per row) so that a team holds a few
 * hundred edges and the grid has enough warps.  bias / relu fuse the rest of the GCN layer
 * into the row flush: Y = relu?(A*X + bias) (`output + self.bias` GCN/GCN.py:44-45 and the
 * nn.ReLU that follows the layer, GCN.py:12); not allowed with accumulate=1.
 * The plan is host logic computed once
 * per graph (graphneuralnetwork_b200/graph.py CSRGraph.long_row_plan / rows_per_team). */
size_t gnn_spmm_csr_workspace_size(int64_t n_chunks, int32_t elem_size);
int gnn_spmm_csr_planned_f32(const int64_t* rowptr, const int32_t* col, const float* val,
                             const float* X, float* Y, int64_t n_rows, int64_t n_cols, int32_t F,
                             int64_t ldx, int64_t ldy,
                             const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                             const int64_t* chunk_off, int64_t n_chunks, int32_t chunk_edges,
                             int accumulate /*1: Y += A*X*/, int32_t rows_per_team,
                             const float* bias /*nullable [F]*/, int32_t relu,
                             void* workspace, size_t workspace_bytes, gnn_stream_t stream);
int gnn_spmm_csr_planned_bf16(const int64_t* rowptr, const int32_t* col, const float* val,
                              const void* X, void* Y, int64_t n_rows, int64_t n_cols, int32_t F,
                              int64_t ldx, int64_t ldy,
                              const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                              const int64_t* chunk_off, int64_t n_chunks, int32_t chunk_edges,
                              int accumulate, int32_t rows_per_team,
                              const float* bias /*nullable [F], fp32*/, int32_t relu,
                              void* workspace, size_t workspace_bytes, gnn_stream_t stream);

/* Extended form of the planned SpMM for ROW SUBSETS and TWO SOURCE TABLES — the consumers of the
 * wave-pipelined halo exchange of the partitioned SpMM (SURVEY.md §8e; reference seam GCN/GCN.py:43).
 * The CSR passed in is compact over the selected rows (rowptr has n_rows+1 entries):
 *   row_map (nullable, int32 [n_rows], distinct rows in any order): compact row r writes Y row row_map[r];
 *   accumulate_prefix: compact rows [0, accumulate_prefix) add into Y (their local-column part was
 *     written by an earlier pass), the others overwrite — one launch serves both kinds of row;
 *   X2/ldx2/split: a column id c >= split reads row (c - split) of X2 (the halo buffer) instead of X,
 *     so rows that need local AND remote columns finish in ONE pass with no read-modify-write of Y;
 *   bias/relu: the GCN epilogue y = relu?(. + bias) of the planned entry, here allowed in EVERY form:
 *     with accumulate / accumulate_prefix it applies after the add, y = relu?(y_prev + sum + bias),
 *     and with X2 to the two-table sum, so each output row gets it once, in the launch that writes
 *     the row's last contribution (the planned entry still refuses accumulate with bias/relu);
 *   epilogue_skip_prefix: compact rows [0, epilogue_skip_prefix) get NO epilogue even when bias/relu
 *     are set — the first pass of two-pass rows, written in the same launch as finished rows;
 *   exclusion_smem_bytes: token dynamic shared memory per CTA (<= 48 KB), for callers that keep this
 *     kernel off SMs a shared-memory-filling mover kernel has claimed.  0 = none.
 * Every per-call choice is an argument: no process-global state is consulted.
 * struct_size = sizeof(gnn_spmm_opts) (ABI versioning); zero-initialise the rest.  A struct_size of
 * offsetof(gnn_spmm_opts, epilogue_skip_prefix) (the layout before that field was appended) is also
 * accepted and reads as epilogue_skip_prefix = 0; any other size is refused. */
typedef struct gnn_spmm_opts {
  int32_t struct_size;
  int32_t accumulate;
  int64_t accumulate_prefix;
  int32_t rows_per_team;
  int32_t relu;
  const float* bias;
  const int32_t* row_map;
  const void* X2;
  int64_t ldx2;
  int64_t split;
  const int64_t* long_rows;
  int64_t n_long;
  int64_t long_threshold;
  const int64_t* chunk_off;
  int64_t n_chunks;
  int32_t chunk_edges;
  int32_t exclusion_smem_bytes;
  void* workspace;
  size_t workspace_bytes;
  int64_t epilogue_skip_prefix;
} gnn_spmm_opts;
int gnn_spmm_csr_ex_f32(const int64_t* rowptr, const int32_t* col, const float* val,
                        const float* X, float* Y, int64_t n_rows, int64_t n_cols, int32_t F,
                        int64_t ldx, int64_t ldy, const gnn_spmm_opts* opts, gnn_stream_t stream);
int gnn_spmm_csr_ex_bf16(const int64_t* rowptr, const int32_t* col, const float* val,
                         const void* X, void* Y, int64_t n_rows, int64_t n_cols, int32_t F,
                         int64_t ldx, int64_t ldy, const gnn_spmm_opts* opts, gnn_stream_t stream);

/* Edge-gradient SDDMM: out[e] = <A[row[e], 0:F], B[col[e], 0:F]> for e in [0, nnz).
 * The gradient of Y = S·B with respect to the VALUES of S is dY_i · B_j on the pattern of S:
 * GAT/models/layers.py:55-61 (SpecialSpmmFunction.backward) forms the dense N x N product
 * `grad_output.matmul(b.t())` and indexes it with row*N+col; this forms only the nnz dots.
 * row / col: device id arrays of idx_bits (32|64) bits in any edge order (COO); edge-parallel,
 * deterministic. */
int gnn_sddmm_coo_f32(const void* row, const void* col, int idx_bits, int64_t nnz,
                      const float* A, int64_t lda, const float* B, int64_t ldb, int32_t F,
                      float* out /*[nnz]*/, gnn_stream_t stream);

/* ---- GraphSAGE: fused gather + reduce over fixed-fanout index blocks ----------- */
/* out[i,:] = reduce_k table[idx[i*fanout+k], :]
 * (replaces the CPU gather GraphSAGE_Pytorch/data_utils.py:64 + .mean/.sum/.max(dim=1)
 *  Aggregator.py:19-24; GraphSAGE/graph_utils.py:6 + torch.embedding GraphSAGE.py:47-49).
 * idx == NULL => identity block: neighbours of source i are table rows
 * [i*fanout,(i+1)*fanout) — the pre-gathered [n_src,fanout,F] tensor of Aggregator.py:18.
 * idx_bits 32|64.  Negative ids contribute nothing (mean still divides by fanout).
 * argmax (nullable, int32 [n_src, ld_out], max mode only) records the winning k.
 * When the table rows are 16-byte aligned (ld_table*sizeof(T) % 16 == 0) the rows are
 * fetched with TMA bulk copies into a shared-memory ring; otherwise with vector loads. */
int gnn_gather_reduce_f32(const float* table, int64_t ld_table, int64_t n_table_rows,
                          const void* idx, int idx_bits, int64_t n_src, int32_t fanout, int32_t F,
                          int reduce, float* out, int64_t ld_out, int32_t* argmax, gnn_stream_t stream);
int gnn_gather_reduce_bf16(const void* table, int64_t ld_table, int64_t n_table_rows,
                           const void* idx, int idx_bits, int64_t n_src, int32_t fanout, int32_t F,
                           int reduce, void* out, int64_t ld_out, int32_t* argmax, gnn_stream_t stream);
/* Up to 4 index blocks over the SAME table in one launch (the hops of one minibatch:
 * GraphSAGE_Pytorch/models/GraphSage.py:24-27 sends every hop through the same layer).  The
 * *_host arrays are host arrays of n_blocks entries: device id pointers (nullable = identity),
 * source counts, fanouts, device output pointers and their leading dimensions. */
int gnn_gather_reduce_multi_f32(const float* table, int64_t ld_table, int64_t n_table_rows, int32_t F, int reduce,
                                int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                const int64_t* n_src_host, const int32_t* fanout_host,
                                void* const* out_host, const int64_t* ld_out_host, gnn_stream_t stream);
int gnn_gather_reduce_multi_bf16(const void* table, int64_t ld_table, int64_t n_table_rows, int32_t F, int reduce,
                                 int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                 const int64_t* n_src_host, const int32_t* fanout_host,
                                 void* const* out_host, const int64_t* ld_out_host, gnn_stream_t stream);
/* Same launch, fp32 table, but every reduced value x leaves as TWO fp16 numbers: hi = fp16(x) at out_hi[b] and
 * lo = fp16(x - hi) lo_off[b] fp16 elements further (ld_out / lo_off count fp16 elements; the same bytes as an
 * fp32 output).  hi + lo carries 22 mantissa bits (x - hi is exact in fp32; a residual below fp16's normal range
 * costs < 3e-8 absolute): the A-operand of the 3-product fp16 tensor-core GEMM (A_hi.B_hi + A_lo.B_hi + A_hi.B_lo,
 * fp32 accumulate) that stands in for the fp32 `X.W` product of SageGCN.py:24-27 at fp32-level accuracy — the
 * split is fused into the gather's row flush instead of being a separate pass over the operand.  The caller
 * guarantees |x| < 65504.  TMA path only (16-byte aligned rows >= 256 bytes), mean/sum. */
int gnn_gather_reduce_multi_f32_split(const float* table, int64_t ld_table, int64_t n_table_rows, int32_t F, int reduce,
                                      int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                      const int64_t* n_src_host, const int32_t* fanout_host,
                                      void* const* out_hi_host, const int64_t* ld_out_host,
                                      const int64_t* lo_off_host, gnn_stream_t stream);
/* A feature table split into contiguous row blocks (shards), e.g. one per GPU of a node: shard s holds the global
 * rows [row_begin[s], row_begin[s+1]) at device address base[s] (this device's memory or a peer's gnn_peer_open
 * mapping).  All shards share ld_table, F and the element type.  row_begin[0] = 0, non-decreasing,
 * row_begin[n_shards] = global row count; base[s] may be NULL for an empty shard, else 16-byte aligned.
 * struct_size = sizeof(gnn_sharded_table) (ABI versioning). */
#define GNN_MAX_SHARDS 8
typedef struct gnn_sharded_table {
  int32_t struct_size;
  int32_t n_shards; /* 1..GNN_MAX_SHARDS */
  const void* base[GNN_MAX_SHARDS];
  int64_t row_begin[GNN_MAX_SHARDS + 1];
} gnn_sharded_table;
/* gnn_gather_reduce_multi_{f32,bf16,f32_split} over a sharded table.  Same blocks and semantics (ids < 0 or >= the
 * global row count contribute nothing); each output row is the same ordered sum as over the concatenated table, bit
 * for bit: only the address each row is copied from differs.  TMA path only: ld_table * elem % 16 == 0 and rows of
 * 256 bytes or more (GNN_ERR_MISALIGNED / GNN_ERR_UNSUPPORTED otherwise).  The table is validated before anything
 * is launched. */
int gnn_gather_reduce_multi_sharded_f32(const gnn_sharded_table* table, int64_t ld_table, int32_t F, int reduce,
                                        int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                        const int64_t* n_src_host, const int32_t* fanout_host,
                                        void* const* out_host, const int64_t* ld_out_host, gnn_stream_t stream);
int gnn_gather_reduce_multi_sharded_bf16(const gnn_sharded_table* table, int64_t ld_table, int32_t F, int reduce,
                                         int32_t n_blocks, const void* const* idx_host, int idx_bits,
                                         const int64_t* n_src_host, const int32_t* fanout_host,
                                         void* const* out_host, const int64_t* ld_out_host, gnn_stream_t stream);
int gnn_gather_reduce_multi_sharded_f32_split(const gnn_sharded_table* table, int64_t ld_table, int32_t F,
                                              int reduce, int32_t n_blocks, const void* const* idx_host,
                                              int idx_bits, const int64_t* n_src_host, const int32_t* fanout_host,
                                              void* const* out_hi_host, const int64_t* ld_out_host,
                                              const int64_t* lo_off_host, gnn_stream_t stream);
/* Edge-type axis (GATNE): table [n_nodes, n_types, F] (ld_row = stride between (node,type)
 * rows), idx [n_src, n_types, fanout]; out[(b*n_types+t), :] = reduce_k table[idx[b,t,k], t, :]
 * — the per-type neighbour aggregation of GATNE_Pytorch/models/GATNE.py:57-77 (`torch.cat` of T
 * per-type gathers, then sum/mean over dim 2) and GATNE/models/GATNE.py:50-58 (gather of all T
 * embeddings of every neighbour + `torch.diagonal` + sum), without the [B,T,K,(T,)U]
 * intermediates.  reduce: sum or mean. */
int gnn_gather_reduce_typed_f32(const float* table, int64_t ld_row, int64_t n_nodes, int32_t n_types,
                                const void* idx, int idx_bits, int64_t n_src, int32_t fanout, int32_t F,
                                int reduce, float* out, int64_t ld_out, gnn_stream_t stream);
/* Backward of mean/sum into the table: dTable[r,:] = scale * sum_{p: idx[p]==r} dOut[p/fanout,:]
 * walking the gnn_index_block_transpose structure (ordered, no atomics). */
int gnn_gather_reduce_bwd_f32(const int64_t* rowptr_t, const int32_t* pos_t, int64_t n_table_rows,
                              int32_t fanout, float scale, const float* d_out, int64_t ld_dout,
                              float* d_table, int64_t ld_dtable, int32_t F, gnn_stream_t stream);
/* Backward of the identity block (pre-gathered input): dNeigh[i,k,:] = scale*dOut[i,:],
 * or for max: dNeigh[i,argmax,:] = dOut[i,:], 0 elsewhere. */
int gnn_gather_reduce_bwd_dense_f32(const float* d_out, int64_t ld_dout, const int32_t* argmax /*nullable*/,
                                    int64_t n_src, int32_t fanout, int32_t F, float scale,
                                    float* d_neigh /*[n_src,fanout,F] contiguous*/, gnn_stream_t stream);

/* Fixed-fanout neighbour sampler on the device (SURVEY.md §8f rank 1; semantics of
 * GraphSAGE_Pytorch/sample_utils.py:4-17): for each source id, k DISTINCT neighbours uniformly at
 * random if it has at least k (random.sample), else k draws with replacement (random.choices);
 * out[i*k+j], src-major (sample_utils.py:16).  Counter-based RNG keyed by (seed, i, j):
 * deterministic for a seed, semantically (not bit-) equal to the Mersenne-Twister reference.
 * A source without neighbours (or a negative source id) yields -1 ids, which the gather skips.
 * seed_offset_dev (nullable): a device int64 mixed into the seed at run time, so that a captured
 * CUDA graph draws a fresh sample on every replay. */
int gnn_sample_neighbors(const int64_t* rowptr, const int32_t* col, const void* src, int src_bits,
                         int64_t n_src, int32_t k, uint64_t seed, const int64_t* seed_offset_dev,
                         void* out, int out_bits, gnn_stream_t stream);

/* Node-set union with remap (the `set(nodes) | set(samples)` and id -> position maps of the de-duplicating
 * GraphSAGE collate, GraphSAGE/data_utils.py:100-116), ordered by ascending global id instead of CPython's set order:
 *   out_ids[0..count)  = the ascending unique ids of ids_a ∪ {ids_b >= 0}; out_ids[count..n_a+n_b) = -1, so a padded
 *                        set can be handed to gnn_sample_neighbors and to the next union as it is;
 *   map_a[i] / map_b[j] = position in out_ids of ids_a[i] / ids_b[j], -1 where the id is negative;
 *   *out_count_dev     = count (stays on the device).
 * ids_a, ids_b and out_ids are int32 or int64 (id_bits), the maps int64.  One radix sort of (id, slot) pairs over
 * n_a + n_b keys, a head flag per run, a scan and a scatter: O(n_a + n_b) work and memory, nothing over the node
 * count.  No floating point, no atomics: the same input gives the same bits.  n_a + n_b == 0 writes a count of 0.
 * Bad sizes (negative, or n_a + n_b >= 2^31) and null pointers return GNN_ERR_BAD_ARG before any CUDA call. */
int gnn_node_union_workspace_size(int64_t n_a, int64_t n_b, size_t* bytes_host /*out*/);
int gnn_node_union(const void* ids_a, int64_t n_a, const void* ids_b, int64_t n_b, int id_bits,
                   void* out_ids /*[n_a+n_b]*/, int64_t* out_count_dev /*[1]*/,
                   int64_t* map_a /*[n_a]*/, int64_t* map_b /*[n_b]*/,
                   void* workspace, size_t workspace_bytes, gnn_stream_t stream);

/* ---- GAT / HAN: fused multi-head attention aggregation ---------------------------- */
/* Per-node, per-head halves of the edge score (GAT/models/layers.py:25-26 decomposes
 * exactly: a·[Wh_i || Wh_j] = a[:F']·Wh_i + a[F':]·Wh_j):
 *   s[i,h] = sum_f Wh[i,h*Fp+f]*a_src[h,f],  t[i,h] = sum_f Wh[i,h*Fp+f]*a_dst[h,f]. */
int gnn_gat_scores_f32(const float* Wh, int64_t ldw, const float* a_src, const float* a_dst,
                       int64_t n, int32_t H, int32_t Fp, float* s, float* t, gnn_stream_t stream);
/* out[i, h*Fp+f] = act( sum_j att[i,j,h] * Wh[j, h*Fp+f] ), j over CSR row i, with
 *   mode SOFTMAX: att = softmax_j(LeakyReLU_alpha(s[i,h]+t[j,h]))   (layers.py:26-32)
 *   mode EXPNEG : att = exp(-LeakyReLU_alpha(.)) / sum_j exp(-LeakyReLU_alpha(.)) (layers.py:108-122)
 * apply_elu: 0 none, 1 ELU (layers.py:35), 2 ELU twice (HAN/models/NodeAttention.py:35 then :62).
 * Rows with no edge reproduce the reference's softmax over an all -9e15 row: the
 * uniform mean over ALL nodes, passed in as col_mean[H*Fp] (nullable if no such row).
 * edge_keep (nullable, fp32 [nnz,H]): post-softmax dropout factor per edge and head
 * (0 or 1/(1-p)), layers.py:31.  row_max/row_sum [n,H] are saved for the backward.
 * Schedule: one warp per row; the rows of long_rows[n_long] (those with more than
 * long_threshold edges: the caller's plan, CSRGraph.gat_long_rows) get one CTA each (4 warps on
 * alternate 128-edge chunks, merged in warp order); when nnz/n >= the "gat.coop_min_avg_deg"
 * knob (dense metapath adjacencies) every row gets a CTA and the list is ignored.
 * Rectangular use: Wh and t are read only through col, so col may address n_cols >= n table rows (Wh [n_cols, ldw],
 * t [n_cols, H]; s, out and the row statistics stay [n, .]) — a row block of a partitioned graph whose columns index
 * [own rows ; halo rows].  col_mean (rows without edges) and batch_nodes are not defined for that use: pass NULL / 0
 * (gnn_gat_fused_bwd_ex_f32 is the matching backward). */
int gnn_gat_fused_fwd_f32(const int64_t* rowptr, const int32_t* col, const float* Wh, int64_t ldw,
                          const float* s, const float* t, int64_t n, int64_t nnz /*schedule hint, 0 if unknown*/,
                          int32_t H, int32_t Fp,
                          float alpha, int mode, int apply_elu, const float* col_mean,
                          const float* edge_keep, float* out, int64_t ldo,
                          float* row_max, float* row_sum,
                          const int64_t* long_rows /*nullable*/, int64_t n_long, int64_t long_threshold,
                          int64_t batch_nodes /*0 = one graph; see "batched graphs" below*/,
                          gnn_stream_t stream);
/* Batched graphs (batch_nodes > 0): HAN runs M independent multi-head GATs over M metapath adjacencies of the SAME
 * N nodes (HAN/models/HAN.py:16-23).  One launch serves all of them: the CSR passed in is the block diagonal of the
 * M graphs (n = M*N rows, row r = graph r / N, node r % N, column ids offset by the graph's first row); s, t, the
 * row statistics, d_s and d_t are [M*N, H] indexed by the batched row; graph m's feature columns are the block
 * [m*H*Fp, (m+1)*H*Fp) of Wh / out / out_pre / d_out / d_Wh, whose leading dimensions are >= M*H*Fp — so `out` IS the
 * [N, M, H*Fp] stack HANLayer builds with torch.stack (HAN.py:21).  col_mean is [M*H*Fp]. */

/* Seeded attention dropout (GAT/models/layers.py:31, HAN/models/NodeAttention.py:31): instead of a materialised
 * [nnz,H] mask the kernels recompute, from (seed, forward edge slot, head), whether an attention weight is kept
 * (probability 1-p, kept weights scaled by 1/(1-p)) — identically in the forward and in both backward passes.
 * seed_dev (nullable) is a device int64 mixed into the seed at run time, so a captured CUDA graph draws a fresh
 * mask on every replay.  Semantically (not bit-) equal to F.dropout on the dense attention matrix; the explicit
 * `edge_keep` mask remains for parity tests.
 * edge_slot_base: the keep factor of local edge slot e is the one of slot e + edge_slot_base.  A row block of a
 * larger CSR (a contiguous edge range starting at global slot rowptr[lo]) passes rowptr[lo] and draws exactly the
 * mask the whole graph draws for its edges.  It offsets the seeded stream only, not an explicit edge_keep mask, and
 * needs seed_dev == NULL (GNN_ERR_UNSUPPORTED otherwise): the caller mixes the device half into seed itself.
 * struct_size = sizeof(gnn_gat_dropout) (ABI versioning).  A struct_size of offsetof(gnn_gat_dropout,
 * edge_slot_base) (the layout before that field was appended) is also accepted and reads as edge_slot_base = 0;
 * any other size is refused. */
typedef struct gnn_gat_dropout {
  int32_t struct_size;
  float p;
  uint64_t seed;
  const int64_t* seed_dev;
  int64_t edge_slot_base;
} gnn_gat_dropout;

/* Training form of the forward: writes the PRE-activation aggregate to out_pre (saved for the backward) and, when
 * apply_elu > 0, the activated aggregate to out_act in the same launch — the ELU after every concatenated head
 * (layers.py:35) and HAN's second ELU (NodeAttention.py:62) are never separate launches, in training either.
 * dropout (nullable) selects the seeded dropout above; edge_keep (nullable) an explicit mask; not both. */
int gnn_gat_fused_fwd_train_f32(const int64_t* rowptr, const int32_t* col, const float* Wh, int64_t ldw,
                                const float* s, const float* t, int64_t n, int64_t nnz, int32_t H, int32_t Fp,
                                float alpha, int mode, int apply_elu, const float* col_mean,
                                const float* edge_keep, const gnn_gat_dropout* dropout,
                                float* out_pre, float* out_act /*nullable when apply_elu == 0*/, int64_t ldo,
                                float* row_max, float* row_sum,
                                const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                                int64_t batch_nodes, gnn_stream_t stream);
int gnn_gat_fused_fwd_train_bf16(const int64_t* rowptr, const int32_t* col, const void* Wh, int64_t ldw,
                                 const float* s, const float* t, int64_t n, int64_t nnz, int32_t H, int32_t Fp,
                                 float alpha, int mode, int apply_elu, const float* col_mean,
                                 const float* edge_keep, const gnn_gat_dropout* dropout,
                                 void* out_pre, void* out_act, int64_t ldo,
                                 float* row_max, float* row_sum,
                                 const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                                 int64_t batch_nodes, gnn_stream_t stream);

/* Backward.  out_pre is the pre-activation aggregate of the forward.  d_out is the gradient w.r.t. the
 * pre-activation aggregate when apply_elu == 0; with apply_elu > 0 it is the gradient w.r.t. the ACTIVATED
 * output of gnn_gat_fused_fwd_train_* and the ELU derivative chain is applied inside (d_pre: [n, ldo] scratch of
 * the feature type that receives the pre-activation gradient the two passes gather).  Produces
 *   d_s [n,H]                       (pass 1, row-parallel over the CSR),
 *   d_Wh [n,H*Fp] and d_t [n,H]     (pass 2, row-parallel over the transposed CSR rowptr_t/col_t).
 * Both passes have the forward kernel's shape, because the edge gradient
 *   dz_ij = a_ij * slope_ij * (keep_ij * <dOut_i, Wh_j> - D_i),  D_i = <dOut_i, out_pre_i>   (per head)
 * factorises into weighted row sums: d_s[i] = <dOut_i, sum_j w2_ij Wh_j> - D_i sum_j a_ij slope_ij,
 * d_t[j] = <Wh_j, sum_i w2_ij dOut_i> - sum_i a_ij slope_ij D_i, d_Wh[j] = sum_i w1_ij dOut_i (w1 = keep*a,
 * w2 = w1*slope).  This is the edge-gradient SDDMM (GAT/models/layers.py:59-61) and the transpose SpMM
 * (layers.py:63) without the dense N x N intermediate, without per-edge dot products, without a per-edge
 * stash between the passes and without atomics: ordered sums only.
 * perm_t (transposed slot -> forward edge slot) is read only when a dropout (edge_keep or seeded) is given.
 * row_scratch: [n,4,H] fp32 scratch (per-row s, max, 1/sum, D packed for the transposed pass). */
int gnn_gat_fused_bwd_f32(const int64_t* rowptr, const int32_t* col,
                          const int64_t* rowptr_t, const int32_t* col_t, const int64_t* perm_t /*nullable*/,
                          const float* Wh, int64_t ldw, const float* s, const float* t,
                          const float* row_max, const float* row_sum,
                          const float* out_pre, const float* d_out, int64_t ldo,
                          int64_t n, int32_t H, int32_t Fp, float alpha, int mode,
                          const float* edge_keep,
                          float* d_Wh, int64_t ld_dwh, float* d_s, float* d_t, float* row_scratch /*[n,4,H]*/,
                          int64_t nnz,
                          const int64_t* long_rows, int64_t n_long /*forward CSR*/,
                          const int64_t* long_rows_t, int64_t n_long_t /*transposed CSR*/, int64_t long_threshold,
                          int apply_elu, float* d_pre /*nullable when apply_elu == 0*/,
                          const gnn_gat_dropout* dropout /*nullable*/, int64_t batch_nodes,
                          gnn_stream_t stream);
/* Rectangular backward (fp32): the forward ran over n_rows CSR rows whose columns address n_cols >= n_rows table
 * rows of Wh / t.  The row-record kernel and pass 1 (d_s [n_rows,H]) walk the n_rows forward rows; pass 2 walks the
 * transposed [n_cols, n_rows] CSR (rowptr_t has n_cols + 1 entries) and writes d_Wh [n_cols, ld_dwh] and d_t
 * [n_cols, H] for every table row (zero for a row no edge reads) — its grid, its long-row list (long_rows_t) and its
 * cooperative-schedule choice follow n_cols.  row_scratch is [n_rows,4,H].  One graph only (no batch_nodes).
 * gnn_gat_fused_bwd_f32 is this function with n_rows == n_cols == n. */
int gnn_gat_fused_bwd_ex_f32(const int64_t* rowptr, const int32_t* col,
                             const int64_t* rowptr_t, const int32_t* col_t, const int64_t* perm_t /*nullable*/,
                             const float* Wh, int64_t ldw, const float* s, const float* t,
                             const float* row_max, const float* row_sum,
                             const float* out_pre, const float* d_out, int64_t ldo,
                             int64_t n_rows, int64_t n_cols, int32_t H, int32_t Fp, float alpha, int mode,
                             const float* edge_keep,
                             float* d_Wh, int64_t ld_dwh, float* d_s, float* d_t, float* row_scratch,
                             int64_t nnz,
                             const int64_t* long_rows, int64_t n_long,
                             const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold,
                             int apply_elu, float* d_pre, const gnn_gat_dropout* dropout /*nullable*/,
                             gnn_stream_t stream);

/* Batched AND rectangular graphs (fp32; bf16 below): a rank's row block of HAN's M metapath graphs, each renamed into one shared
 * combined column space of cols_per_graph >= rows_per_graph table rows ([own rows ; halo rows]).  The CSR is the
 * block diagonal of the M blocks: n = n_graphs*rows_per_graph rows, row r = graph r / rows_per_graph, and graph m's
 * column ids lie in [m*cols_per_graph, (m+1)*cols_per_graph), addressing row c - m*cols_per_graph of Wh's column block
 * m.  Wh is [cols_per_graph, ldw] and t [n_graphs*cols_per_graph, H]; s, the row statistics and d_s are
 * [n_graphs*rows_per_graph, H]; out / out_pre / d_out are [rows_per_graph, ldo] with graph m's columns at m*H*Fp;
 * d_Wh / d_t follow Wh / t.  The backward's transposed CSR has n_graphs*cols_per_graph rows (transposed row r is
 * graph r / cols_per_graph).
 * slot_shift (device int64 [n_graphs], nullable): the seeded dropout of graph m's local edge slot e is the one of slot
 * e + slot_shift[m] (after any edge_slot_base), so a row block draws exactly the mask of the whole batched graph
 * (on one GPU: Σ_{m'<m} nnz_{m'} + rowptr_m[lo] - the block's own first slot of graph m).  An explicit edge_keep
 * mask is in local slots.  Every row must have an edge (the rule for an empty row needs all N nodes).
 * struct_size = sizeof(gnn_gat_batch); 1 <= n_graphs <= 32, H*Fp <= 256.  With cols_per_graph == rows_per_graph and
 * no shift these entries compute the same bits as gnn_gat_fused_{fwd_train,bwd}_f32 with batch_nodes. */
typedef struct gnn_gat_batch {
  int32_t struct_size;
  int32_t n_graphs;
  int64_t rows_per_graph;
  int64_t cols_per_graph;
  const int64_t* slot_shift;
} gnn_gat_batch;
int gnn_gat_fused_fwd_batch_f32(const int64_t* rowptr, const int32_t* col, const float* Wh, int64_t ldw,
                                const float* s, const float* t, int64_t nnz, int32_t H, int32_t Fp,
                                float alpha, int mode, int apply_elu,
                                const float* edge_keep, const gnn_gat_dropout* dropout,
                                float* out_pre, float* out_act /*nullable when apply_elu == 0*/, int64_t ldo,
                                float* row_max, float* row_sum,
                                const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                                const gnn_gat_batch* batch, gnn_stream_t stream);
int gnn_gat_fused_bwd_batch_f32(const int64_t* rowptr, const int32_t* col,
                                const int64_t* rowptr_t, const int32_t* col_t, const int64_t* perm_t /*nullable*/,
                                const float* Wh, int64_t ldw, const float* s, const float* t,
                                const float* row_max, const float* row_sum,
                                const float* out_pre, const float* d_out, int64_t ldo,
                                int32_t H, int32_t Fp, float alpha, int mode,
                                const float* edge_keep,
                                float* d_Wh, int64_t ld_dwh, float* d_s, float* d_t, float* row_scratch,
                                int64_t nnz,
                                const int64_t* long_rows, int64_t n_long,
                                const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold,
                                int apply_elu, float* d_pre, const gnn_gat_dropout* dropout /*nullable*/,
                                const gnn_gat_batch* batch, gnn_stream_t stream);
/* bf16-feature variants (north_star: "bf16-feature variants within 1e-2"): Wh, out, out_pre, d_out and
 * d_Wh are bf16; the scores s/t, the softmax statistics and every accumulation stay fp32.
 * Same reference call site (GAT/models/layers.py:22-37). */
int gnn_gat_fused_fwd_bf16(const int64_t* rowptr, const int32_t* col, const void* Wh, int64_t ldw,
                           const float* s, const float* t, int64_t n, int64_t nnz, int32_t H, int32_t Fp,
                           float alpha, int mode, int apply_elu, const float* col_mean,
                           const float* edge_keep, void* out, int64_t ldo,
                           float* row_max, float* row_sum,
                           const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                           int64_t batch_nodes, gnn_stream_t stream);
int gnn_gat_fused_bwd_bf16(const int64_t* rowptr, const int32_t* col,
                           const int64_t* rowptr_t, const int32_t* col_t, const int64_t* perm_t,
                           const void* Wh, int64_t ldw, const float* s, const float* t,
                           const float* row_max, const float* row_sum,
                           const void* out_pre, const void* d_out, int64_t ldo,
                           int64_t n, int32_t H, int32_t Fp, float alpha, int mode,
                           const float* edge_keep,
                           void* d_Wh, int64_t ld_dwh, float* d_s, float* d_t, float* row_scratch,
                           int64_t nnz,
                           const int64_t* long_rows, int64_t n_long,
                           const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold,
                           int apply_elu, void* d_pre, const gnn_gat_dropout* dropout, int64_t batch_nodes,
                           gnn_stream_t stream);
/* bf16 rectangular and batched-rectangular forms (a rank's row block of a bf16 PartitionedGraph /
 * PartitionedMetapaths): the same argument lists and semantics as gnn_gat_fused_bwd_ex_f32 and
 * gnn_gat_fused_{fwd,bwd}_batch_f32, with the feature buffers bf16.  The non-batched rectangular forward is
 * gnn_gat_fused_fwd{,_train}_bf16 itself (Wh and t are read only through col).  With cols_per_graph ==
 * rows_per_graph and no shift the batched entries compute the same bits as gnn_gat_fused_{fwd_train,bwd}_bf16 with
 * batch_nodes. */
int gnn_gat_fused_bwd_ex_bf16(const int64_t* rowptr, const int32_t* col,
                              const int64_t* rowptr_t, const int32_t* col_t, const int64_t* perm_t /*nullable*/,
                              const void* Wh, int64_t ldw, const float* s, const float* t,
                              const float* row_max, const float* row_sum,
                              const void* out_pre, const void* d_out, int64_t ldo,
                              int64_t n_rows, int64_t n_cols, int32_t H, int32_t Fp, float alpha, int mode,
                              const float* edge_keep,
                              void* d_Wh, int64_t ld_dwh, float* d_s, float* d_t, float* row_scratch,
                              int64_t nnz,
                              const int64_t* long_rows, int64_t n_long,
                              const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold,
                              int apply_elu, void* d_pre, const gnn_gat_dropout* dropout /*nullable*/,
                              gnn_stream_t stream);
int gnn_gat_fused_fwd_batch_bf16(const int64_t* rowptr, const int32_t* col, const void* Wh, int64_t ldw,
                                 const float* s, const float* t, int64_t nnz, int32_t H, int32_t Fp,
                                 float alpha, int mode, int apply_elu,
                                 const float* edge_keep, const gnn_gat_dropout* dropout,
                                 void* out_pre, void* out_act /*nullable when apply_elu == 0*/, int64_t ldo,
                                 float* row_max, float* row_sum,
                                 const int64_t* long_rows, int64_t n_long, int64_t long_threshold,
                                 const gnn_gat_batch* batch, gnn_stream_t stream);
int gnn_gat_fused_bwd_batch_bf16(const int64_t* rowptr, const int32_t* col,
                                 const int64_t* rowptr_t, const int32_t* col_t, const int64_t* perm_t /*nullable*/,
                                 const void* Wh, int64_t ldw, const float* s, const float* t,
                                 const float* row_max, const float* row_sum,
                                 const void* out_pre, const void* d_out, int64_t ldo,
                                 int32_t H, int32_t Fp, float alpha, int mode,
                                 const float* edge_keep,
                                 void* d_Wh, int64_t ld_dwh, float* d_s, float* d_t, float* row_scratch,
                                 int64_t nnz,
                                 const int64_t* long_rows, int64_t n_long,
                                 const int64_t* long_rows_t, int64_t n_long_t, int64_t long_threshold,
                                 int apply_elu, void* d_pre, const gnn_gat_dropout* dropout /*nullable*/,
                                 const gnn_gat_batch* batch, gnn_stream_t stream);

/* ---- HAN semantic attention: everything around its one GEMM -------------------- */
/* HAN/models/SemanticAttention.py:15-20:
 *     w = project(z).mean(0); beta = softmax(w, dim=0); out = (beta.expand(N,M,1) * z).sum(1)
 * with project = Linear(D,K) -> Tanh -> Linear(K,1,bias=False) (SemanticAttention.py:8-12).
 * The caller keeps P = z·W1^T [N*M, K] (row n*M+m) as a library GEMM; these four launches replace the tanh, the
 * K->1 projection, the mean over nodes, the softmax over the M metapaths, the weighted sum and all their
 * gradients.  z and dz are contiguous [N, M, D]; M <= 32, K <= 256.  Ordered sums (deterministic).
 * workspace: gnn_semantic_workspace_size(K) bytes, 16-byte aligned, ZERO before its first use (its first word is a
 * ticket counter every call leaves at zero again); calls sharing a workspace must be stream-ordered. */
int64_t gnn_semantic_workspace_size(int32_t K);
/* scores[m] = 1/N sum_n sum_k q[k] tanh(P[n*M+m, k] + bias[k]) (bias nullable); beta = softmax_M(scores) */
int gnn_semantic_scores_f32(const float* P, int64_t ldp, const float* bias /*[K]*/, const float* q /*[K]*/,
                            int64_t N, int32_t M, int32_t K, float* scores /*[M]*/, float* beta /*[M]*/,
                            void* workspace, int64_t workspace_bytes, gnn_stream_t stream);
/* out[n, :] = sum_m beta[m] z[n, m, :] */
int gnn_semantic_combine_f32(const float* beta, const float* z, int64_t N, int32_t M, int32_t D,
                             float* out /*[N, D]*/, gnn_stream_t stream);
/* dz[n, m, :] = beta[m] d_out[n, :] (the direct term; the caller adds dP·W1);
 * d_scores_over_n[m] = beta[m] (dbeta[m] - sum_j beta[j] dbeta[j]) / N with dbeta[m] = sum_n <d_out[n], z[n, m]> */
int gnn_semantic_combine_bwd_f32(const float* d_out, const float* z, const float* beta, int64_t N, int32_t M,
                                 int32_t D, float* dz, float* d_scores_over_n /*[M]*/, void* workspace,
                                 int64_t workspace_bytes, gnn_stream_t stream);
/* dP[r, k] = d_scores_over_n[r % M] q[k] (1 - tanh^2(P[r, k] + bias[k])); dq[k] = sum_r d_scores_over_n[r % M] tanh(.);
 * dbias[k] = sum_r dP[r, k] (dbias nullable) */
int gnn_semantic_scores_bwd_f32(const float* P, int64_t ldp, const float* bias, const float* q,
                                const float* d_scores_over_n, int64_t N, int32_t M, int32_t K,
                                float* dP, int64_t lddp, float* dq /*[K]*/, float* dbias /*[K]*/,
                                void* workspace, int64_t workspace_bytes, gnn_stream_t stream);
/* The two node sums split at the rank boundary (rows of one rank; N = its row count, 0 allowed): the caller adds
 * the ranks' [M] partials in rank order and finalizes with the GLOBAL node count n_total.  With one part, partial +
 * finalize computes the same bits as the fused entry.
 *   scores_partial:   sums[m] = sum_n sum_k q[k] tanh(P[n*M+m, k] + bias[k]) (the fused entry's sum before / N)
 *   scores_finalize:  scores = sums / n_total, beta = softmax_M(scores)
 *   combine_bwd_partial:  dz[n, m, :] = beta[m] d_out[n, :], dbeta[m] = sum_n <d_out[n], z[n, m]>
 *   combine_bwd_finalize: d_scores_over_n[m] = beta[m] (dbeta[m] - sum_j beta[j] dbeta[j]) / n_total
 * gnn_semantic_scores_bwd_f32 then takes d_scores_over_n over the rank's rows (its dq / dbias are the rank's share). */
int gnn_semantic_scores_partial_f32(const float* P, int64_t ldp, const float* bias, const float* q, int64_t N,
                                    int32_t M, int32_t K, float* sums /*[M]*/, void* workspace,
                                    int64_t workspace_bytes, gnn_stream_t stream);
int gnn_semantic_scores_finalize_f32(const float* sums, int64_t n_total, int32_t M, float* scores, float* beta,
                                     gnn_stream_t stream);
int gnn_semantic_combine_bwd_partial_f32(const float* d_out, const float* z, const float* beta, int64_t N, int32_t M,
                                         int32_t D, float* dz, float* dbeta /*[M]*/, void* workspace,
                                         int64_t workspace_bytes, gnn_stream_t stream);
int gnn_semantic_combine_bwd_finalize_f32(const float* dbeta, const float* beta, int64_t n_total, int32_t M,
                                          float* d_scores_over_n, gnn_stream_t stream);

/* ---- synthetic graphs for the benchmark shapes (SURVEY.md §8d) ---------------- */
/* Power-law CSR generated on the device, row by row, from a counter-based hash of
 * (seed,row,k): degrees ~ truncated Pareto with the given mean, targets skewed to
 * low ids (hubs), columns ascending within a row, one self-loop per row, values
 * d_i^-1/2 d_j^-1/2 as GCN/data_utils.py:54-60 computes them.  Two steps. */
int gnn_synth_powerlaw_degrees(int64_t n_rows, int64_t row_offset, double mean_degree, double exponent,
                               int64_t max_degree, uint64_t seed, int64_t* deg /*[n_rows]*/, gnn_stream_t stream);
int gnn_synth_powerlaw_fill(int64_t n_rows, int64_t row_offset, int64_t n_cols, const int64_t* rowptr,
                            double skew, double p_local /*share of edges within +-|window| of the row*/,
                            int64_t window /*<0: also scatter the hub ids by a fixed bijection*/,
                            uint64_t seed, int32_t* col, gnn_stream_t stream);
int gnn_synth_gcn_values(int64_t n_rows, int64_t row_offset, const int64_t* rowptr, const int32_t* col,
                         const int64_t* deg_all /*[n_cols] global degrees*/, float* val, gnn_stream_t stream);

/* ---- multi-GPU halo exchange over NVLink peer memory (SURVEY.md §8e) ------------ */
/* Copy-engine transfer between two device allocations of this process' address space (a peer's
 * gnn_peer_open mapping included): cudaMemcpyAsync device-to-device on `stream` (zero SMs).  Used for
 * the contiguous segments of the partitioned backward's reverse halo exchange and by transport="ce". */
int gnn_peer_copy_async(void* dst, const void* src, size_t bytes, gnn_stream_t stream);

/* Peer buffers are plain cudaMalloc allocations (zero-initialised) exported with CUDA IPC, one
 * process per GPU: gnn_peer_alloc on the owner, gnn_peer_open of the 64-byte handle on every peer. */
int gnn_peer_alloc(size_t bytes, void** dev_ptr, void* ipc_handle_64B_host);
int gnn_peer_open(const void* ipc_handle_64B_host, void** dev_ptr);
int gnn_peer_close(void* dev_ptr);
int gnn_peer_free(void* dev_ptr);

/* Fused pack + transfer of halo rows.  For every peer q the rows
 *   send_rows[seg_begin[q] + k], k in [0, seg_rows[q])      (send_rows == NULL: local rows seg_begin[q] + k)
 * of the local X [*, ldx] (elem_size 4 = fp32, 2 = bf16 wire for the bf16 variant) are written to row
 * dst_row[q] + k of peer q's buffer peer_dst[q] [*, ld_dst] over NVLink, segments served in rotated
 * order starting at opts->first_peer.  A call moves ONE WAVE: the caller passes the sub-range of each
 * peer segment that belongs to the wave and signals the peers afterwards (gnn_peer_signal).
 * Every scheduling choice is an explicit argument (no process-global knobs):
 *   mover          0 auto | 1 vector loads/stores | 2 TMA bulk copies (rows must be 16-byte multiples
 *                  <= 16 KB and ld_dst == F; GNN_ERR_UNSUPPORTED otherwise)
 *   ctas           CTAs launched (0 = one per SM)
 *   warps_per_cta  0 = default (TMA: 1 — a 48 KB ring next to the SpMM CTAs of every SM; vector: 8)
 *   claim_smem_bytes  vector mover only: dynamic shared memory each CTA claims so that a kernel asking
 *                  for gnn_spmm_opts.exclusion_smem_bytes cannot share its SM (SM partition)
 * opts == NULL selects the defaults.  struct_size = sizeof(gnn_halo_opts). */
typedef struct gnn_halo_opts {
  int32_t struct_size;
  int32_t mover;
  int32_t ctas;
  int32_t warps_per_cta;
  int32_t claim_smem_bytes;
  int32_t first_peer;
} gnn_halo_opts;
int gnn_halo_push(const void* X, int64_t ldx, int32_t F, int32_t elem_size,
                  const int32_t* send_rows /*nullable*/,
                  const int64_t* seg_begin_host /*[n_peers]*/, const int64_t* seg_rows_host /*[n_peers]*/,
                  void* const* peer_dst_host /*[n_peers] device ptrs*/, const int64_t* dst_row_host /*[n_peers]*/,
                  int64_t ld_dst, int32_t n_peers, const gnn_halo_opts* opts, gnn_stream_t stream);

/* All waves of a step in ONE launch of the TMA mover, the arrival flags raised from inside the kernel:
 * seg_table_dev is a device int64 [n_segs][5] table (first send_rows entry | rows | destination ADDRESS
 * of the segment's first row (contiguous rows of F*elem_size bytes) | first chunk id | wave), sorted by
 * wave; a chunk is gnn_halo_rows_per_stage(F*elem_size) rows and never straddles a segment; n_chunks is
 * the total.  When the last warp of the grid has finished wave w (own bulk stores performed, fenced) it
 * stores flag_base + w + 1 into slot my_slot of every peer's flag array (gnn_peer_wait on the other side).
 * wave_done_dev: n_waves device counters (scratch, reset by the call).  opts: ctas / warps_per_cta. */
int gnn_halo_rows_per_stage(int32_t row_bytes);
int gnn_halo_push_waves(const void* X, int64_t ldx, int32_t F, int32_t elem_size, const int32_t* send_rows /*nullable*/,
                        const int64_t* seg_table_dev, int32_t n_segs, int32_t n_waves, int64_t n_chunks,
                        uint32_t* wave_done_dev, uint32_t* const* peer_flags_host /*[n_peers] device ptrs*/,
                        int32_t n_peers, int32_t my_slot, uint32_t flag_base, const gnn_halo_opts* opts,
                        gnn_stream_t stream);

/* Per-peer arrival flags: monotonic uint32 counters living in peer memory (one array of n_peers slots
 * per rank, slot p written by rank p).  gnn_peer_signal stores `value` into slot my_slot of every
 * peer's array (release, system scope) — stream-ordered behind the pushes it announces.
 * gnn_peer_wait makes `stream` wait (a one-warp kernel polling with acquire loads) until every slot
 * except skip_slot has reached `value`; after timeout_ms it gives up and writes 1 + the late slot to
 * *status (nullable) instead of hanging the GPU.  These replace a collective barrier: the consumer of
 * wave w waits only for wave w's flags. */
int gnn_peer_signal(uint32_t* const* peer_flags_host /*[n_peers] device ptrs*/, int32_t n_peers, int32_t my_slot,
                    int32_t skip_peer, uint32_t value, gnn_stream_t stream);
int gnn_peer_wait(const uint32_t* flags, int32_t n_slots, int32_t skip_slot, uint32_t value,
                  uint32_t* status /*nullable device word*/, int64_t timeout_ms, gnn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GNN_B200_H */
