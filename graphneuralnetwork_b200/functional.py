"""torch.autograd.Function wrappers over the C ABI (the seam of SURVEY.md §1:
drop-in nn.Module.forward -> autograd.Function -> libgnn_b200.so -> sm_100a kernels).

Every function here launches the CUDA library on the caller's current stream; a CPU
tensor raises.  torch supplies device memory, streams and autograd bookkeeping only.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from .graph import CSRGraph, _p, _require_cuda, _stream_ptr, index_block_transpose
from .partition import ShardedTable


def _rowmajor(x: torch.Tensor) -> torch.Tensor:
    """Rows must be unit-stride in the feature dimension; the row stride is free."""
    if x.dim() != 2:
        raise _lib.GnnError(f"expected a 2-D feature matrix, got shape {tuple(x.shape)}")
    if x.stride(1) != 1 and x.shape[1] > 1:
        x = x.contiguous()
    if x.shape[0] > 1 and x.stride(0) < x.shape[1]:
        x = x.contiguous()
    return x


def _ld(x: torch.Tensor) -> int:
    return x.stride(0) if x.shape[0] > 1 else max(x.shape[1], 1)


def _padded_empty(rows: int, F: int, dtype, device) -> torch.Tensor:
    """[rows, F] view of a buffer whose row stride is a multiple of 16 bytes."""
    per16 = 16 // torch.empty((), dtype=dtype).element_size()
    ld = (F + per16 - 1) // per16 * per16
    return torch.empty((rows, ld), dtype=dtype, device=device)[:, :F]


# --------------------------------------------------------------------------------------
# GCN: Y = Â·X
# --------------------------------------------------------------------------------------
def spmm_raw(g: CSRGraph, X: torch.Tensor, out: Optional[torch.Tensor] = None, planned: bool = True,
             accumulate: bool = False, bias: Optional[torch.Tensor] = None, relu: bool = False) -> torch.Tensor:
    """Y = Â·X (or Y += Â·X into `out`) through gnn_spmm_csr_* (no autograd).
    bias / relu: fused epilogue Y = relu?(Â·X + bias) of the planned entry point."""
    _require_cuda(X)
    lib = _lib.load()
    X = _rowmajor(X)
    if X.shape[0] != g.n_cols:
        raise _lib.GnnError(f"spmm: X has {X.shape[0]} rows, adjacency has {g.n_cols} columns")
    F = X.shape[1]
    if out is None:
        out = torch.empty((g.n_rows, F), dtype=X.dtype, device=X.device)
    st = _stream_ptr()
    if X.dtype not in (torch.float32, torch.bfloat16):
        raise _lib.GnnError(f"spmm: unsupported dtype {X.dtype} (fp32 and bf16 only)")
    f32 = X.dtype == torch.float32
    plan = g.long_row_plan() if planned else None
    if bias is not None:
        _require_cuda(bias)
        if bias.dtype != torch.float32 or bias.numel() != F:
            raise _lib.GnnError(f"spmm: bias must be fp32 with {F} entries")
        bias = bias.contiguous()
    if planned or accumulate or bias is not None or relu:
        lr, thr, chunk_off, n_chunks, chunk, ws = plan if plan is not None else (None, 0, None, 0, 0, None)
        fn = lib.gnn_spmm_csr_planned_f32 if f32 else lib.gnn_spmm_csr_planned_bf16
        _lib.check(fn(_p(g.rowptr), _p(g.col), _p(g.val), _p(_nonempty(X)), _p(out), g.n_rows, g.n_cols, F, _ld(X),
                      _ld(out), _p(lr), 0 if lr is None else lr.numel(), thr, _p(chunk_off), n_chunks, chunk,
                      1 if accumulate else 0, g.rows_per_team() if planned else 0, _p(bias), 1 if relu else 0,
                      _p(ws), 0 if ws is None else ws.numel(), st),
                   "gnn_spmm_csr_planned")
    else:
        fn = lib.gnn_spmm_csr_f32 if f32 else lib.gnn_spmm_csr_bf16
        _lib.check(fn(_p(g.rowptr), _p(g.col), _p(g.val), _p(_nonempty(X)), _p(out), g.n_rows, g.n_cols, F, _ld(X),
                      _ld(out), st), "gnn_spmm_csr")
    return out


def spmm_ex(g: CSRGraph, X: torch.Tensor, out: torch.Tensor, row_map: Optional[torch.Tensor] = None,
            accumulate: bool = False, accumulate_prefix: int = 0, X2: Optional[torch.Tensor] = None, split: int = 0,
            exclusion_smem: int = 0, bias: Optional[torch.Tensor] = None, relu: bool = False,
            epilogue_skip_prefix: int = 0) -> torch.Tensor:
    """Row-subset / two-table SpMM (gnn_spmm_csr_ex_*, no autograd): `g` is a CSR that is COMPACT over the
    selected rows; compact row r writes `out[row_map[r]]` (row_map None: out[r]); rows below
    `accumulate_prefix` (or all, with accumulate) add into `out`; column ids >= `split` read row
    (c - split) of X2.  bias / relu: the epilogue relu?(. + bias), applied after the add of accumulating rows,
    except on compact rows below `epilogue_skip_prefix`.  The consumers of the partitioned SpMM's waves
    (partition.py)."""
    import ctypes as C
    _require_cuda(X, out, row_map, X2, bias)
    lib = _lib.load()
    X = _rowmajor(X)
    if X.dtype not in (torch.float32, torch.bfloat16) or out.dtype != X.dtype:
        raise _lib.GnnError(f"spmm_ex: unsupported dtypes {X.dtype} / {out.dtype}")
    F = X.shape[1]
    n_src = X.shape[0] + (X2.shape[0] if X2 is not None else 0)
    if X2 is None and X.shape[0] != g.n_cols:
        raise _lib.GnnError(f"spmm_ex: X has {X.shape[0]} rows, adjacency has {g.n_cols} columns")
    if X2 is not None and (X2.dtype != X.dtype or X2.shape[1] != F or split != X.shape[0] or n_src < g.n_cols):
        raise _lib.GnnError("spmm_ex: X2 must match X in dtype and width, split must equal X.shape[0] and the "
                            "two tables must cover the adjacency's columns")
    if row_map is not None and (row_map.dtype != torch.int32 or row_map.numel() != g.n_rows):
        raise _lib.GnnError("spmm_ex: row_map must be int32 with one entry per compact row")
    if out.stride(1) != 1 or out.shape[1] != F:
        raise _lib.GnnError("spmm_ex: `out` must be [*, F] with unit column stride")
    if bias is not None:
        if bias.dtype != torch.float32 or bias.numel() != F:
            raise _lib.GnnError(f"spmm_ex: bias must be fp32 with {F} entries")
        bias = bias.contiguous()
    plan = g.long_row_plan()
    lr, thr, chunk_off, n_chunks, chunk, ws = plan if plan is not None else (None, 0, None, 0, 0, None)
    o = _lib.SpmmOpts()
    o.struct_size = C.sizeof(_lib.SpmmOpts)
    o.accumulate = 1 if accumulate else 0
    o.accumulate_prefix = int(accumulate_prefix)
    o.rows_per_team = g.rows_per_team()
    o.row_map = _p(row_map)
    if X2 is not None:
        X2 = _rowmajor(X2)
        o.X2, o.ldx2, o.split = _p(X2), _ld(X2), int(split)
    o.long_rows, o.n_long, o.long_threshold = _p(lr), 0 if lr is None else lr.numel(), thr
    o.chunk_off, o.n_chunks, o.chunk_edges = _p(chunk_off), n_chunks, chunk
    o.exclusion_smem_bytes = int(exclusion_smem)
    o.bias, o.relu, o.epilogue_skip_prefix = _p(bias), 1 if relu else 0, int(epilogue_skip_prefix)
    o.workspace, o.workspace_bytes = _p(ws), 0 if ws is None else ws.numel()
    fn = lib.gnn_spmm_csr_ex_f32 if X.dtype == torch.float32 else lib.gnn_spmm_csr_ex_bf16
    _lib.check(fn(_p(g.rowptr), _p(g.col), _p(g.val), _p(X), _p(out), g.n_rows, max(g.n_cols, n_src), F, _ld(X),
                  _ld(out), C.byref(o), _stream_ptr()), "gnn_spmm_csr_ex")
    return out


class _SpmmFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X, g: CSRGraph):
        ctx.g = g
        return spmm_raw(g, X)

    @staticmethod
    def backward(ctx, dY):
        # autograd of torch.spmm (GCN/GCN.py:43): dX = Âᵀ·dY, no gradient to Â
        dX = spmm_raw(ctx.g.transpose(), dY.contiguous()) if ctx.needs_input_grad[0] else None
        return dX, None


def spmm(g: CSRGraph, X: torch.Tensor) -> torch.Tensor:
    """Y = Â·X with autograd (replaces torch.spmm(adj, support), GCN/GCN.py:43)."""
    return _SpmmFn.apply(X, g)


def sddmm(rows: torch.Tensor, cols: torch.Tensor, A: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    """out[e] = <A[rows[e]], B[cols[e]]> (gnn_sddmm_coo_f32): the edge-gradient contraction, nnz dot
    products instead of the dense `A @ B.T` of GAT/models/layers.py:59-61.  No autograd."""
    _require_cuda(rows, cols, A, B)
    lib = _lib.load()
    A, B = _rowmajor(A), _rowmajor(B)
    if A.dtype != torch.float32 or B.dtype != torch.float32 or A.shape[1] != B.shape[1]:
        raise _lib.GnnError(f"sddmm: fp32 operands with equal widths expected, got {tuple(A.shape)} {tuple(B.shape)}")
    if rows.dtype != cols.dtype or rows.dtype not in (torch.int32, torch.int64) or rows.numel() != cols.numel():
        raise _lib.GnnError("sddmm: rows / cols must be int32 or int64 arrays of equal length")
    rows, cols = rows.contiguous(), cols.contiguous()
    out = torch.empty(rows.numel(), dtype=torch.float32, device=A.device)
    _lib.check(lib.gnn_sddmm_coo_f32(_p(rows), _p(cols), 32 if rows.dtype == torch.int32 else 64, rows.numel(), _p(A),
                                     _ld(A), _p(B), _ld(B), A.shape[1], _p(out), _stream_ptr()), "gnn_sddmm_coo_f32")
    return out


class _SpmmValuesFn(torch.autograd.Function):
    """Y = S·X where the VALUES of S are an autograd input (pattern fixed, CSR order).
    Backward: dX = Sᵀ·dY (transpose SpMM on the cached transposed pattern),
              dval[e] = <dY[row(e)], X[col(e)]> (edge-gradient SDDMM)."""

    @staticmethod
    def forward(ctx, val, X, pattern: CSRGraph):
        ctx.pattern = pattern
        ctx.save_for_backward(val, X)
        return spmm_raw(pattern.with_values(val), X)

    @staticmethod
    def backward(ctx, dY):
        val, X = ctx.saved_tensors
        g = ctx.pattern
        dY = dY.contiguous()
        dval = dX = None
        if ctx.needs_input_grad[0]:
            dval = sddmm(g.edge_rows(), g.col, dY, X)
        if ctx.needs_input_grad[1]:
            gt = g.transpose()  # pattern transpose + permutation, cached on the pattern graph
            dX = spmm_raw(gt.with_values(val.detach()[g.perm_t]), dY)
        return dval, dX, None


def spmm_values(pattern: CSRGraph, val: torch.Tensor, X: torch.Tensor) -> torch.Tensor:
    """Y = S·X with autograd into BOTH the edge values `val` (CSR order of `pattern`) and X:
    the sparse product of GAT/models/layers.py:43-64 (SpecialSpmmFunction) and of a GCN over a
    learned adjacency (GTN/models/GTN.py:49-52)."""
    _require_cuda(val, X)
    if val.dtype != torch.float32 or val.numel() != pattern.nnz:
        raise _lib.GnnError(f"spmm_values: {pattern.nnz} fp32 edge values expected")
    return _SpmmValuesFn.apply(val, X, pattern)


def _col_or_dummy(g: CSRGraph) -> torch.Tensor:
    # an empty tensor has no address; the kernels read no column of a graph without entries
    return g.col if g.nnz else torch.zeros(1, dtype=torch.int32, device=g.device)


def _nonempty(t: torch.Tensor) -> torch.Tensor:
    # an empty tensor (the permutation of a graph without entries, the X of a graph without columns) has no address;
    # the kernels read none of it
    return t if t.numel() else torch.zeros(1, dtype=t.dtype, device=t.device)


def _spgemm_ws(n_a: int, k: int, dev) -> torch.Tensor:
    return torch.empty(max(_lib.load().gnn_spgemm_workspace_size(n_a, k), 1), dtype=torch.uint8, device=dev)


def spgemm_values_raw(A: CSRGraph, a_val: torch.Tensor, B: CSRGraph, b_val: torch.Tensor, C_pattern: CSRGraph,
                      path_rows: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Values [C_pattern.nnz, C] of A·B on C_pattern, channel by channel (gnn_spgemm_values_f32, no autograd).
    B is read through its cached transpose.  path_rows: an int64[2] CUDA tensor that receives the rows each
    kernel path took (warp, CTA)."""
    lib = _lib.load()
    C = a_val.shape[1]
    c_val = torch.empty((C_pattern.nnz, C), dtype=torch.float32, device=a_val.device)
    Bt = B.transpose()
    ws = _spgemm_ws(A.n_rows, A.n_cols, a_val.device)
    _lib.check(lib.gnn_spgemm_values_f32(
        _p(A.rowptr), _p(_col_or_dummy(A)), _p(a_val), A.n_rows, A.n_cols, A.nnz,
        _p(Bt.rowptr), _p(_col_or_dummy(Bt)), _p(_nonempty(B.perm_t)), _p(b_val), B.n_cols, B.nnz,
        _p(C_pattern.rowptr), _p(_col_or_dummy(C_pattern)), _p(_nonempty(c_val)), C, _p(path_rows),
        _p(ws), ws.numel(), _stream_ptr()), "gnn_spgemm_values_f32")
    return c_val


def spgemm_values_bwd_raw(A: CSRGraph, a_val: torch.Tensor, B: CSRGraph, b_val: torch.Tensor, C_pattern: CSRGraph,
                          dc: torch.Tensor, need_a: bool = True, need_b: bool = True,
                          path_rows: Optional[torch.Tensor] = None):
    """(dA [A.nnz, C], dB [B.nnz, C]) of spgemm_values_raw for the output gradient dc, each restricted to its
    operand's pattern (gnn_spgemm_values_bwd_f32; None where not asked for).  Aᵀ and Cᵀ are the cached transposes.
    path_rows: an int64[4] CUDA tensor, the rows each path took for dA and then for dB."""
    lib = _lib.load()
    C = dc.shape[1]
    dev = dc.device
    da = torch.zeros((A.nnz, C), dtype=torch.float32, device=dev) if need_a else None
    db = torch.zeros((B.nnz, C), dtype=torch.float32, device=dev) if need_b else None
    da_k = None if da is None else _nonempty(da)  # rows without entries still take their path
    db_k = None if db is None else _nonempty(db)
    if da_k is None and db_k is None:
        return da, db
    At = A.transpose() if db_k is not None else None
    Ct = C_pattern.transpose() if db_k is not None else None
    ws = _spgemm_ws(A.n_rows, A.n_cols, dev)
    _lib.check(lib.gnn_spgemm_values_bwd_f32(
        _p(A.rowptr), _p(_col_or_dummy(A)), _p(a_val), A.n_rows, A.n_cols, A.nnz,
        None if At is None else _p(At.rowptr), None if At is None else _p(_col_or_dummy(At)),
        None if At is None else _p(_nonempty(A.perm_t)),
        _p(B.rowptr), _p(_col_or_dummy(B)), _p(b_val), B.n_cols, B.nnz,
        _p(C_pattern.rowptr), _p(_col_or_dummy(C_pattern)),
        None if Ct is None else _p(Ct.rowptr), None if Ct is None else _p(_col_or_dummy(Ct)),
        None if Ct is None else _p(_nonempty(C_pattern.perm_t)), _p(_nonempty(dc)), C_pattern.nnz, C,
        _p(da_k), _p(db_k), _p(path_rows), _p(ws), ws.numel(), _stream_ptr()), "gnn_spgemm_values_bwd_f32")
    return da, db


class _SpgemmValuesFn(torch.autograd.Function):
    """C = A·B with C channels of values on fixed patterns; gradients into both value tensors, on their patterns."""

    @staticmethod
    def forward(ctx, a_val, b_val, A: CSRGraph, B: CSRGraph, C_pattern: CSRGraph):
        ctx.graphs = (A, B, C_pattern)
        ctx.save_for_backward(a_val, b_val)
        return spgemm_values_raw(A, a_val, B, b_val, C_pattern)

    @staticmethod
    def backward(ctx, dc):
        a_val, b_val = ctx.saved_tensors
        A, B, C_pattern = ctx.graphs
        da, db = spgemm_values_bwd_raw(A, a_val, B, b_val, C_pattern, dc.contiguous(), ctx.needs_input_grad[0],
                                       ctx.needs_input_grad[1])
        return da, db, None, None, None


def spgemm_values(A: CSRGraph, a_val: torch.Tensor, B: CSRGraph, b_val: torch.Tensor,
                  C_pattern: CSRGraph) -> torch.Tensor:
    """Values [C_pattern.nnz, C] of the sparse product A·B on the pattern C_pattern (from `CSRGraph.pattern_product`),
    each of the C channels its own product: the learned metapath composition of GTN (GTN/models/GTLayer.py, there a
    dense torch.bmm).  a_val [A.nnz, C] and b_val [B.nnz, C] are fp32 in CSR slot order; autograd reaches both.
    The rows of A, B and C_pattern hold ascending unique column ids (what pattern products and the CSR builders
    produce).  Every output entry is one sum in ascending order of the inner index: the same bits on every run."""
    _require_cuda(a_val, b_val, A.rowptr, B.rowptr, C_pattern.rowptr)
    if a_val.dtype != torch.float32 or b_val.dtype != torch.float32:
        raise _lib.GnnError(f"spgemm_values: fp32 values expected, got {a_val.dtype} / {b_val.dtype}")
    if a_val.dim() != 2 or b_val.dim() != 2 or a_val.shape != (A.nnz, a_val.shape[1]) \
            or b_val.shape != (B.nnz, a_val.shape[1]):
        raise _lib.GnnError(f"spgemm_values: values [A.nnz = {A.nnz}, C] and [B.nnz = {B.nnz}, C] expected, got "
                            f"{tuple(a_val.shape)} / {tuple(b_val.shape)}")
    if A.n_cols != B.n_rows or C_pattern.n_rows != A.n_rows or C_pattern.n_cols != B.n_cols:
        raise _lib.GnnError(f"spgemm_values: [{A.n_rows}, {A.n_cols}]·[{B.n_rows}, {B.n_cols}] does not give the "
                            f"[{C_pattern.n_rows}, {C_pattern.n_cols}] pattern")
    return _SpgemmValuesFn.apply(a_val.contiguous(), b_val.contiguous(), A, B, C_pattern)


def column_normalize(pattern: CSRGraph, val: torch.Tensor, reduce=None) -> torch.Tensor:
    """val [nnz, C] on `pattern` with every column of every channel divided by its sum (inf -> 0), autograd into
    val: the column normalisation of GTN's `norm` (GTN/models/GTN.py:7-19) on a pattern without its diagonal.  The
    column sums are the ordered row sums of the cached transpose (one SpMM per channel), not an atomic scatter.
    reduce: on a row block of the pattern (partition.PartitionedRelationStack) the sums are partial, and
    `reduce([n_cols, C])` returns the sums over every rank's rows (`rank_all_reduce`); None keeps them as they are."""
    t = pattern.transpose()
    ones = torch.ones((pattern.n_rows, 1), dtype=torch.float32, device=val.device)
    perm = pattern.perm_t
    sums = torch.cat([spmm_values(t, val[:, c][perm].contiguous(), ones) for c in range(val.shape[1])], dim=1)
    if reduce is not None:
        sums = reduce(sums)
    inv = sums.pow(-1)
    inv = torch.where(torch.isinf(inv), torch.zeros_like(inv), inv)
    return val * inv[pattern.col.long()]


def peer_reduce_rows_raw(src_ptrs, ld_src: int, F: int, row_lo: int, row_hi: int, out: torch.Tensor,
                         relu: bool = False) -> torch.Tensor:
    """out[r, :F] = relu?(Σ_q src_q[row_lo + r, :F]) over the fp32 row buffers at the device addresses `src_ptrs`
    (this process' or peers' IPC mappings), added in list order in fp32 (gnn_peer_reduce_rows_f32, no autograd)."""
    import ctypes as C
    _require_cuda(out)
    if out.dtype != torch.float32 or out.dim() != 2 or out.shape[0] < row_hi - row_lo or out.shape[1] < F \
            or (out.shape[1] > 1 and out.stride(1) != 1):
        raise _lib.GnnError(f"peer_reduce_rows: fp32 out of at least [{row_hi - row_lo}, {F}] expected, got "
                            f"{out.dtype} {tuple(out.shape)}")
    if row_hi == row_lo:
        return out
    src = (C.c_void_p * len(src_ptrs))(*[int(p) for p in src_ptrs])
    _lib.check(_lib.load().gnn_peer_reduce_rows_f32(src, len(src_ptrs), ld_src, F, row_lo, row_hi, _p(out), _ld(out),
                                                    1 if relu else 0, _stream_ptr()), "gnn_peer_reduce_rows_f32")
    return out


class _RankAllReduceFn(torch.autograd.Function):
    """y = Σ over the ranks of x, added in rank order (partition.PeerRowReduce.all_reduce at `site`); every rank gets
    the same bits.  Backward: the same all-reduce of dy (site + "_bwd"), since every rank's y depends on every x."""

    @staticmethod
    def forward(ctx, x, red, site: str):
        ctx.red, ctx.site = red, site
        return red.all_reduce(site, x.contiguous())

    @staticmethod
    def backward(ctx, dy):
        # always run: the reduction is a collective every rank takes part in
        return ctx.red.all_reduce(ctx.site + "_bwd", dy.contiguous()), None, None


def rank_all_reduce(red, site: str, x: torch.Tensor) -> torch.Tensor:
    """Σ over the ranks of the fp32 [rows, F] partial x, in rank order, with autograd (collective, both ways)."""
    _require_cuda(x)
    return _RankAllReduceFn.apply(x, red, site)


class _RowReduceScatterFn(torch.autograd.Function):
    """y = relu?(Σ over the ranks of x)[own rows] (partition.PeerRowReduce.reduce_scatter, ReLU fused into the reduce).
    Backward: dz = dy ⊙ [y > 0], then the all-gather of every rank's dz (site + "_bwd"): each rank's x reaches every
    output row."""

    @staticmethod
    def forward(ctx, x, red, site: str, relu: bool):
        y = red.reduce_scatter(site, x.contiguous(), relu)
        ctx.red, ctx.site, ctx.relu = red, site, relu
        if relu:
            ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        dz = dy
        if ctx.relu:
            (y,) = ctx.saved_tensors
            dz = dy * (y > 0).to(dy.dtype)
        # always run: the all-gather is a collective every rank takes part in
        return ctx.red.all_gather(ctx.site + "_bwd", dz.contiguous()), None, None, None


def row_reduce_scatter(red, site: str, x: torch.Tensor, relu: bool = False) -> torch.Tensor:
    """relu?(Σ over the ranks of the fp32 [N, F] partial x), this rank's rows only, with autograd (collective)."""
    _require_cuda(x)
    return _RowReduceScatterFn.apply(x, red, site, relu)


class _GcnAggregateFn(torch.autograd.Function):
    """Y = relu?(Â·S + b) in ONE launch: the aggregation (GCN/GCN.py:43), the bias add
    (GCN.py:44-45) and the ReLU that follows every hidden layer (GCN.py:12,19) fused into the
    row flush of the SpMM.  Backward: dZ = dY ⊙ [Y > 0];  dS = Âᵀ·dZ;  db = Σ_rows dZ."""

    @staticmethod
    def forward(ctx, S, bias, g: CSRGraph, relu: bool):
        Y = spmm_raw(g, S, bias=bias, relu=relu)
        ctx.g, ctx.relu, ctx.has_bias = g, relu, bias is not None
        if relu:
            ctx.save_for_backward(Y)
        return Y

    @staticmethod
    def backward(ctx, dY):
        dZ = dY
        if ctx.relu:
            (Y,) = ctx.saved_tensors
            dZ = dY * (Y > 0).to(dY.dtype)
        dS = spmm_raw(ctx.g.transpose(), dZ.contiguous()) if ctx.needs_input_grad[0] else None
        db = dZ.sum(dim=0, dtype=torch.float32) if (ctx.has_bias and ctx.needs_input_grad[1]) else None  # bias is fp32
        return dS, db, None, None


def gcn_aggregate(g: CSRGraph, S: torch.Tensor, bias: Optional[torch.Tensor] = None, relu: bool = False) -> torch.Tensor:
    """relu?(Â·S + bias) with autograd into S and bias (fp32 bias; S fp32 or bf16)."""
    if bias is not None and bias.dtype != torch.float32:
        bias = bias.float()
    return _GcnAggregateFn.apply(S, bias, g, relu)


class _PartitionedGcnAggregateFn(torch.autograd.Function):
    """The rank's rows of relu?(Â·S + b) on a row-partitioned graph (partition.PartitionedGraph), the contract of
    _GcnAggregateFn: the halo exchange and the partitioned SpMM with the bias/ReLU epilogue fused into the launch
    that writes each row's last contribution.  Backward: dZ = dY ⊙ [Y > 0];  dS = (Âᵀ·dZ)[own rows] (the
    partitioned backward: every rank's dZ reaches the rows it reads);  db = Σ dZ over the OWN rows only — the sum
    over the ranks (partition.allreduce_gradients) is the full bias gradient."""

    @staticmethod
    def forward(ctx, S, bias, op, relu: bool):
        Y = op.forward(S, bias=bias, relu=relu)
        ctx.op, ctx.relu, ctx.has_bias = op, relu, bias is not None
        if relu:
            ctx.save_for_backward(Y)
        return Y

    @staticmethod
    def backward(ctx, dY):
        dZ = dY
        if ctx.relu:
            (Y,) = ctx.saved_tensors
            dZ = dY * (Y > 0).to(dY.dtype)
        dZ = dZ.contiguous()
        # always run: the backward exchange is a collective every rank takes part in
        dS = ctx.op.backward(dZ)
        db = dZ.sum(dim=0, dtype=torch.float32) if (ctx.has_bias and ctx.needs_input_grad[1]) else None  # bias is fp32
        return (dS if ctx.needs_input_grad[0] else None), db, None, None


_DTYPE_NAME = {torch.float32: "fp32", torch.bfloat16: "bf16"}


def require_partition_dtype(pg, X: torch.Tensor, what: str):
    """A partition's peer buffers are built for one feature dtype (`pg.dtype`, the `dtype=` of its constructor): a
    tensor of another dtype is refused.  The refusal depends on the dtypes only, so every rank raises together."""
    if X.dtype != pg.dtype:
        name = _DTYPE_NAME.get(pg.dtype, str(pg.dtype))
        raise _lib.GnnError(f"{what}: the partition was built for {name} features "
                            f"(dtype={pg.dtype}), got {X.dtype}")


def partitioned_gcn_aggregate(pg, S: torch.Tensor, bias: Optional[torch.Tensor] = None,
                              relu: bool = False) -> torch.Tensor:
    """relu?(Â·S + bias)[own rows] with autograd into S and bias, over a partition.PartitionedGraph `pg`; S = the
    rank's own rows, of the partition's dtype (fp32 or bf16); the bias is applied in fp32 (cast as in
    `gcn_aggregate`) and its gradient reduced in fp32.  Collective: every rank calls it, and its backward, in the same
    order."""
    _require_cuda(S, bias)
    require_partition_dtype(pg, S, "partitioned_gcn_aggregate")
    if bias is not None and bias.dtype != torch.float32:
        bias = bias.float()
    if S.dim() != 2 or S.shape[0] != pg.n_local:
        raise _lib.GnnError(f"partitioned_gcn_aggregate: S must be [{pg.n_local}, F] (this rank's rows), "
                            f"got {tuple(S.shape)}")
    return _PartitionedGcnAggregateFn.apply(S.contiguous(), bias, pg.op(S.shape[1]), relu)


class _HaloExchangeFn(torch.autograd.Function):
    """X_comb = [X_local ; halo rows] of a row-partitioned graph.  Backward: dX_local = dX_comb[:n_local] plus the
    halo rows' gradients every peer returns, added in fixed (peer, slot) order (partition.PartitionedSpmm)."""

    @staticmethod
    def forward(ctx, X, op):
        ctx.op = op
        return op.gather_halo(X)

    @staticmethod
    def backward(ctx, dX_comb):
        # always run: the gradient return is a collective every rank takes part in
        return ctx.op.return_halo_grad(dX_comb.contiguous()), None


def halo_exchange(pg, X_local: torch.Tensor) -> torch.Tensor:
    """[X_local ; halo] ([n_local + n_halo, F], the partition's dtype: fp32 or bf16) over a partition.PartitionedGraph
    `pg`: the table whose rows the combined column ids of `pg.attention()` address, as a private copy (its backward
    needs the halo rows after later exchanges may have reused the peer buffer).  Collective, with autograd: every
    rank calls it, and its backward, in the same order.  In bf16 the halo rows travel as bf16 and the returned
    gradient rows are bf16 partials that the owner adds in fp32, rounding once per row (PartitionedSpmm)."""
    _require_cuda(X_local)
    require_partition_dtype(pg, X_local, "halo_exchange")
    if X_local.dim() != 2 or X_local.shape[0] != pg.n_local:
        raise _lib.GnnError(f"halo_exchange: X_local must be [{pg.n_local}, F] (this rank's rows), "
                            f"got {tuple(X_local.shape)}")
    return _HaloExchangeFn.apply(X_local.contiguous(), pg.op(X_local.shape[1]))


# --------------------------------------------------------------------------------------
# GraphSAGE: fused gather + reduce
# --------------------------------------------------------------------------------------
def pad_table(table: torch.Tensor) -> torch.Tensor:
    """Copy a feature table once into a buffer whose rows are 16-byte aligned and return
    the [N,F] view (602 fp32 columns -> row stride 604); this is what enables the TMA path."""
    _require_cuda(table)
    N, F = table.shape
    out = _padded_empty(N, F, table.dtype, table.device)
    out.copy_(table)
    if out.stride(0) > F:
        out.as_strided((N, out.stride(0) - F), (out.stride(0), 1), F).zero_()
    return out


def gather_reduce_raw(table: torch.Tensor, idx: Optional[torch.Tensor], n_src: int, fanout: int, reduce: str = "mean",
                      out: Optional[torch.Tensor] = None, argmax: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One gnn_gather_reduce_{f32,bf16} launch (no autograd).  idx=None: identity block."""
    if reduce not in _lib.REDUCE:  # the reference's own error (GraphSAGE_Pytorch/models/Aggregator.py:26)
        raise ValueError("Unknown aggr type, expected sum, max, or mean, but got {}".format(reduce))
    _require_cuda(table, idx)
    lib = _lib.load()
    table = _rowmajor(table)
    N, F = table.shape
    if idx is not None:
        idx = idx.contiguous().view(-1)
        if idx.dtype not in (torch.int32, torch.int64):
            idx = idx.to(torch.int64)
        if idx.numel() != n_src * fanout:
            raise _lib.GnnError(f"index block has {idx.numel()} ids, expected n_src*fanout = {n_src * fanout}")
    if out is None:
        out = _padded_empty(n_src, F, table.dtype, table.device)
    bits = 64 if (idx is None or idx.dtype == torch.int64) else 32
    fn = {torch.float32: lib.gnn_gather_reduce_f32, torch.bfloat16: lib.gnn_gather_reduce_bf16}.get(table.dtype)
    if fn is None:
        raise _lib.GnnError(f"gather_reduce: unsupported dtype {table.dtype}")
    _lib.check(fn(_p(table), _ld(table), N, _p(idx), bits, n_src, fanout, F, _lib.REDUCE[reduce], _p(out), _ld(out),
                  _p(argmax), _stream_ptr()), "gnn_gather_reduce")
    return out


def _table_head(table, plain, sharded):
    """(C entry point, leading arguments) for a tensor table [N, F] or a ShardedTable: `plain` / `sharded` map the
    dtype to the entry point of that form.  A sharded call takes (descriptor, ld, F), a plain one (ptr, ld, N, F)."""
    import ctypes as C
    if isinstance(table, ShardedTable):
        fn = sharded.get(table.dtype)
        head = (C.byref(table.desc), table.ld, table.F)
    else:
        _require_cuda(table)
        table = _rowmajor(table)
        fn = plain.get(table.dtype)
        head = (_p(table), _ld(table), table.shape[0], table.shape[1])
    if fn is None:
        raise _lib.GnnError(f"gather_reduce: unsupported dtype {table.dtype}")
    return fn, head


def gather_reduce_multi_raw(table, blocks, reduce: str = "mean", outs=None):
    """Several fixed-fanout id blocks over the SAME table in ONE launch
    (gnn_gather_reduce_multi_*): `blocks` = [(idx, n_src, fanout), ...] (idx=None: identity).
    The hops of a GraphSAGE minibatch (GraphSage.py:24-27) are such a set.  No autograd.
    `table`: a tensor, or a partition.ShardedTable (gnn_gather_reduce_multi_sharded_*, the same result bit for bit)."""
    import ctypes as C
    if reduce not in _lib.REDUCE:
        raise ValueError("Unknown aggr type, expected sum, max, or mean, but got {}".format(reduce))
    _require_cuda(*[b[0] for b in blocks])
    lib = _lib.load()
    fn, head = _table_head(table, {torch.float32: lib.gnn_gather_reduce_multi_f32,
                                   torch.bfloat16: lib.gnn_gather_reduce_multi_bf16},
                           {torch.float32: lib.gnn_gather_reduce_multi_sharded_f32,
                            torch.bfloat16: lib.gnn_gather_reduce_multi_sharded_bf16})
    F = table.shape[1]
    nb = len(blocks)
    idxs, bits = [], None
    for idx, n_src, fanout in blocks:
        if idx is not None:
            idx = idx.contiguous().view(-1)
            if idx.dtype not in (torch.int32, torch.int64):
                idx = idx.to(torch.int64)
            b = 32 if idx.dtype == torch.int32 else 64
            if bits is not None and b != bits:
                idx, b = idx.to(torch.int64 if bits == 64 else torch.int32), bits
            bits = b
            if idx.numel() != n_src * fanout:
                raise _lib.GnnError(f"index block has {idx.numel()} ids, expected n_src*fanout = {n_src * fanout}")
        idxs.append(idx)
    if outs is None:
        outs = [_padded_empty(n_src, F, table.dtype, table.device) for _, n_src, _ in blocks]
    idx_arr = (C.c_void_p * nb)(*[_p(i) for i in idxs])
    nsrc_arr = (C.c_int64 * nb)(*[int(b[1]) for b in blocks])
    fan_arr = (C.c_int32 * nb)(*[int(b[2]) for b in blocks])
    out_arr = (C.c_void_p * nb)(*[_p(o) for o in outs])
    ldo_arr = (C.c_int64 * nb)(*[_ld(o) for o in outs])
    _lib.check(fn(*head, _lib.REDUCE[reduce], nb, idx_arr, bits or 64, nsrc_arr, fan_arr, out_arr, ldo_arr,
                  _stream_ptr()), "gnn_gather_reduce_multi")
    return outs


def gather_reduce_multi_split_raw(table, blocks, reduce: str, outs_hi, lo_off: int):
    """gnn_gather_reduce_multi_f32_split: like gather_reduce_multi_raw on an fp32 table, but every reduced value x
    is written as hi = fp16(x) into `outs_hi[b]` (fp16 [n_src, F] views) and lo = fp16(x - hi) `lo_off` fp16
    elements further along the row.  Raises GnnError(unsupported) off the TMA path.  `table`: a tensor or a
    partition.ShardedTable."""
    import ctypes as C
    _require_cuda(*[b[0] for b in blocks])
    lib = _lib.load()
    if table.dtype != torch.float32:
        raise _lib.GnnError("gather_reduce_multi_split: fp32 table only")
    fn, head = _table_head(table, {torch.float32: lib.gnn_gather_reduce_multi_f32_split},
                           {torch.float32: lib.gnn_gather_reduce_multi_sharded_f32_split})
    nb = len(blocks)
    idxs, bits = [], None
    for idx, n_src, fanout in blocks:
        idx = idx.contiguous().view(-1)
        if idx.dtype not in (torch.int32, torch.int64):
            idx = idx.to(torch.int64)
        b = 32 if idx.dtype == torch.int32 else 64
        if bits is not None and b != bits:
            idx, b = idx.to(torch.int64 if bits == 64 else torch.int32), bits
        bits = b
        if idx.numel() != n_src * fanout:
            raise _lib.GnnError(f"index block has {idx.numel()} ids, expected n_src*fanout = {n_src * fanout}")
        idxs.append(idx)
    for o in outs_hi:
        if o.dtype != torch.float16 or o.stride(1) != 1:
            raise _lib.GnnError("gather_reduce_multi_split: outputs must be fp16 views with unit column stride")
    idx_arr = (C.c_void_p * nb)(*[_p(i) for i in idxs])
    nsrc_arr = (C.c_int64 * nb)(*[int(b[1]) for b in blocks])
    fan_arr = (C.c_int32 * nb)(*[int(b[2]) for b in blocks])
    out_arr = (C.c_void_p * nb)(*[_p(o) for o in outs_hi])
    ldo_arr = (C.c_int64 * nb)(*[_ld(o) for o in outs_hi])
    lo_arr = (C.c_int64 * nb)(*[int(lo_off)] * nb)
    _lib.check(fn(*head, _lib.REDUCE[reduce], nb, idx_arr, bits or 64, nsrc_arr, fan_arr, out_arr, ldo_arr, lo_arr,
                  _stream_ptr()), "gnn_gather_reduce_multi_f32_split")


def sample_neighbors(g: CSRGraph, src: torch.Tensor, k: int, seed: int, out_dtype=torch.int32,
                     seed_offset: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """k sampled neighbour ids per source (gnn_sample_neighbors), flat and src-major like
    GraphSAGE_Pytorch/sample_utils.py:4-17: without replacement when deg >= k, else with."""
    _require_cuda(src)
    lib = _lib.load()
    src = src.contiguous().view(-1)
    if src.dtype not in (torch.int32, torch.int64):
        src = src.to(torch.int64)
    if out is None:
        out = torch.empty(src.numel() * k, dtype=out_dtype, device=src.device)
    assert seed_offset is None or (seed_offset.dtype == torch.int64 and seed_offset.is_cuda)
    _lib.check(lib.gnn_sample_neighbors(_p(g.rowptr), _p(g.col), _p(src), 32 if src.dtype == torch.int32 else 64,
                                        src.numel(), int(k), int(seed) & 0xFFFFFFFFFFFFFFFF, _p(seed_offset), _p(out),
                                        32 if out.dtype == torch.int32 else 64, _stream_ptr()), "gnn_sample_neighbors")
    return out


def multihop_sampling(g: CSRGraph, src_nodes: torch.Tensor, sample_nums, seed: int, out_dtype=torch.int32,
                      seed_offset: Optional[torch.Tensor] = None):
    """GraphSAGE_Pytorch/sample_utils.py:20-35 on the device: [src, hop-1 ids, hop-2 ids, ...]."""
    result = [src_nodes.to(out_dtype) if src_nodes.dtype != out_dtype else src_nodes]
    for hop, k in enumerate(sample_nums):
        result.append(sample_neighbors(g, result[hop], k, seed + 0x9E3779B9 * (hop + 1), out_dtype, seed_offset))
    return result


def node_union(ids_a: torch.Tensor, ids_b: torch.Tensor):
    """gnn_node_union: (out_ids, count_dev, map_a, map_b).  out_ids [n_a + n_b] holds the ascending unique ids of
    ids_a ∪ {ids_b >= 0} followed by -1 padding; map_a / map_b (int64) give each input's position in it, -1 for a
    negative id; count_dev is a device int64 [1].  ids_a and ids_b share one dtype, int32 or int64."""
    _require_cuda(ids_a, ids_b)
    lib = _lib.load()
    ids_a, ids_b = ids_a.contiguous().view(-1), ids_b.contiguous().view(-1)
    if ids_a.dtype != ids_b.dtype or ids_a.dtype not in (torch.int32, torch.int64):
        raise _lib.GnnError(f"node_union: ids must share int32 or int64, got {ids_a.dtype} and {ids_b.dtype}")
    import ctypes as C
    n_a, n_b = ids_a.numel(), ids_b.numel()
    ws_bytes = C.c_size_t(0)
    _lib.check(lib.gnn_node_union_workspace_size(n_a, n_b, C.byref(ws_bytes)), "gnn_node_union_workspace_size")
    dev = ids_a.device
    ws = torch.empty(max(ws_bytes.value, 1), dtype=torch.uint8, device=dev)
    out_ids = torch.empty(n_a + n_b, dtype=ids_a.dtype, device=dev)
    count = torch.empty(1, dtype=torch.int64, device=dev)
    map_a = torch.empty(n_a, dtype=torch.int64, device=dev)
    map_b = torch.empty(n_b, dtype=torch.int64, device=dev)
    _lib.check(lib.gnn_node_union(_p(ids_a), n_a, _p(ids_b), n_b, 32 if ids_a.dtype == torch.int32 else 64,
                                  _p(out_ids), _p(count), _p(map_a), _p(map_b), _p(ws), ws_bytes.value, _stream_ptr()),
               "gnn_node_union")
    return out_ids, count, map_a, map_b


class DedupBatch:
    """One minibatch of the de-duplicating GraphSAGE (GraphSAGE/data_utils.py:82-162), built on the device by
    `dedup_layer_nodes`.  With L layers and S_{L-1} the batch, S_i = S_{i+1} ∪ samples(S_{i+1}):
      nodes[l]      int64 [n_l]      S_l; the batch keeps its order, every other set is ascending global id;
      counts[l]     int              n_l = |S_l| (host ints);
      center_map    int64 [L-1, n_0] row i: the position in S_i of each node of S_{i+1}, then -1;
      neigh_map     int64 [L-1, n_0, k] row r of map i: the positions in S_i of the k draws of node r of S_{i+1},
                                     in draw order; rows past n_{i+1} are -1 (the reference's layout: `forward` takes it);
      neighbors[l]  int64 [n_l, k]   the global ids drawn for S_l; neighbors[0] are the outermost neighbours, which
                                     the layer gathers straight from the feature table (`outer_neighbors`)."""

    def __init__(self, nodes, counts, center_map, neigh_map, neighbors):
        self.nodes, self.counts, self.center_map, self.neigh_map, self.neighbors = (nodes, counts, center_map,
                                                                                    neigh_map, neighbors)

    @property
    def outer_neighbors(self) -> torch.Tensor:
        return self.neighbors[0]


def dedup_layer_nodes(g: CSRGraph, batch_ids, num_layers: int, k: int, seed: int) -> DedupBatch:
    """GraphSAGE/data_utils.py:82-117 (`get_layer_adj_nodes`) and the id half of its collate_fn (:154-162) on the
    device.  For l = L-2 … 0: draw k neighbours of every node of S_{l+1} (`sample_neighbors`, seed mixed per layer
    as `multihop_sampling` does) and unite S_{l+1} with them (`node_union`); then draw k neighbours of S_0 once more,
    not de-duplicated, for the outermost gather.  Sets are ascending global id instead of the reference's CPython
    set order (only which row sits where differs; the maps carry it).

    Every set stays padded to its bound n_{l+1}·(k+1) with -1 ids until the end, so the layers need no host sizes;
    ONE device-to-host read of the L-1 union counts per batch then gives the shapes: that is the one
    synchronisation.  A batch given on the device costs one more, for the range check of its ids.
    A graph with a row without edges is refused (GnnError): the reference's `random.sample` fails there."""
    if num_layers < 1 or k < 1:
        raise ValueError(f"num_layers and k must be positive (got {num_layers}, {k})")
    if g.has_empty_rows():
        raise _lib.GnnError("dedup_layer_nodes: the graph has a row without edges; the reference's random.sample "
                            "cannot draw from it")
    dev = g.device
    batch = torch.as_tensor(batch_ids).view(-1)
    if batch.numel() == 0:
        raise ValueError("dedup_layer_nodes: empty batch")
    lo, hi = torch.stack([batch.min(), batch.max()]).tolist()
    if lo < 0 or hi >= g.n_rows:
        raise IndexError(f"dedup_layer_nodes: batch ids must lie in [0, {g.n_rows}), got [{lo}, {hi}]")
    batch = batch.to(device=dev, dtype=torch.int64)
    L = num_layers

    def layer_seed(l):
        return seed + 0x9E3779B9 * (L - l)  # hop L-1-l of multihop_sampling

    padded, draws, maps, count_devs = [batch], [], [], []
    for l in range(L - 2, -1, -1):
        d = sample_neighbors(g, padded[0], k, layer_seed(l + 1), torch.int64)
        out_ids, count, map_a, map_b = node_union(padded[0], d)
        padded.insert(0, out_ids)
        draws.insert(0, d)
        maps.insert(0, (map_a, map_b))
        count_devs.insert(0, count)
    counts = (torch.cat(count_devs).tolist() if count_devs else []) + [batch.numel()]
    nodes = [p[:n] for p, n in zip(padded, counts)]
    n0 = counts[0]
    center_map = torch.full((L - 1, n0), -1, dtype=torch.int64, device=dev)
    neigh_map = torch.full((L - 1, n0, k), -1, dtype=torch.int64, device=dev)
    neighbors = [None] * L
    for i, (map_a, map_b) in enumerate(maps):
        n = counts[i + 1]
        center_map[i, :n] = map_a[:n]
        neigh_map[i, :n] = map_b.view(-1, k)[:n]
        neighbors[i + 1] = draws[i].view(-1, k)[:n]
    neighbors[0] = sample_neighbors(g, nodes[0], k, layer_seed(0), torch.int64).view(n0, k)
    return DedupBatch(nodes, counts, center_map, neigh_map, neighbors)


class _GatherReduceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, table, idx, n_src, fanout, reduce):
        ctx.meta = (n_src, fanout, reduce, tuple(table.shape))
        argmax = None
        out = _padded_empty(n_src, table.shape[1], table.dtype, table.device)
        if reduce == "max" and ctx.needs_input_grad[0]:
            argmax = torch.empty((n_src, out.stride(0)), dtype=torch.int32, device=table.device)[:, :table.shape[1]]
        gather_reduce_raw(table, idx, n_src, fanout, reduce, out=out, argmax=argmax)
        ctx.save_for_backward(idx if idx is not None else torch.empty(0), argmax if argmax is not None else torch.empty(0))
        ctx.has_idx = idx is not None
        return out

    @staticmethod
    def backward(ctx, d_out):
        n_src, fanout, reduce, (N, F) = ctx.meta
        idx, argmax = ctx.saved_tensors
        if not ctx.needs_input_grad[0]:
            return None, None, None, None, None
        # bf16-feature variant: the ordered scatter accumulates in fp32 (the fp32 kernels) and the table gradient is
        # returned in the table's dtype — one rounding at the end, like every other bf16 path here
        out_dtype = d_out.dtype
        if d_out.dtype == torch.bfloat16:
            d_out = d_out.float()
        elif d_out.dtype != torch.float32:
            raise _lib.GnnError(f"gather_reduce backward: unsupported dtype {d_out.dtype}")
        lib = _lib.load()
        d_out = d_out.contiguous()
        scale = 1.0 / fanout if reduce == "mean" else 1.0
        if not ctx.has_idx:
            # pre-gathered [n_src*fanout, F] input (Aggregator.py:18): dense broadcast / argmax routing
            d_table = torch.empty((N, F), dtype=torch.float32, device=d_out.device)
            am = argmax[:, :F].contiguous() if reduce == "max" else None
            _lib.check(lib.gnn_gather_reduce_bwd_dense_f32(_p(d_out), _ld(d_out), _p(am), n_src, fanout, F, scale,
                                                           _p(d_table), _stream_ptr()), "gnn_gather_reduce_bwd_dense_f32")
            if N > n_src * fanout:
                d_table[n_src * fanout:].zero_()
            return d_table.to(out_dtype), None, None, None, None
        if reduce == "max":
            raise _lib.GnnError("max backward into a gathered table is not implemented (the reference's max path "
                                "raises TypeError, GraphSAGE_Pytorch/models/Aggregator.py:24,29)")
        rowptr_t, pos_t = index_block_transpose(idx, N)
        d_table = torch.empty((N, F), dtype=torch.float32, device=d_out.device)
        _lib.check(lib.gnn_gather_reduce_bwd_f32(_p(rowptr_t), _p(pos_t), N, fanout, scale, _p(d_out), _ld(d_out),
                                                 _p(d_table), _ld(d_table), F, _stream_ptr()),
                   "gnn_gather_reduce_bwd_f32")
        return d_table.to(out_dtype), None, None, None, None


def gather_reduce(table: torch.Tensor, idx: Optional[torch.Tensor], n_src: int, fanout: int,
                  reduce: str = "mean") -> torch.Tensor:
    """out[i] = reduce_k table[idx[i*fanout+k]] with autograd into `table`."""
    if reduce not in _lib.REDUCE:
        raise ValueError("Unknown aggr type, expected sum, max, or mean, but got {}".format(reduce))
    return _GatherReduceFn.apply(table, idx, n_src, fanout, reduce)


class _TypedGatherFn(torch.autograd.Function):
    """out[b,t,:] = reduce_k table[idx[b,t,k], t, :] (gnn_gather_reduce_typed_f32).  Backward into the
    table walks the transposed index block of the flat (node*T + t) ids: ordered, no atomics."""

    @staticmethod
    def forward(ctx, table, idx, reduce):
        N, T, U = table.shape
        B, T2, K = idx.shape
        out = torch.empty((B, T, U), dtype=torch.float32, device=table.device)
        lib = _lib.load()
        _lib.check(lib.gnn_gather_reduce_typed_f32(_p(table), table.stride(1), N, T, _p(idx),
                                                   32 if idx.dtype == torch.int32 else 64, B, K, U,
                                                   _lib.REDUCE[reduce], _p(out), U, _stream_ptr()),
                   "gnn_gather_reduce_typed_f32")
        ctx.save_for_backward(idx)
        ctx.meta = (N, T, U, K, reduce)
        return out

    @staticmethod
    def backward(ctx, d_out):
        (idx,) = ctx.saved_tensors
        N, T, U, K, reduce = ctx.meta
        if not ctx.needs_input_grad[0]:
            return None, None, None
        lib = _lib.load()
        flat = (idx.to(torch.int64) * T + torch.arange(T, device=idx.device).view(1, T, 1)).reshape(-1)
        rowptr_t, pos_t = index_block_transpose(flat, N * T)
        d_out = d_out.contiguous().view(-1, U)
        d_table = torch.empty((N, T, U), dtype=torch.float32, device=d_out.device)
        _lib.check(lib.gnn_gather_reduce_bwd_f32(_p(rowptr_t), _p(pos_t), N * T, K, 1.0 / K if reduce == "mean" else 1.0,
                                                 _p(d_out), U, _p(d_table), U, U, _stream_ptr()),
                   "gnn_gather_reduce_bwd_f32")
        return d_table, None, None


def typed_gather_reduce(table: torch.Tensor, idx: torch.Tensor, reduce: str = "sum") -> torch.Tensor:
    """GATNE's per-edge-type neighbour aggregation: `table` [N, T, U] fp32 (node_type_embeddings),
    `idx` [B, T, K] int32/int64 neighbour ids per edge type -> [B, T, U]; reduce 'sum' | 'mean'
    (GATNE_Pytorch/models/GATNE.py:57-77, GATNE/models/GATNE.py:50-58)."""
    if reduce not in ("sum", "mean"):
        raise ValueError("please choice else aggregator!")  # the reference's message (GATNE.py:77)
    _require_cuda(table, idx)
    if table.dim() != 3 or idx.dim() != 3 or idx.shape[1] != table.shape[1]:
        raise _lib.GnnError(f"typed_gather_reduce: table {tuple(table.shape)} / idx {tuple(idx.shape)} do not agree")
    if table.dtype != torch.float32:
        raise _lib.GnnError("typed_gather_reduce: fp32 table only")
    if idx.dtype not in (torch.int32, torch.int64):
        idx = idx.to(torch.int64)
    return _TypedGatherFn.apply(table.contiguous(), idx.contiguous(), reduce)


# --------------------------------------------------------------------------------------
# GAT / HAN: fused multi-head attention aggregation
# --------------------------------------------------------------------------------------
def gat_scores_raw(Wh: torch.Tensor, a_src: torch.Tensor, a_dst: torch.Tensor, H: int, Fp: int):
    _require_cuda(Wh, a_src, a_dst)
    lib = _lib.load()
    Wh = _rowmajor(Wh)
    n = Wh.shape[0]
    s = torch.empty((n, H), dtype=torch.float32, device=Wh.device)
    t = torch.empty((n, H), dtype=torch.float32, device=Wh.device)
    _lib.check(lib.gnn_gat_scores_f32(_p(Wh), _ld(Wh), _p(a_src.contiguous()), _p(a_dst.contiguous()), n, H, Fp, _p(s),
                                      _p(t), _stream_ptr()), "gnn_gat_scores_f32")
    return s, t


def _gat_groups(H: int, Fp: int):
    """Column groups one kernel call can take (H_g*Fp_g <= 256, H_g <= 32): whole heads when a head fits,
    else column tiles of ONE head.  Yields (h0, h1, f0, f1): heads [h0,h1), columns [f0,f1) of each."""
    if Fp <= 256:
        per = max(1, min(32, 256 // Fp))
        for h0 in range(0, H, per):
            yield h0, min(H, h0 + per), 0, Fp
    else:
        for h in range(H):
            for f0 in range(0, Fp, 256):
                yield h, h + 1, f0, min(Fp, f0 + 256)


class AttentionDropout:
    """Seeded post-softmax attention dropout (GAT/models/layers.py:31) for the fused kernels: probability `p`, a host
    seed and a device int64 tensor mixed into it (so a captured CUDA graph draws a fresh mask per replay).  The
    kernels recompute the keep factor of every (edge, head) from the stream — no [nnz, H] mask is materialised.
    edge_slot_base: local edge slot e draws the factor of slot e + edge_slot_base (a row block of a larger CSR passes
    its first global slot and draws the whole graph's mask for its edges).
    slot_shift (device int64 [M], batched-rectangular graphs only): graph m's slots are moved by slot_shift[m] as
    well (partition.PartitionedMetapaths.attention)."""

    def __init__(self, p: float, seed: int, seed_dev: Optional[torch.Tensor] = None, edge_slot_base: int = 0,
                 slot_shift: Optional[torch.Tensor] = None):
        self.p, self.seed, self.seed_dev = float(p), int(seed) & 0xFFFFFFFFFFFFFFFF, seed_dev
        self.edge_slot_base = int(edge_slot_base)
        self.slot_shift = slot_shift
        assert seed_dev is None or (seed_dev.dtype == torch.int64 and seed_dev.is_cuda and seed_dev.numel() == 1)
        assert slot_shift is None or (slot_shift.dtype == torch.int64 and slot_shift.is_cuda)

    def c_struct(self):
        import ctypes as C
        d = _lib.GatDropout()
        d.struct_size = C.sizeof(_lib.GatDropout)
        d.p, d.seed, d.seed_dev = self.p, self.seed, _p(self.seed_dev)
        d.edge_slot_base = self.edge_slot_base
        return d

    def with_slot_base(self, edge_slot_base: int) -> "AttentionDropout":
        """The same stream for a row block whose first edge is global slot `edge_slot_base`.  The kernels take a slot
        base only with the whole seed on the host, so the device half is read back here (one synchronisation)."""
        seed = self.seed
        if self.seed_dev is not None:
            seed ^= (int(self.seed_dev.item()) * 0xD6E8FEB86659FD93) & 0xFFFFFFFFFFFFFFFF
        return AttentionDropout(self.p, seed, None, edge_slot_base)


_drop_counters = {}


def next_attention_dropout(p: float, device) -> AttentionDropout:
    """A fresh dropout stream: host seed from torch's CPU generator (so torch.manual_seed controls it), device half =
    a private copy of a per-device counter that is incremented IN PLACE on the stream — under CUDA-graph capture
    the increment and the copy are replayed, hence a new mask per replay, and the forward and the backward of one
    call see the same value."""
    dev = torch.device(device)
    ctr = _drop_counters.get(dev)
    if ctr is None:
        ctr = _drop_counters[dev] = torch.zeros(1, dtype=torch.int64, device=dev)
    ctr.add_(1)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())  # CPU generator: no device synchronisation
    return AttentionDropout(p, seed, ctr.clone())


def attention_keep_mask_from_seed(g: CSRGraph, H: int, drop: AttentionDropout) -> torch.Tensor:
    """The [nnz, H] keep factors the kernels derive from `drop` (torch restatement of keep_factor in csrc/gat.cu:
    splitmix64 of seed + (edge slot * H + head + 1)), for tests and for inspecting a mask."""
    M64 = (1 << 64) - 1

    def s64(x):  # python int (mod 2^64) -> signed int64 value
        x &= M64
        return x - (1 << 64) if x >= (1 << 63) else x

    def lsr(z, k):  # logical shift right on int64 tensors
        return (z >> k) & ((1 << (64 - k)) - 1)

    seed = drop.seed
    if drop.seed_dev is not None:
        seed ^= (int(drop.seed_dev.item()) * 0xD6E8FEB86659FD93) & M64
    idx = torch.arange(g.nnz * H, dtype=torch.int64, device=g.device) + (drop.edge_slot_base * H + 1)
    z = idx * s64(0x9E3779B97F4A7C15) + s64(seed)
    z = (z ^ lsr(z, 30)) * s64(0xBF58476D1CE4E5B9)
    z = (z ^ lsr(z, 27)) * s64(0x94D049BB133111EB)
    z = z ^ lsr(z, 31)
    keep_prob = torch.tensor(1.0, dtype=torch.float32) - torch.tensor(drop.p, dtype=torch.float32)  # 1.f - p
    thresh = int((keep_prob * 16777216.0).item())  # float32 arithmetic, as in the kernel
    scale = float((1.0 / keep_prob).item())
    keep = (lsr(z, 40) < thresh).to(torch.float32) * scale
    return keep.view(g.nnz, H)


def gat_fwd_raw(g: CSRGraph, Wh, s, t, H, Fp, alpha, mode=_lib.GAT_SOFTMAX, elu=0, keep=None, save_stats=False,
                out=None, dropout: Optional[AttentionDropout] = None, out_act: Optional[torch.Tensor] = None,
                batch: int = 1):
    """Forward of the fused attention aggregation (no autograd).  Wh fp32 or bf16 ([n, H*Fp]); s, t fp32 [n,H];
    `out` has Wh's dtype.  Layers wider than one call's 256 columns (e.g. 8 heads x 64) are run as head groups /
    column tiles of a head; the softmax statistics are per head, so a tiled head recomputes them per tile.
    Training form (`out_act` given): `out` receives the PRE-activation aggregate and `out_act` the activated one
    (elu applied `elu` times) in the same launch.  `dropout`: seeded attention dropout (or `keep`: explicit mask).
    batch = M > 1: `g` is the block diagonal of M graphs over the same N nodes (CSRGraph.block_diagonal), Wh / out are
    [N, M*H*Fp] (graph m's columns at m*H*Fp), s / t are [M*N, H] (batched-row major) — HAN's metapaths in one launch.
    Rectangular `g` (n_cols > n_rows, a row block whose columns address [own rows ; halo rows]): Wh and t have n_cols
    rows, s and out n_rows; fp32 or bf16, H*Fp <= 256 and no row without edges.  With batch = M > 1 as well, `g` is
    the block diagonal of M such blocks over one combined table (partition.PartitionedMetapaths.attention): Wh is
    [n_cols / M, M*H*Fp], t [n_cols, H], s [n_rows, H], out [n_rows / M, M*H*Fp]; `dropout.slot_shift` moves each
    graph's dropout slots."""
    _require_cuda(Wh, s, t, keep)
    lib = _lib.load()
    Wh = _rowmajor(Wh)
    if Wh.dtype not in (torch.float32, torch.bfloat16):
        raise _lib.GnnError(f"gat: unsupported dtype {Wh.dtype} (fp32 and bf16 only)")
    s = s.float().contiguous()
    t = t.float().contiguous()
    n, nc = g.n_rows, g.n_cols
    M = int(batch)
    nodes = n // M
    if (M < 1 or n % M or nc < n or Wh.shape != (nc // M, M * H * Fp) or s.shape != (n, H)
            or t.shape != (nc, H)):
        raise _lib.GnnError(f"gat: Wh {tuple(Wh.shape)} / s {tuple(s.shape)} / t {tuple(t.shape)} do not match graph "
                            f"rows={n}, cols={nc}, batch={M}, H*Fp={H * Fp}")
    if nc != n and H * Fp > 256:
        raise _lib.GnnError("gat: a rectangular graph (table rows != rows) takes H*Fp <= 256")
    if M > 1 and H * Fp > 256:
        raise _lib.GnnError("gat: batched graphs need H*Fp <= 256 per graph")
    if out is None:
        out = torch.empty((nodes, M * H * Fp), dtype=Wh.dtype, device=Wh.device)
    elif out.shape != (nodes, M * H * Fp) or out.dtype != Wh.dtype or out.stride(1) != 1 or not out.is_cuda:
        raise _lib.GnnError("gat: `out` must be a CUDA [nodes, batch*H*Fp] view of Wh's dtype with unit column stride")
    if out_act is not None and (out_act.shape != out.shape or out_act.dtype != out.dtype or
                                out_act.stride() != out.stride()):
        raise _lib.GnnError("gat: `out_act` must match `out` in shape, dtype and strides")
    row_max = torch.empty((n, H), dtype=torch.float32, device=Wh.device) if save_stats else None
    row_sum = torch.empty((n, H), dtype=torch.float32, device=Wh.device) if save_stats else None
    if nc != n and g.has_empty_rows():
        raise _lib.GnnError("gat: rows without edges take the mean of ALL table rows (GAT/models/layers.py:28-30), "
                            "which a rectangular graph does not define")
    col_mean = Wh.float().mean(dim=0).contiguous() if g.has_empty_rows() else None
    bn = nodes if M > 1 else 0
    lr, thr = g.gat_long_rows()
    f32 = Wh.dtype == torch.float32
    import ctypes as C
    if _batched_rect(g, M, dropout):
        # batched and rectangular: one group, the training entry (it writes the activated form to out_act)
        pre_buf, act_buf = (out, out_act) if (out_act is not None or elu == 0) else (torch.empty_like(out), out)
        dstruct = dropout.c_struct() if (dropout is not None and dropout.p > 0.0) else None
        bstruct = _batch_struct(M, nodes, nc // M, dropout)
        fb = lib.gnn_gat_fused_fwd_batch_f32 if f32 else lib.gnn_gat_fused_fwd_batch_bf16
        _lib.check(fb(
            _p(g.rowptr), _p(g.col), _p(Wh), _ld(Wh), _p(s), _p(t), g.nnz, H, Fp, float(alpha), mode,
            elu if act_buf is not None else 0, _p(keep), C.byref(dstruct) if dstruct is not None else None,
            _p(pre_buf), _p(act_buf), _ld(out), _p(row_max), _p(row_sum), _p(lr), lr.numel(), thr, C.byref(bstruct),
            _stream_ptr()), "gnn_gat_fused_fwd_batch")
        return out, row_max, row_sum
    train = out_act is not None or (dropout is not None and dropout.p > 0.0)
    pre_buf, act_buf = out, out_act
    if train and out_act is None and elu > 0:
        # seeded dropout without autograd (train mode under no_grad): the training entry point writes the
        # activated aggregate to its second output; the pre-activation goes to a scratch buffer
        pre_buf, act_buf = torch.empty_like(out), out
    if train:
        fn = lib.gnn_gat_fused_fwd_train_f32 if f32 else lib.gnn_gat_fused_fwd_train_bf16
    else:
        fn = lib.gnn_gat_fused_fwd_f32 if f32 else lib.gnn_gat_fused_fwd_bf16
    groups = list(_gat_groups(H, Fp))
    if dropout is not None and dropout.p > 0.0 and len(groups) > 1:
        # a head group restarts the head index at 0: materialise the stream once so every group sees its own heads
        keep, dropout = attention_keep_mask_from_seed(g, H, dropout), None
    dstruct = dropout.c_struct() if (dropout is not None and dropout.p > 0.0) else None
    for h0, h1, f0, f1 in groups:
        whole = len(groups) == 1
        Hg, Fg = h1 - h0, f1 - f0
        c0 = h0 * Fp + f0
        sg = s if whole else s[:, h0:h1].contiguous()
        tg = t if whole else t[:, h0:h1].contiguous()
        kg = keep if (whole or keep is None) else keep[:, h0:h1].contiguous()
        cm = col_mean if (whole or col_mean is None) else col_mean[c0:c0 + Hg * Fg].contiguous()
        rm = row_max if (whole or row_max is None) else torch.empty((n, Hg), dtype=torch.float32, device=Wh.device)
        rs = row_sum if (whole or row_sum is None) else torch.empty((n, Hg), dtype=torch.float32, device=Wh.device)
        esz = Wh.element_size()
        if train:
            _lib.check(fn(_p(g.rowptr), _p(g.col), Wh.data_ptr() + c0 * esz, _ld(Wh), _p(sg), _p(tg), n, g.nnz, Hg, Fg,
                          float(alpha), mode, elu if act_buf is not None else 0, _p(cm), _p(kg),
                          C.byref(dstruct) if dstruct is not None else None, pre_buf.data_ptr() + c0 * esz,
                          None if act_buf is None else act_buf.data_ptr() + c0 * esz, _ld(out), _p(rm), _p(rs),
                          _p(lr), lr.numel(), thr, bn, _stream_ptr()), "gnn_gat_fused_fwd_train")
        else:
            _lib.check(fn(_p(g.rowptr), _p(g.col), Wh.data_ptr() + c0 * esz, _ld(Wh), _p(sg), _p(tg), n, g.nnz, Hg, Fg,
                          float(alpha), mode, elu, _p(cm), _p(kg), out.data_ptr() + c0 * esz, _ld(out), _p(rm), _p(rs),
                          _p(lr), lr.numel(), thr, bn, _stream_ptr()), "gnn_gat_fused_fwd")
        if not whole and save_stats:
            row_max[:, h0:h1] = rm
            row_sum[:, h0:h1] = rs
    return out, row_max, row_sum


def _batched_rect(g: CSRGraph, M: int, dropout: Optional[AttentionDropout]) -> bool:
    """The batched-rectangular entries serve a batched graph whose table rows differ from its rows, or whose seeded
    dropout carries per-graph slot shifts (a rank's block without halo rows is square)."""
    shifted = dropout is not None and dropout.p > 0.0 and dropout.slot_shift is not None
    return M > 1 and (g.n_cols != g.n_rows or shifted)


def _batch_struct(M: int, rows: int, cols: int, dropout: Optional[AttentionDropout]):
    b = _lib.GatBatch()
    import ctypes as C
    b.struct_size = C.sizeof(_lib.GatBatch)
    b.n_graphs, b.rows_per_graph, b.cols_per_graph = int(M), int(rows), int(cols)
    shift = None if (dropout is None or dropout.p <= 0.0) else dropout.slot_shift
    if shift is not None and (shift.numel() != M or not shift.is_contiguous()):
        raise _lib.GnnError(f"gat: slot_shift must be a contiguous [{M}] int64 tensor")
    b.slot_shift = _p(shift)
    return b


class _GatFn(torch.autograd.Function):
    """Fused attention aggregation with autograd.  Returns the ACTIVATED aggregate (elu applied `elu` times in the
    kernel epilogue); the pre-activation aggregate is saved for the backward, which applies the ELU derivative
    chain inside its first kernel — neither the activations nor their gradients are separate launches."""

    @staticmethod
    def forward(ctx, Wh, s, t, g: CSRGraph, H, Fp, alpha, mode, keep, elu, dropout, batch=1):
        Wh = _rowmajor(Wh)
        if dropout is not None and dropout.p > 0.0 and len(list(_gat_groups(H, Fp))) > 1:
            keep, dropout = attention_keep_mask_from_seed(g, H, dropout), None
        out_pre = torch.empty((g.n_rows // batch, batch * H * Fp), dtype=Wh.dtype, device=Wh.device)
        out_act = torch.empty_like(out_pre) if elu > 0 else None
        _, row_max, row_sum = gat_fwd_raw(g, Wh, s, t, H, Fp, alpha, mode, elu=elu, keep=keep, save_stats=True,
                                          out=out_pre, dropout=dropout, out_act=out_act, batch=batch)
        ctx.g, ctx.cfg = g, (H, Fp, float(alpha), mode, int(elu))
        ctx.batch = int(batch)
        ctx.dropout = dropout
        ctx.st_dtypes = (s.dtype, t.dtype)
        ctx.save_for_backward(Wh, s.float().contiguous(), t.float().contiguous(), row_max, row_sum, out_pre,
                              keep if keep is not None else torch.empty(0))
        return out_act if elu > 0 else out_pre

    @staticmethod
    def backward(ctx, d_out):
        import ctypes as C
        Wh, s, t, row_max, row_sum, out, keep = ctx.saved_tensors
        g = ctx.g
        H, Fp, alpha, mode, elu = ctx.cfg
        lib = _lib.load()
        keep = keep if keep.numel() > 0 else None
        drop = ctx.dropout if (ctx.dropout is not None and ctx.dropout.p > 0.0) else None
        dstruct = drop.c_struct() if drop is not None else None
        n, nc = g.n_rows, g.n_cols
        d_out = d_out.to(Wh.dtype)
        if d_out.stride(1) != 1 or d_out.stride(0) != out.stride(0):
            d_out = d_out.contiguous()  # out is contiguous [n, H*Fp]: one leading dimension for both
        gt = g.transpose()
        dev = Wh.device
        M = ctx.batch
        bn = n // M if M > 1 else 0
        d_Wh = torch.empty_like(Wh)
        d_s = torch.empty((n, H), dtype=torch.float32, device=dev)
        d_t = torch.empty((nc, H), dtype=torch.float32, device=dev)
        d_pre = torch.empty_like(out) if elu > 0 else None
        (lr, thr), (lrt, _) = g.gat_long_rows(), gt.gat_long_rows()
        fn = lib.gnn_gat_fused_bwd_f32 if Wh.dtype == torch.float32 else lib.gnn_gat_fused_bwd_bf16
        groups = list(_gat_groups(H, Fp))
        esz = Wh.element_size()
        need_perm = keep is not None or drop is not None
        f32 = Wh.dtype == torch.float32
        if _batched_rect(g, M, drop):  # batched and rectangular (one group, no empty row: checked by the forward)
            row_scratch = torch.empty((n, 4, H), dtype=torch.float32, device=dev)
            bstruct = _batch_struct(M, n // M, nc // M, drop)
            fb = lib.gnn_gat_fused_bwd_batch_f32 if f32 else lib.gnn_gat_fused_bwd_batch_bf16
            _lib.check(fb(
                _p(g.rowptr), _p(g.col), _p(gt.rowptr), _p(gt.col), _p(g.perm_t) if need_perm else None, _p(Wh), _ld(Wh),
                _p(s), _p(t), _p(row_max), _p(row_sum), _p(out), _p(d_out), _ld(out), H, Fp, alpha, mode,
                _p(keep), _p(d_Wh), _ld(d_Wh), _p(d_s), _p(d_t), _p(row_scratch), g.nnz, _p(lr), lr.numel(), _p(lrt),
                lrt.numel(), thr, elu, _p(d_pre), C.byref(dstruct) if dstruct is not None else None, C.byref(bstruct),
                _stream_ptr()), "gnn_gat_fused_bwd_batch")
            groups = []
        elif nc != n:  # rectangular (one group, checked by the forward): table rows get d_Wh / d_t
            row_scratch = torch.empty((n, 4, H), dtype=torch.float32, device=dev)
            fx = lib.gnn_gat_fused_bwd_ex_f32 if f32 else lib.gnn_gat_fused_bwd_ex_bf16
            _lib.check(fx(
                _p(g.rowptr), _p(g.col), _p(gt.rowptr), _p(gt.col), _p(g.perm_t) if need_perm else None, _p(Wh), _ld(Wh),
                _p(s), _p(t), _p(row_max), _p(row_sum), _p(out), _p(d_out), _ld(out), n, nc, H, Fp, alpha, mode,
                _p(keep), _p(d_Wh), _ld(d_Wh), _p(d_s), _p(d_t), _p(row_scratch), g.nnz, _p(lr), lr.numel(), _p(lrt),
                lrt.numel(), thr, elu, _p(d_pre), C.byref(dstruct) if dstruct is not None else None, _stream_ptr()),
                "gnn_gat_fused_bwd_ex")
            groups = []
        for gi, (h0, h1, f0, f1) in enumerate(groups):
            whole = len(groups) == 1
            Hg, Fg = h1 - h0, f1 - f0
            c0 = h0 * Fp + f0
            sg = s if whole else s[:, h0:h1].contiguous()
            tg = t if whole else t[:, h0:h1].contiguous()
            kg = keep if (whole or keep is None) else keep[:, h0:h1].contiguous()
            rm = row_max if whole else row_max[:, h0:h1].contiguous()
            rs = row_sum if whole else row_sum[:, h0:h1].contiguous()
            ds = d_s if whole else torch.empty((n, Hg), dtype=torch.float32, device=dev)
            dt = d_t if whole else torch.empty((n, Hg), dtype=torch.float32, device=dev)
            row_scratch = torch.empty((n, 4, Hg), dtype=torch.float32, device=dev)
            _lib.check(fn(_p(g.rowptr), _p(g.col), _p(gt.rowptr), _p(gt.col), _p(g.perm_t) if need_perm else None,
                          Wh.data_ptr() + c0 * esz, _ld(Wh), _p(sg), _p(tg), _p(rm), _p(rs), out.data_ptr() + c0 * esz,
                          d_out.data_ptr() + c0 * esz, _ld(out), n, Hg, Fg, alpha, mode, _p(kg),
                          d_Wh.data_ptr() + c0 * esz, _ld(d_Wh), _p(ds), _p(dt), _p(row_scratch), g.nnz, _p(lr),
                          lr.numel(), _p(lrt), lrt.numel(), thr, elu,
                          None if d_pre is None else d_pre.data_ptr() + c0 * esz,
                          C.byref(dstruct) if dstruct is not None else None, bn, _stream_ptr()), "gnn_gat_fused_bwd")
            if not whole:
                # dz is linear in (head dot, row dot): the tiles of one head add up (first tile assigns)
                if f0 == 0:
                    d_s[:, h0:h1] = ds
                    d_t[:, h0:h1] = dt
                else:
                    d_s[:, h0:h1] += ds
                    d_t[:, h0:h1] += dt
        if g.has_empty_rows():
            # rows without edges output the mean of all Wh rows (GAT/models/layers.py:28-30).  Sync-free
            # (no boolean-mask indexing): this runs inside CapturedTrainStep's CUDA-graph capture
            dpre = (d_pre if elu > 0 else d_out).float()
            if M > 1:  # per graph: its empty rows spread their gradient over its own column block
                mask = g.empty_row_mask().view(M, n // M, 1)
                blocks = dpre.view(n // M, M, H * Fp).permute(1, 0, 2)
                d_Wh += ((blocks * mask).sum(dim=1) / (n // M)).reshape(1, M * H * Fp).to(d_Wh.dtype)
            else:
                d_Wh += ((dpre * g.empty_row_mask().unsqueeze(1)).sum(dim=0, keepdim=True) / n).to(d_Wh.dtype)
        return (d_Wh, d_s.to(ctx.st_dtypes[0]), d_t.to(ctx.st_dtypes[1]), None, None, None, None, None, None, None, None,
                None)


def gat_aggregate(g: CSRGraph, Wh: torch.Tensor, s: torch.Tensor, t: torch.Tensor, H: int, Fp: int, alpha: float,
                  mode: int = _lib.GAT_SOFTMAX, elu: int = 0, keep: Optional[torch.Tensor] = None,
                  out: Optional[torch.Tensor] = None, dropout: Optional[AttentionDropout] = None,
                  batch: int = 1) -> torch.Tensor:
    """Fused edge-score + LeakyReLU + edge-softmax + weighted aggregation over all H heads, with the ELU(s) that
    follow (elu = 0 | 1 | 2) in the kernel epilogue — with and without autograd.
    Wh may be fp32 or bf16 (the bf16-feature variant: bf16 rows, fp32 scores / softmax / accumulation).
    keep: explicit [nnz, H] post-softmax dropout factors (parity tests); dropout: seeded stream (training)."""
    need_grad = torch.is_grad_enabled() and (Wh.requires_grad or s.requires_grad or t.requires_grad)
    if not need_grad:
        # `out` (optional): a strided [n, H*Fp] view the kernel writes in place, e.g. one metapath's
        # slice of HAN's [N, M, H*Fp] semantic stack
        return gat_fwd_raw(g, Wh, s, t, H, Fp, alpha, mode, elu=elu, keep=keep, out=out, dropout=dropout, batch=batch)[0]
    if out is not None:
        raise _lib.GnnError("gat_aggregate: `out` is only supported without autograd")
    return _GatFn.apply(Wh, s, t, g, H, Fp, alpha, mode, keep, elu, dropout, batch)


def attention_keep_mask(g: CSRGraph, H: int, p: float, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """Per-edge, per-head post-softmax dropout factors (0 or 1/(1-p)), GAT/models/layers.py:31."""
    keep = torch.empty((g.nnz, H), dtype=torch.float32, device=g.device)
    keep.bernoulli_(1.0 - p, generator=generator).div_(1.0 - p)
    return keep


# ---- HAN semantic attention (HAN/models/SemanticAttention.py:15-20) --------------------------------------------
_semantic_ws = {}


def _semantic_workspace(K: int, device) -> torch.Tensor:
    """Zeroed once per (device, stream, K): the kernels' ticket counter must start at zero and every call leaves it
    zero; one workspace per stream keeps concurrent streams apart, and it persists for CUDA-graph replays."""
    key = (torch.device(device), torch.cuda.current_stream(device).cuda_stream, int(K))
    ws = _semantic_ws.get(key)
    if ws is None:
        nbytes = int(_lib.load().gnn_semantic_workspace_size(int(K)))
        if nbytes < 0:
            raise _lib.GnnError(f"semantic_attention: hidden width {K} unsupported")
        ws = _semantic_ws[key] = torch.zeros(nbytes, dtype=torch.uint8, device=device)
    return ws


SEMANTIC_MAX_M, SEMANTIC_MAX_K = 32, 256


def _rank_ordered_sum(x: torch.Tensor, world: int, group) -> torch.Tensor:
    """Σ over the ranks of x, added in rank order starting from rank 0's tensor (one all_gather): the same bits on
    every rank whatever the backend's reduction algorithm, and x itself at world 1."""
    if world == 1:
        return x
    import torch.distributed as dist
    parts = [torch.empty_like(x) for _ in range(world)]
    dist.all_gather(parts, x.contiguous(), group=group)
    acc = parts[0]
    for p in parts[1:]:
        acc = acc + p
    return acc


class _SemanticFn(torch.autograd.Function):
    """out = sum_m softmax_M(mean_N(q . tanh(z W1^T + b)))_m z[:, m, :]: one GEMM + two launches forward, two
    launches + two GEMMs backward (csrc/semantic.cu).
    dist = (n_total, world, group): z is a rank's rows of a row-partitioned node set, and the node sums behind mean_N
    (forward) and dβ (backward) are split at the rank boundary: partial over the own rows, a rank-ordered sum of the
    [M] partials, then finalize with the global node count.  Collective in both directions."""

    @staticmethod
    def forward(ctx, z, W1, b1, q, dist):
        lib = _lib.load()
        N, M, D = z.shape
        K = W1.shape[0]
        dev = z.device
        z = z.contiguous()
        W1c, qv = W1.contiguous(), q.reshape(-1).contiguous()
        b1c = None if b1 is None else b1.contiguous()
        P = torch.mm(z.view(N * M, D), W1c.t())                      # [N*M, K], the library GEMM
        ws = _semantic_workspace(K, dev)
        scores = torch.empty(M, dtype=torch.float32, device=dev)
        beta = torch.empty(M, dtype=torch.float32, device=dev)
        st = _stream_ptr()
        if dist is None:
            _lib.check(lib.gnn_semantic_scores_f32(_p(P), P.stride(0), _p(b1c), _p(qv), N, M, K, _p(scores), _p(beta),
                                                   _p(ws), ws.numel(), st), "gnn_semantic_scores_f32")
        else:
            n_total, world, group = dist
            sums = torch.empty(M, dtype=torch.float32, device=dev)
            _lib.check(lib.gnn_semantic_scores_partial_f32(_p(P), P.stride(0), _p(b1c), _p(qv), N, M, K, _p(sums),
                                                           _p(ws), ws.numel(), st), "gnn_semantic_scores_partial_f32")
            sums = _rank_ordered_sum(sums, world, group)
            _lib.check(lib.gnn_semantic_scores_finalize_f32(_p(sums), n_total, M, _p(scores), _p(beta), st),
                       "gnn_semantic_scores_finalize_f32")
        out = torch.empty((N, D), dtype=torch.float32, device=dev)
        _lib.check(lib.gnn_semantic_combine_f32(_p(beta), _p(z), N, M, D, _p(out), st), "gnn_semantic_combine_f32")
        ctx.save_for_backward(z, W1c, b1c if b1c is not None else z.new_empty(0), qv, P, beta)
        ctx.has_bias, ctx.q_shape, ctx.dist = b1 is not None, tuple(q.shape), dist
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        z, W1, b1, qv, P, beta = ctx.saved_tensors
        N, M, D = z.shape
        K = W1.shape[0]
        dev = z.device
        d_out = d_out.contiguous()
        ws = _semantic_workspace(K, dev)
        dz = torch.empty_like(z)
        dsn = torch.empty(M, dtype=torch.float32, device=dev)
        st = _stream_ptr()
        if ctx.dist is None:
            _lib.check(lib.gnn_semantic_combine_bwd_f32(_p(d_out), _p(z), _p(beta), N, M, D, _p(dz), _p(dsn), _p(ws),
                                                        ws.numel(), st), "gnn_semantic_combine_bwd_f32")
        else:
            n_total, world, group = ctx.dist
            dbeta = torch.empty(M, dtype=torch.float32, device=dev)
            _lib.check(lib.gnn_semantic_combine_bwd_partial_f32(_p(d_out), _p(z), _p(beta), N, M, D, _p(dz), _p(dbeta),
                                                                _p(ws), ws.numel(), st),
                       "gnn_semantic_combine_bwd_partial_f32")
            dbeta = _rank_ordered_sum(dbeta, world, group)
            _lib.check(lib.gnn_semantic_combine_bwd_finalize_f32(_p(dbeta), _p(beta), n_total, M, _p(dsn), st),
                       "gnn_semantic_combine_bwd_finalize_f32")
        # dq / db are column sums over the rows (on a partition the rank's share, which partition.allreduce_gradients
        # adds up): the kernel writes them, and a rank without rows contributes zeros
        alloc = torch.empty if N > 0 else torch.zeros
        dq = alloc(K, dtype=torch.float32, device=dev)
        db = alloc(K, dtype=torch.float32, device=dev) if ctx.has_bias else None
        dP = torch.empty_like(P)
        if N > 0:
            _lib.check(lib.gnn_semantic_scores_bwd_f32(_p(P), P.stride(0), _p(b1) if ctx.has_bias else None, _p(qv),
                                                       _p(dsn), N, M, K, _p(dP), dP.stride(0), _p(dq), _p(db), _p(ws),
                                                       ws.numel(), st), "gnn_semantic_scores_bwd_f32")
        z2 = z.view(N * M, D)
        dW1 = torch.mm(dP.t(), z2) if ctx.needs_input_grad[1] else None                 # [K, D]
        if ctx.needs_input_grad[0]:
            dz = torch.addmm(dz.view(N * M, D), dP, W1).view(N, M, D)                    # direct term + dP·W1
        else:
            dz = None
        return dz, dW1, db, dq.view(ctx.q_shape), None


def _semantic(z: torch.Tensor, W1: torch.Tensor, b1: Optional[torch.Tensor], q: torch.Tensor, dist=None):
    """The shape checks of both entries: dist None needs rows in z, a partition a positive global node count."""
    _require_cuda(z, W1, q)
    if z.dtype != torch.float32 or z.dim() != 3 or z.shape[1] > SEMANTIC_MAX_M or W1.shape[0] > SEMANTIC_MAX_K or \
            W1.shape[1] != z.shape[2] or q.numel() != W1.shape[0] or (z.shape[0] if dist is None else dist[0]) <= 0:
        raise _lib.GnnError(f"semantic_attention: unsupported shapes z {tuple(z.shape)} W1 {tuple(W1.shape)} "
                            f"q {tuple(q.shape)}" + ("" if dist is None else f" n_total {dist[0]}"))
    return _SemanticFn.apply(z, W1, b1, q, dist)


def semantic_attention(z: torch.Tensor, W1: torch.Tensor, b1: Optional[torch.Tensor], q: torch.Tensor) -> torch.Tensor:
    """HAN semantic attention over z [N, M, D] with project = Linear(D,K; W1,b1) -> tanh -> Linear(K,1; q, no bias)
    (SemanticAttention.py:8-20): returns [N, D].  fp32, M <= 32, K <= 256."""
    return _semantic(z, W1, b1, q)


def semantic_attention_partitioned(z: torch.Tensor, W1: torch.Tensor, b1: Optional[torch.Tensor], q: torch.Tensor,
                                   n_total: int, world: int, group=None) -> torch.Tensor:
    """`semantic_attention` over this rank's rows z [n_local, M, D] of a row-partitioned node set of n_total nodes:
    β is the one of all n_total nodes, identical on every rank (rank-ordered sums of the per-rank node sums).
    Collective, forward and backward; at world 1 it computes the same bits as `semantic_attention`."""
    return _semantic(z, W1, b1, q, (int(n_total), int(world), group))
