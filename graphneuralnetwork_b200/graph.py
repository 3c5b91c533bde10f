"""Device-resident graph structures built through the C ABI.

`CSRGraph` is what the kernels walk: int64 rowptr, int32 col, optional fp32 val, plus a
lazily built transpose (for the deterministic backward) and the long-row plan.  The
builders accept exactly the adjacency forms the reference layers are handed
(SURVEY.md §8b "Accepted adj forms"):
  - torch sparse COO fp32          (GCN/data_utils.py:63-70)
  - dense [N,N] fp32 / fp64 mask   (GAT/data_utils.py:85, HAN/utils/data_utils.py:85-89)
  - fixed-fanout index blocks      (GraphSAGE_Pytorch/sample_utils.py:20-35)
torch is used here for device memory and streams only.
"""
from __future__ import annotations

import weakref
from typing import Optional

import torch

from . import _lib


def _stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require_cuda(*tensors) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise _lib.GnnError("tensor is not on a CUDA device: the message-passing path has no CPU fallback")


class CSRGraph:
    """CSR adjacency on the device (rows = destination nodes)."""

    def __init__(self, rowptr: torch.Tensor, col: torch.Tensor, val: Optional[torch.Tensor], n_rows: int, n_cols: int):
        _require_cuda(rowptr, col, val)
        assert rowptr.dtype == torch.int64 and col.dtype == torch.int32
        assert val is None or val.dtype == torch.float32
        self.rowptr, self.col, self.val = rowptr.contiguous(), col.contiguous(), None if val is None else val.contiguous()
        self.n_rows, self.n_cols = int(n_rows), int(n_cols)
        self.nnz = int(col.numel())
        self._t: Optional["CSRGraph"] = None
        self._perm_t: Optional[torch.Tensor] = None
        self._long_rows: Optional[torch.Tensor] = None
        self._plan = None
        self._zero_rows: Optional[bool] = None

    @property
    def device(self):
        return self.rowptr.device

    def with_values(self, val: Optional[torch.Tensor]) -> "CSRGraph":
        """Same pattern, other edge values (learned / per-step weights): shares rowptr, col and every
        host-side plan that depends on the pattern only, so nothing is re-planned or re-synchronised."""
        self.long_row_plan()  # plans are cached on the pattern owner before the copy shares them
        self.rows_per_team()
        g = CSRGraph.__new__(CSRGraph)
        g.__dict__.update(self.__dict__)
        g.val = None if val is None else val.contiguous()
        g._t = None  # the transpose carries values: rebuilt (from the cached permutation) on demand
        return g

    def edge_rows(self) -> torch.Tensor:
        """int32 row id of every CSR slot (rowptr expanded once; cached with the pattern)."""
        if getattr(self, "_edge_rows", None) is None:
            counts = self.rowptr[1:] - self.rowptr[:-1]
            self._edge_rows = torch.repeat_interleave(torch.arange(self.n_rows, device=self.device, dtype=torch.int32),
                                                      counts, output_size=self.nnz)
        return self._edge_rows

    # -- plans ---------------------------------------------------------------------
    def transpose(self) -> "CSRGraph":
        """CSR of the transpose, stable in source order (gnn_csr_transpose); cached."""
        if self._t is None:
            lib = _lib.load()
            dev = self.device
            rowptr_t = torch.empty(self.n_cols + 1, dtype=torch.int64, device=dev)
            col_t = torch.empty(self.nnz, dtype=torch.int32, device=dev)
            val_t = None if self.val is None else torch.empty(self.nnz, dtype=torch.float32, device=dev)
            perm_t = torch.empty(self.nnz, dtype=torch.int64, device=dev)
            ws_bytes = lib.gnn_csr_transpose_workspace_size(self.nnz, self.n_rows, self.n_cols)
            ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
            _lib.check(lib.gnn_csr_transpose(_p(self.rowptr), _p(self.col), _p(self.val), self.n_rows, self.n_cols,
                                             self.nnz, _p(rowptr_t), _p(col_t), _p(val_t), _p(perm_t), _p(ws),
                                             ws_bytes, _stream_ptr()), "gnn_csr_transpose")
            self._t = CSRGraph(rowptr_t, col_t, val_t, self.n_cols, self.n_rows)
            self._t._t = self
            self._perm_t = perm_t
        return self._t

    @property
    def perm_t(self) -> torch.Tensor:
        self.transpose()
        return self._perm_t

    def long_rows(self) -> torch.Tensor:
        """Rows whose nnz exceeds the spmm.long_row knob (host-side plan, cached)."""
        if self._long_rows is None:
            thr = _lib.get_tuning("spmm.long_row")
            deg = self.rowptr[1:] - self.rowptr[:-1]
            self._long_rows = torch.nonzero(deg > thr).flatten().contiguous()
        return self._long_rows

    def long_row_plan(self):
        """Host-side plan for power-law graphs, computed once per graph: rows longer than the
        `spmm.long_row` knob are cut into chunks of `spmm.chunk` edges.  Returns
        (long_rows int64[n_long], threshold, chunk_off int64[n_long+1], n_chunks, chunk_edges,
        workspace uint8 tensor) or None when no row is long."""
        if self._plan is None:
            thr = _lib.get_tuning("spmm.long_row")
            chunk = _lib.get_tuning("spmm.chunk")
            lr = self.long_rows()
            if lr.numel() == 0:
                self._plan = False
            else:
                deg = self.rowptr[lr + 1] - self.rowptr[lr]
                counts = (deg + chunk - 1) // chunk
                chunk_off = torch.zeros(lr.numel() + 1, dtype=torch.int64, device=self.device)
                torch.cumsum(counts, 0, out=chunk_off[1:])
                n_chunks = int(chunk_off[-1].item())
                ws_bytes = _lib.load().gnn_spmm_csr_workspace_size(n_chunks, 2)  # bf16 tiles are the wider
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
                self._plan = (lr, thr, chunk_off, n_chunks, chunk, ws)
        return self._plan or None

    def rows_per_team(self) -> int:
        """Host-side plan for the row-block streaming SpMM: how many consecutive rows one
        sub-warp team streams, chosen so that a team holds about `spmm.team_edges` edges of
        the rows that are not long (1..32; the kernel clamps to its team width)."""
        if getattr(self, "_rpt", None) is None:
            lr = self.long_rows()
            short_nnz = self.nnz
            if lr.numel() > 0:
                short_nnz -= int((self.rowptr[lr + 1] - self.rowptr[lr]).sum().item())
            mean = short_nnz / max(self.n_rows - lr.numel(), 1)
            target = _lib.get_tuning("spmm.team_edges")
            self._rpt = int(min(32, max(1, -(-target // max(int(mean + 0.5), 1)))))
        return self._rpt

    def gat_long_rows(self):
        """(long_rows int64, threshold): rows the attention kernels hand to a whole CTA (host-side plan,
        cached)."""
        if getattr(self, "_gat_long", None) is None:
            thr = _lib.get_tuning("gat.long_row")
            deg = self.rowptr[1:] - self.rowptr[:-1]
            self._gat_long = (torch.nonzero(deg > thr).flatten().contiguous(), thr)
        return self._gat_long

    def has_empty_rows(self) -> bool:
        if self._zero_rows is None:
            deg = self.rowptr[1:] - self.rowptr[:-1]
            self._zero_rows = bool((deg == 0).any().item()) if self.n_rows > 0 else False
        return self._zero_rows

    def empty_row_mask(self) -> torch.Tensor:
        """fp32 [n_rows] indicator of rows without edges (cached with the pattern)."""
        if getattr(self, "_empty_mask", None) is None:
            self._empty_mask = ((self.rowptr[1:] - self.rowptr[:-1]) == 0).to(torch.float32)
        return self._empty_mask

    _block_cache = {}

    @staticmethod
    def block_diagonal(graphs) -> "CSRGraph":
        """Block diagonal of M square pattern graphs over the same N nodes (HAN's metapath adjacencies): row
        m*N + i is row i of graph m, its column ids offset by m*N.  One fused attention launch walks all M graphs
        (`gat_aggregate(..., batch=M)`).  Cached per tuple of graphs."""
        graphs = list(graphs)
        key = tuple(id(g) for g in graphs)
        hit = CSRGraph._block_cache.get(key)
        if hit is not None and all(a is b for a, b in zip(hit[0], graphs)):
            return hit[1]
        n = graphs[0].n_rows
        assert all(g.n_rows == n and g.n_cols == n and g.val is None for g in graphs), "square pattern graphs over the same nodes"
        parts, cols, off = [], [], 0
        for m, g in enumerate(graphs):
            parts.append(g.rowptr[:-1] + off)
            cols.append(g.col + m * n)
            off += g.nnz
        parts.append(torch.tensor([off], dtype=torch.int64, device=graphs[0].device))
        big = CSRGraph(torch.cat(parts), torch.cat(cols).to(torch.int32), None, len(graphs) * n, len(graphs) * n)
        if len(CSRGraph._block_cache) >= 8:
            CSRGraph._block_cache.pop(next(iter(CSRGraph._block_cache)))
        CSRGraph._block_cache[key] = (graphs, big)
        return big

    # -- builders --------------------------------------------------------------------
    @staticmethod
    def from_coo(row: torch.Tensor, col: torch.Tensor, val: Optional[torch.Tensor], n_rows: int, n_cols: int,
                 return_perm: bool = False, validate: bool = True):
        """COO -> CSR, stable in row (gnn_build_csr_from_coo).  return_perm: also return the int64
        input position of every CSR slot (values given in COO order are `val[perm]` in CSR order).
        validate: ids outside [0, n_rows) x [0, n_cols) raise IndexError here (one host read per graph build;
        the reference's torch.spmm / indexing raises likewise) instead of becoming out-of-bounds accesses."""
        _require_cuda(row, col, val)
        lib = _lib.load()
        dev = row.device
        row = row.to(torch.int64).contiguous()
        col = col.to(torch.int64).contiguous()
        if validate and row.numel():
            bad = ((row < 0) | (row >= n_rows) | (col < 0) | (col >= n_cols)).any()
            if bool(bad.item()):
                raise IndexError(f"COO index out of range for a [{n_rows}, {n_cols}] adjacency")
        if val is not None:
            val = val.to(torch.float32).contiguous()
        nnz = int(row.numel())
        rowptr = torch.empty(n_rows + 1, dtype=torch.int64, device=dev)
        col32 = torch.empty(nnz, dtype=torch.int32, device=dev)
        val32 = None if val is None else torch.empty(nnz, dtype=torch.float32, device=dev)
        ws_bytes = lib.gnn_build_csr_from_coo_workspace_size(nnz, n_rows)
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
        perm = torch.empty(nnz, dtype=torch.int64, device=dev) if return_perm else None
        _lib.check(lib.gnn_build_csr_from_coo(_p(row), _p(col), _p(val), nnz, n_rows, n_cols, _p(rowptr), _p(col32),
                                              _p(val32), _p(perm), _p(ws), ws_bytes, _stream_ptr()),
                   "gnn_build_csr_from_coo")
        g = CSRGraph(rowptr, col32, val32, n_rows, n_cols)
        return (g, perm) if return_perm else g

    @staticmethod
    def from_torch_sparse(adj: torch.Tensor) -> "CSRGraph":
        """torch sparse COO (the tensor GCN/data_utils.py:70 builds) -> CSR.

        The reference tensor is flagged uncoalesced but holds no duplicates and is
        row-major sorted (SURVEY.md §8 a1); `_indices()/_values()` are used as they are,
        duplicates — if a caller passes any — simply stay separate edges, which sums to the
        same product as torch.spmm."""
        assert adj.layout == torch.sparse_coo
        idx = adj._indices()
        return CSRGraph.from_coo(idx[0], idx[1], adj._values(), adj.shape[0], adj.shape[1])

    @staticmethod
    def from_dense_mask(adj: torch.Tensor) -> "CSRGraph":
        """Dense [N,M] adjacency used only as `adj > 0` -> CSR pattern in adj.nonzero() order."""
        _require_cuda(adj)
        if adj.dtype not in (torch.float32, torch.float64):
            adj = adj.to(torch.float32)
        if adj.stride(-1) != 1:
            adj = adj.contiguous()
        lib = _lib.load()
        dev = adj.device
        n_rows, n_cols = adj.shape
        ld = adj.stride(0) if n_rows > 1 else max(n_cols, 1)
        dt = 0 if adj.dtype == torch.float32 else 1
        rowptr = torch.empty(n_rows + 1, dtype=torch.int64, device=dev)
        ws_bytes = lib.gnn_dense_mask_count_workspace_size(n_rows)
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
        _lib.check(lib.gnn_dense_mask_count(_p(adj), dt, n_rows, n_cols, ld, _p(rowptr), _p(ws), ws_bytes,
                                            _stream_ptr()), "gnn_dense_mask_count")
        nnz = int(rowptr[-1].item())  # one host read: nnz sizes the col array
        col = torch.empty(nnz, dtype=torch.int32, device=dev)
        if nnz == 0:  # an adjacency without a single positive entry: nothing to fill
            return CSRGraph(rowptr, col, None, n_rows, n_cols)
        _lib.check(lib.gnn_dense_mask_fill(_p(adj), dt, n_rows, n_cols, ld, _p(rowptr), _p(col), _stream_ptr()),
                   "gnn_dense_mask_fill")
        return CSRGraph(rowptr, col, None, n_rows, n_cols)

    @staticmethod
    def pattern_product(A: "CSRGraph", B: "CSRGraph", row_range=None, self_loops: bool = False,
                        max_nnz: Optional[int] = None, validate: bool = True,
                        path_rows: Optional[torch.Tensor] = None) -> "CSRGraph":
        """Pattern of A·B (values ignored), rows `row_range` = (lo, hi) of A (default all): row r lists, once each and
        ascending, every column j some x connects, (lo + r, x) in A and (x, j) in B (gnn_pattern_product_count/fill).
        That is scipy's ((A_bool @ B_bool) > 0) after sort_indices(), the metapath adjacency HAN builds densely
        (HAN/utils/data_utils.py:85-89).  self_loops adds column i to row i (square products only).  Column ids
        stay global.  One host read of nnz sizes `col`; nnz above `max_nnz` raises GnnError before it is allocated.
        validate: ids outside A's or B's columns raise IndexError (one host read).  path_rows: an int64[3] CUDA
        tensor that receives the rows each kernel path took (warp sort, CTA sort, bitmap)."""
        lo, hi = _pattern_args(A, B, row_range, validate)
        rowptr = _pattern_count(A, B, lo, hi, self_loops, path_rows)
        nnz = int(rowptr[-1].item())  # one host read: nnz sizes the col array
        if max_nnz is not None and nnz > max_nnz:
            raise _lib.GnnError(f"pattern_product: the product has {nnz} entries, more than max_nnz = {max_nnz} "
                                f"({4 * nnz + 8 * (hi - lo + 1)} bytes for col and rowptr)")
        return CSRGraph(rowptr, _pattern_fill(A, B, lo, hi, self_loops, rowptr, nnz), None, hi - lo, B.n_cols)

    @staticmethod
    def metapath(R: "CSRGraph", self_loops: bool = False, max_nnz: Optional[int] = None) -> "CSRGraph":
        """Metapath adjacency pattern(R·Rᵀ) of a relation R [N x X] (paper x author, paper x subject), with
        `self_loops` the (R·Rᵀ + I) > 0 HAN trains on.  Rᵀ is R's cached `transpose()`."""
        _require_ids_in_range(R)  # before the transpose, which sorts by column id
        return CSRGraph.pattern_product(R, R.transpose(), self_loops=self_loops, max_nnz=max_nnz, validate=False)


def _pattern_args(A: CSRGraph, B: CSRGraph, row_range, validate: bool):
    """(lo, hi) of a pattern product after the checks the kernels rely on."""
    _require_cuda(A.rowptr, B.rowptr)
    if A.n_cols != B.n_rows:
        raise ValueError(f"pattern_product: A is [{A.n_rows}, {A.n_cols}] but B has {B.n_rows} rows")
    lo, hi = (0, A.n_rows) if row_range is None else (int(row_range[0]), int(row_range[1]))
    if not 0 <= lo <= hi <= A.n_rows:
        raise IndexError(f"pattern_product: row range [{lo}, {hi}) outside the {A.n_rows} rows of A")
    if validate:
        _require_ids_in_range(A, B)
    return lo, hi


def _require_ids_in_range(*graphs: CSRGraph) -> None:
    """IndexError if a column id of one of `graphs` lies outside its columns (one host read)."""
    bad = [((g.col < 0) | (g.col >= g.n_cols)).any() for g in graphs if g.nnz]
    if bad and bool(torch.stack(bad).any().item()):
        raise IndexError("pattern_product: a column id outside [0, n_cols) of " +
                         " or ".join(f"a [{g.n_rows}, {g.n_cols}] graph" for g in graphs))


def _col_or_dummy(g: CSRGraph) -> torch.Tensor:
    # an empty tensor has no address; the kernels read no column of a graph without entries
    return g.col if g.nnz else torch.zeros(1, dtype=torch.int32, device=g.device)


def _pattern_ws(n_rows: int, dev) -> torch.Tensor:
    return torch.empty(_lib.load().gnn_pattern_product_count_workspace_size(n_rows), dtype=torch.uint8, device=dev)


def _pattern_count(A: CSRGraph, B: CSRGraph, lo: int, hi: int, self_loops: bool,
                   path_rows: Optional[torch.Tensor] = None) -> torch.Tensor:
    """int64 rowptr [hi - lo + 1] of rows [lo, hi) of pattern(A·B) (no host read)."""
    _require_cuda(path_rows)
    if path_rows is not None and (path_rows.dtype != torch.int64 or path_rows.numel() != 3
                                  or not path_rows.is_contiguous()):
        raise ValueError("pattern_product: path_rows must be a contiguous int64 tensor of 3 elements")
    lib = _lib.load()
    rowptr = torch.empty(hi - lo + 1, dtype=torch.int64, device=A.device)
    ws = _pattern_ws(hi - lo, A.device)
    _lib.check(lib.gnn_pattern_product_count(_p(A.rowptr), _p(_col_or_dummy(A)), A.n_rows, A.n_cols, _p(B.rowptr),
                                             _p(_col_or_dummy(B)), B.n_cols, lo, hi, int(self_loops), _p(rowptr),
                                             _p(path_rows), _p(ws), ws.numel(), _stream_ptr()),
               "gnn_pattern_product_count")
    return rowptr


def _pattern_fill(A: CSRGraph, B: CSRGraph, lo: int, hi: int, self_loops: bool, rowptr: torch.Tensor,
                  nnz: int) -> torch.Tensor:
    """int32 col [nnz] of rows [lo, hi) of pattern(A·B), given their rowptr (global column ids)."""
    col = torch.empty(nnz, dtype=torch.int32, device=A.device)
    if nnz == 0:
        return col
    lib = _lib.load()
    ws = _pattern_ws(hi - lo, A.device)
    _lib.check(lib.gnn_pattern_product_fill(_p(A.rowptr), _p(_col_or_dummy(A)), A.n_rows, A.n_cols, _p(B.rowptr),
                                            _p(_col_or_dummy(B)), B.n_cols, lo, hi, int(self_loops),
                                            _p(rowptr.contiguous()), _p(col), _p(ws), ws.numel(), _stream_ptr()),
               "gnn_pattern_product_fill")
    return col


class _AdjCache:
    """Converts an adjacency tensor to CSR once and reuses it while the tensor is unchanged
    (keyed by data_ptr, _version, shape — SURVEY.md §8b)."""

    def __init__(self, max_entries: int = 16):
        self._entries = {}
        self._max = max_entries

    def get(self, adj) -> CSRGraph:
        if isinstance(adj, CSRGraph):
            return adj
        if adj.layout == torch.sparse_coo:
            key = ("coo", adj._values().data_ptr(), adj._indices().data_ptr(), adj._values()._version, tuple(adj.shape))
        else:
            key = ("dense", adj.data_ptr(), adj._version, tuple(adj.shape), adj.dtype)
        hit = self._entries.get(key)
        if hit is not None:
            ref, g = hit
            if ref() is adj:
                return g
        g = CSRGraph.from_torch_sparse(adj) if adj.layout == torch.sparse_coo else CSRGraph.from_dense_mask(adj)
        if len(self._entries) >= self._max:
            self._entries.pop(next(iter(self._entries)))
        try:
            ref = weakref.ref(adj)
        except TypeError:  # pragma: no cover
            ref = lambda: adj
        self._entries[key] = (ref, g)
        return g


adj_cache = _AdjCache()


_idx_transpose_cache = {}


def index_block_transpose(idx: torch.Tensor, n_table_rows: int, cache: bool = True):
    """Fixed-fanout index block -> (rowptr_t, pos_t) for the ordered gather backward.
    cache: the transpose (a CUB sort) is kept per index TENSOR (identity + version guarded by a weakref, as the
    adjacency caches are), so a block that is walked backward again — the same minibatch in the next epoch, or
    several layers sharing one map — is sorted once."""
    _require_cuda(idx)
    lib = _lib.load()
    key = (idx.data_ptr(), idx._version, tuple(idx.shape), idx.dtype, int(n_table_rows))
    if cache:
        hit = _idx_transpose_cache.get(key)
        if hit is not None and hit[0]() is idx:
            return hit[1]
    src = idx
    idx = idx.contiguous().view(-1)
    bits = 32 if idx.dtype == torch.int32 else 64
    if idx.dtype not in (torch.int32, torch.int64):
        idx = idx.to(torch.int64)
    n = int(idx.numel())
    dev = idx.device
    rowptr_t = torch.empty(n_table_rows + 1, dtype=torch.int64, device=dev)
    pos_t = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    ws_bytes = lib.gnn_index_block_transpose_workspace_size(n, n_table_rows)
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
    _lib.check(lib.gnn_index_block_transpose(_p(idx), bits, n, n_table_rows, _p(rowptr_t), _p(pos_t), _p(ws), ws_bytes,
                                             _stream_ptr()), "gnn_index_block_transpose")
    if cache:
        for k in [k for k, (r, _) in _idx_transpose_cache.items() if r() is None]:
            _idx_transpose_cache.pop(k)
        if len(_idx_transpose_cache) >= 32:
            _idx_transpose_cache.pop(next(iter(_idx_transpose_cache)))
        try:
            _idx_transpose_cache[key] = (weakref.ref(src), (rowptr_t, pos_t))
        except TypeError:  # pragma: no cover
            pass
    return rowptr_t, pos_t
