"""Drop-in GTN pieces (class / function names, ctor signatures, parameter names and forward signatures of
/root/reference GTN/models/{GTN,GTLayer,GTConv}.py) — SURVEY.md §8f rank 4.

On the message-passing path (re-designed):
  * `gcn_conv(X, H)` (GTN.py:49-52): the GCN over the LEARNED metapath adjacency H.  The reference normalises the
    dense H with two N x N `torch.eye` products (`norm`, GTN.py:7-19: an O(N^3) `torch.mm(deg_inv, H)`) and
    aggregates with a dense `torch.mm(H.t(), X)`.  Here the non-zero pattern of H (off-diagonal) plus the
    self-loops is turned into a CSR of H^T ON THE DEVICE (gnn_dense_mask_count / _fill), the edge values are
    gathered from H (autograd reaches H through the gather), column-normalised in O(nnz), and the aggregation
    is the CSR SpMM with gradients into the edge VALUES (`functional.spmm_values`: SpMM + edge-gradient
    SDDMM + transpose SpMM).
  * `norm(H, add)` keeps the reference's dense-in / dense-out contract for `GTN_Model.normalization`, as
    element-wise work: multiplying by a diagonal matrix is a row scaling, and adds only exact zeros, so the
    result is bit-identical to the reference's `torch.mm(deg_inv, H)`.
  * Sparse composition (DESIGN §4.10): `GTN_Model.forward` also takes a `RelationStack` where the reference passes
    the dense [N, N, K] tensor.  GTConv's soft selection is then a [nnz_U, C] value tensor on the union pattern U
    of the relations, every GTLayer product is `functional.spgemm_values` on a pattern built once per stack
    (P_1 = pattern(U·U), P_{l+1} = pattern(offdiag(P_l)·U)), `norm` is `functional.column_normalize` on the
    pattern without its diagonal, and the final `gcn_conv` runs on the cached pattern of (offdiag(H) + I)^T.
    Same parameters and state_dict as the dense path, which a dense `A` still takes unchanged.
  * Across GPUs (DESIGN §4.10): `GTN_Model.forward(ps, X_local, target_local)` takes a
    `partition.PartitionedRelationStack`, one rank's row block of every composed H_l.  The composition stays local;
    the column sums of `norm` and the degrees of the final gcn_conv are partial sums over the rank's rows that a
    rank-ordered all-reduce completes, and the gcn_conv's partial output is reduce-scattered with its ReLU fused.
"""
import torch
from torch import nn
import torch.nn.functional as F

from .. import _lib
from ..functional import column_normalize, rank_all_reduce, row_reduce_scatter, spgemm_values, spmm_values
from ..graph import CSRGraph, _require_cuda, _require_ids_in_range
from ..partition import PartitionedRelationStack


def norm(H, add=False):
    """GTN/models/GTN.py:7-19: zero the diagonal (add=True: then put ones on it), divide every COLUMN of H by its
    sum (`deg^-1`, inf -> 0).  Dense in, dense out."""
    Ht = H.t()
    n = Ht.shape[0]
    off = (torch.eye(n, device=H.device) == 0).to(torch.float32)
    Ht = Ht * off
    if add:
        Ht = Ht + torch.eye(n, device=H.device, dtype=torch.float32)
    deg = torch.sum(Ht, dim=1)
    deg_inv = deg.pow(-1)
    deg_inv = torch.where(deg_inv == float('inf'), torch.zeros_like(deg_inv), deg_inv)
    return (deg_inv.unsqueeze(1) * Ht).t()


def _pattern_of_learned_adjacency(H):
    """CSR of (offdiag(H) != 0 | I)^T built on the device, plus the flat positions of its edges in H."""
    n = H.shape[0]
    with torch.no_grad():
        mask = (H.detach().t() != 0).to(torch.float32)
        mask.fill_diagonal_(1.0)  # the +I of norm(add=True); the diagonal VALUE of H itself is dropped
        g = CSRGraph.from_dense_mask(mask.contiguous())  # rows = columns of H (H^T), ascending source ids
        rows = g.edge_rows().to(torch.int64)   # j  (row of H^T)
        cols = g.col.to(torch.int64)           # i  (column of H^T) -> entry H[i, j]
    return g, rows, cols


def gcn_conv(X, H, weight):
    """`GTN_Model.gcn_conv` (GTN.py:49-52): D^-1 (offdiag(H) + I)^T (X W) with D the column sums of
    offdiag(H) + I.  X [N, w_in], H [N, N] dense (learned, autograd flows into it), weight [w_in, w_out].
    The gradient w.r.t. H is produced on the support of H (its non-zero entries): the reference's dense autograd
    also fills the structural zeros, but in GTN a zero of the composed adjacency is a zero of every factor
    product, so no parameter receives anything from them (the model-level gradients are identical)."""
    XW = torch.mm(X, weight)
    g, rows, cols = _pattern_of_learned_adjacency(H)
    diag = rows == cols
    vals = torch.where(diag, torch.ones((), device=H.device, dtype=H.dtype), H[cols, rows])  # (offdiag(H) + I)[i, j]
    return _normalized_aggregate(g, vals.float(), XW)


def _normalized_aggregate(g, vals, XW, reduce=None):
    """The tail of `gcn_conv` on g = CSR of (offdiag(H) + I)^T with its values: divide by the column sums of
    offdiag(H) + I (the row sums of g, an ordered SpMM against ones; inf -> 0) and aggregate XW, autograd into vals.
    vals [nnz, C] gives the C channels' outputs side by side, [n_rows, C * w]; vals [nnz] is one channel, [n_rows, w].
    reduce: on a row block (partition.PartitionedRelationStack) the degrees are partial sums, and `reduce([n_rows, C])`
    returns the sums over every rank's rows; None keeps them."""
    V = vals if vals.dim() == 2 else vals.unsqueeze(1)  # not view(nnz, -1): a rank's empty block has nnz = 0
    C = V.shape[1]

    def channel(x, c):  # column c of x [rows, C]; one channel is x itself, without a copy forward or backward
        return x.view(-1) if C == 1 else x[:, c]

    def side_by_side(parts):
        return parts[0] if C == 1 else torch.cat(parts, dim=1)

    ones = torch.ones((g.n_cols, 1), dtype=torch.float32, device=vals.device)
    deg = side_by_side([spmm_values(g, channel(V, c).contiguous(), ones) for c in range(C)])
    if reduce is not None:
        deg = reduce(deg)
    deg_inv = deg.pow(-1)
    deg_inv = torch.where(deg_inv == float('inf'), torch.zeros_like(deg_inv), deg_inv)
    rows = g.edge_rows().long()
    return side_by_side([spmm_values(g, channel(V, c) * channel(deg_inv, c)[rows], XW) for c in range(C)])


def _drop_diagonal(P, lo=0):
    """(pattern of P without its diagonal, int64 slots of P it keeps).  P may be the row block [lo, lo + n_rows) of a
    square pattern: its diagonal is then (r, lo + r).  Setup only: one host read of the count."""
    keep = (P.edge_rows() + lo) != P.col if lo else P.edge_rows() != P.col
    idx = torch.nonzero(keep).flatten()
    cum = torch.zeros(P.nnz + 1, dtype=torch.int64, device=P.device)
    torch.cumsum(keep.to(torch.int64), 0, out=cum[1:])
    return CSRGraph(cum[P.rowptr], P.col[idx].contiguous(), None, P.n_rows, P.n_cols), idx


class RelationStack:
    """GTN's K edge-type adjacencies (the last one usually the identity GTN appends) as ONE union pattern U [N, N]
    with values V [nnz_U, K] (0 where relation k lacks the entry), plus the patterns every layer count needs, built
    once with the pattern-product kernels and cached:
        P_1 = pattern(U·U),  D_l = P_l without its diagonal,  P_{l+1} = pattern(D_l·U),
    and for the final gcn_conv the CSR of (D_L + I)^T.  Pass it to `GTN_Model.forward` in place of the dense
    [N, N, K] tensor.  `max_nnz` bounds every composed pattern: a larger one raises GnnError before its column array
    is allocated (`CSRGraph.pattern_product`)."""

    def __init__(self, U: CSRGraph, V: torch.Tensor, max_nnz=None):
        _require_cuda(U.rowptr, V)
        if U.n_rows != U.n_cols:
            raise ValueError(f"RelationStack: relations must be square, got [{U.n_rows}, {U.n_cols}]")
        if V.dim() != 2 or V.shape[0] != U.nnz:
            raise ValueError(f"RelationStack: V must be [nnz_U = {U.nnz}, K], got {tuple(V.shape)}")
        _require_ids_in_range(U)
        self.U, self.V = U, V.to(torch.float32).contiguous()
        self.n, self.num_edge = U.n_rows, V.shape[1]
        self.max_nnz = max_nnz
        self._P, self._D, self._keep = [], [], []
        self._gcn = {}

    @staticmethod
    def from_dense(A: torch.Tensor, max_nnz=None) -> "RelationStack":
        """From the reference's dense input A [N, N, K] (GTN/main.py builds it with the identity as the last type)."""
        _require_cuda(A)
        if A.dim() != 3 or A.shape[0] != A.shape[1]:
            raise ValueError(f"RelationStack.from_dense: A must be [N, N, K], got {tuple(A.shape)}")
        U = CSRGraph.from_dense_mask((A != 0).any(dim=2).to(torch.float32))
        rows, cols = U.edge_rows().long(), U.col.long()
        return RelationStack(U, A[rows, cols].to(torch.float32), max_nnz)

    @staticmethod
    def from_relations(graphs, max_nnz=None) -> "RelationStack":
        """From K value-carrying CSRGraphs [N, N] (val None: ones), in GTN's edge-type order.  Repeated entries of
        one relation add up.  Ids outside [0, N) raise IndexError."""
        graphs = list(graphs)
        if not graphs:
            raise ValueError("RelationStack.from_relations: no relations")
        n = graphs[0].n_rows
        for g in graphs:
            _require_cuda(g.rowptr)
            if g.n_rows != n or g.n_cols != n:
                raise ValueError(f"RelationStack.from_relations: relations must be [{n}, {n}], got "
                                 f"[{g.n_rows}, {g.n_cols}]")
        _require_ids_in_range(*graphs)
        dev = graphs[0].device
        keys = torch.cat([g.edge_rows().long() * n + g.col.long() for g in graphs])
        kind = torch.cat([torch.full((g.nnz,), k, dtype=torch.int64, device=dev) for k, g in enumerate(graphs)])
        vals = torch.cat([torch.ones(g.nnz, device=dev) if g.val is None else g.val.float() for g in graphs])
        ukeys, inv = torch.unique(keys, sorted=True, return_inverse=True)
        V = torch.zeros((ukeys.numel(), len(graphs)), dtype=torch.float32, device=dev)
        V.index_put_((inv, kind), vals, accumulate=True)
        U, perm = CSRGraph.from_coo(ukeys // n, ukeys % n, None, n, n, return_perm=True, validate=False)
        return RelationStack(U, V[perm], max_nnz)

    def patterns(self, num_layers: int):
        """([P_1 .. P_L], [D_1 .. D_{L-1}], [slots of P_l that D_l keeps]) for L = num_layers (built on first use)."""
        while len(self._P) < num_layers:
            A = self.U if not self._P else self._D[-1]
            P = CSRGraph.pattern_product(A, self.U, max_nnz=self.max_nnz, validate=False)
            D, keep = _drop_diagonal(P)
            for g in (P, D):  # transposes the backward and the column sums walk, and their SpMM plans
                _plan(g)
                _plan(g.transpose())
            self._P.append(P)
            self._D.append(D)
            self._keep.append(keep)
        self.U.transpose()
        return self._P[:num_layers], self._D[:num_layers - 1], self._keep[:num_layers - 1]

    def gcn_pattern(self, num_layers: int):
        """(g, src, diag) for the final gcn_conv on P_L: g the CSR of (D_L + I)^T, src the int64 slot of P_L each
        edge of g reads (0 on the diagonal), diag the bool mask of the self-loops."""
        if num_layers not in self._gcn:
            self.patterns(num_layers)
            self._gcn[num_layers] = _gcn_pattern(self._D[num_layers - 1], self._keep[num_layers - 1], self.n)
        return self._gcn[num_layers]


def _gcn_pattern(D, idx, n, lo=0):
    """(g, src, diag) of the final gcn_conv on the rows [lo, lo + D.n_rows) of D_L (kept slots `idx` of P_L): g the CSR
    of (D_L + I)^T restricted to those rows, [n, D.n_rows] (columns = row index i - lo, self-loops for j in the block),
    src the int64 slot of P_L each edge of g reads (0 on the diagonal), diag the bool mask of the self-loops."""
    n_loc, dev = D.n_rows, D.device
    rows = torch.cat([D.col.long(), torch.arange(lo, lo + n_loc, device=dev)])   # j: row of H^T
    cols = torch.cat([D.edge_rows().long(), torch.arange(n_loc, device=dev)])    # i - lo
    g, perm = CSRGraph.from_coo(rows, cols, None, n, n_loc, return_perm=True, validate=False)
    diag = perm >= D.nnz
    src = idx[torch.where(diag, torch.zeros_like(perm), perm)] if D.nnz else torch.zeros_like(perm)
    _plan(g)
    _plan(g.transpose())
    return g, src, diag


def _plan(g):
    """Host-side SpMM plans of g, computed now so that a training step reads nothing back from the device."""
    g.long_row_plan()
    g.rows_per_team()
    g.edge_rows()


class GTConv(nn.Module):
    """GTN/models/GTConv.py: softmax-weighted sum of the edge-type adjacencies (1x1 convolution)."""

    def __init__(self, in_channels, out_channels, **kwargs):
        super(GTConv, self).__init__(**kwargs)
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.weight = nn.Parameter(torch.Tensor(out_channels, in_channels, 1, 1))
        self.bias = None
        self.scale = nn.Parameter(torch.Tensor([0.1]), requires_grad=False)

    def forward(self, A):
        return torch.sum(A * F.softmax(self.weight, dim=1), dim=1)

    def forward_sparse(self, stack):
        """The same soft selection on a RelationStack: values [nnz_U, out_channels] on its union pattern."""
        s = F.softmax(self.weight, dim=1)[:, :, 0, 0]  # [C, K]
        return torch.sum(stack.V.unsqueeze(1) * s.unsqueeze(0), dim=2)


class GTLayer(nn.Module):
    """GTN/models/GTLayer.py: one metapath-composition step (dense bmm; out of scope, kept as the reference has it)."""

    def __init__(self, in_channels, out_channels, first=True):
        super(GTLayer, self).__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.first = first
        self.conv1 = GTConv(in_channels, out_channels)
        if self.first:
            self.conv2 = GTConv(in_channels, out_channels)

    def forward_sparse(self, stack, P, H_=None, D=None, U_rows=None):
        """One composition step on a RelationStack: H_ None gives a·b on P = pattern(U·U); else H_ holds the
        normalised values on D (an earlier H without its diagonal) and the result is H_·a on P = pattern(D·U).
        U_rows = (rows [lo, hi) of U as a CSRGraph, first slot, end slot): a·b of those rows only, on P = their
        block of pattern(U·U)."""
        a = self.conv1.forward_sparse(stack)
        if self.first:
            A, a_A = (stack.U, a) if U_rows is None else (U_rows[0], a[U_rows[1]:U_rows[2]])
            H = spgemm_values(A, a_A, stack.U, self.conv2.forward_sparse(stack), P)
            W = [(F.softmax(self.conv1.weight, dim=1)).detach(), (F.softmax(self.conv2.weight, dim=1)).detach()]
        else:
            H = spgemm_values(D, H_, stack.U, a, P)
            W = [(F.softmax(self.conv1.weight, dim=1)).detach()]
        return H, W

    def forward(self, A, H_=None):
        if self.first:
            a = self.conv1(A)
            b = self.conv2(A)
            H = torch.bmm(a, b)
            W = [(F.softmax(self.conv1.weight, dim=1)).detach(), (F.softmax(self.conv2.weight, dim=1)).detach()]
        else:
            a = self.conv1(A)
            H = torch.bmm(H_, a)
            W = [(F.softmax(self.conv1.weight, dim=1)).detach()]
        return H, W


class GTN_Model(nn.Module):
    """GTN/models/GTN.py:22-88.  state_dict: `layers.{l}.conv{1,2}.{weight,scale}`, `weight`, `bias`,
    `linear1.*`, `linear2.*`."""

    def __init__(self, num_edge, num_channels, w_in, w_out, num_class, num_layers, is_norm, **kwargs):
        super(GTN_Model, self).__init__(**kwargs)
        self.num_edge = num_edge
        self.num_channels = num_channels
        self.w_in = w_in
        self.w_out = w_out
        self.num_class = num_class
        self.num_layers = num_layers
        self.is_norm = is_norm
        self.layers = nn.ModuleList([GTLayer(num_edge, num_channels, first=(i == 0)) for i in range(num_layers)])
        self.weight = nn.Parameter(torch.Tensor(w_in, w_out))
        self.bias = nn.Parameter(torch.Tensor(w_out))
        self.linear1 = nn.Linear(self.w_out * self.num_channels, self.w_out)
        self.linear2 = nn.Linear(self.w_out, self.num_class)
        self.reset_parameters()

    def reset_parameters(self):
        nn.init.xavier_uniform_(self.weight)
        nn.init.zeros_(self.bias)

    def gcn_conv(self, X, H):
        return gcn_conv(X, H, self.weight)

    def normalization(self, H):
        return torch.stack([norm(H[i, :, :]) for i in range(self.num_channels)], dim=0)

    def forward(self, A, X, target_x):
        if isinstance(A, (RelationStack, PartitionedRelationStack)):
            return self._forward_sparse(A, X, target_x)
        A = A.unsqueeze(0).permute(0, 3, 1, 2)
        Ws = []
        for i in range(self.num_layers):
            if i == 0:
                H, W = self.layers[i](A)
            else:
                H = self.normalization(H)
                H, W = self.layers[i](A, H)
            Ws.append(W)
        X_ = torch.cat([F.relu(self.gcn_conv(X, H[i])) for i in range(self.num_channels)], dim=1)
        X_ = F.relu(self.linear1(X_))
        y = self.linear2(X_[target_x])
        return y, Ws

    def _forward_sparse(self, stack, X, target_x):
        """forward() on a RelationStack: the same computation with every H a [nnz(P_l), C] value tensor.
        On a PartitionedRelationStack, forward() on this rank's rows: X = X[lo:hi], target_x = ids local to the block;
        returns (logits of target_x, Ws).  The column sums of norm and the gcn_conv degrees are then completed by
        rank-ordered all-reduces, and the gcn_conv output by a reduce-scatter.  Collective: every rank runs it, and
        its backward, in the same order."""
        if isinstance(stack, PartitionedRelationStack):
            ps = stack
            if (ps.num_edge, ps.num_layers, ps.width) != (self.num_edge, self.num_layers, self.num_channels * self.w_out):
                raise ValueError(f"GTN_Model: the partitioned stack has {ps.num_edge} edge types, {ps.num_layers} "
                                 f"layers and width {ps.width}; the model {self.num_edge}, {self.num_layers} and "
                                 f"{self.num_channels * self.w_out} (num_channels * w_out)")
            if X.dim() != 2 or X.shape[0] != ps.n_local:
                raise ValueError(f"GTN_Model: X_local must hold this rank's {ps.n_local} rows, got {tuple(X.shape)}")
            stack, (Ps, Ds, keeps), (g, src, diag), U_rows = ps.stack, (ps.P, ps.D, ps.keep), ps.gcn, ps.U_rows
            red = ps.reduce
        else:
            if stack.num_edge != self.num_edge:
                raise ValueError(f"GTN_Model: the stack has {stack.num_edge} edge types, the model {self.num_edge}")
            Ps, Ds, keeps = stack.patterns(self.num_layers)
            g, src, diag = stack.gcn_pattern(self.num_layers)
            red = U_rows = None

        def reduce(site):  # the column sums over every rank's rows; None: one GPU's sums are whole
            return None if red is None else (lambda x: rank_all_reduce(red, site, x))
        Ws = []
        H = None
        for i in range(self.num_layers):
            if i == 0:
                H, W = self.layers[i].forward_sparse(stack, Ps[0], U_rows=U_rows)
            else:
                # norm(H): diagonal dropped, columns scaled
                Hn = column_normalize(Ds[i - 1], H[keeps[i - 1]], reduce=reduce(f"norm{i}"))
                H, W = self.layers[i].forward_sparse(stack, Ps[i], Hn, Ds[i - 1])
            Ws.append(W)
        XW = torch.mm(X, self.weight)
        one = torch.ones((), device=H.device, dtype=H.dtype)
        vals = torch.where(diag.unsqueeze(1), one, H[src])
        Y = _normalized_aggregate(g, vals, XW, reduce=reduce("deg"))  # [N, C * w_out]; partial on a row block
        X_ = F.relu(Y) if red is None else row_reduce_scatter(red, "out", Y, relu=True)
        X_ = F.relu(self.linear1(X_))
        y = self.linear2(X_[target_x])
        return y, Ws
