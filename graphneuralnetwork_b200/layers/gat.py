"""Drop-in GAT layers and models (class names, ctor signatures, parameter names/shapes and
forward signatures of /root/reference GAT/models/layers.py and GAT/models/GAT.py).

What changes: the all-pairs `[N,N,2F']` score tensor, masked softmax and dense
`attention·Wh` (GAT/models/layers.py:25-32) become one fused kernel over the CSR of
`adj > 0`; `GATBase.forward` runs all heads of a layer in ONE launch by concatenating the
per-head `W` (state_dict stays `attentions.AttentionHead{k}.W [in,F']`, `.a [2F',1]`).
The dense `h·W` stays torch.mm; the per-node score halves `Wh·a[:F']`, `Wh·a[F':]` are a
[N,H·F']x[H·F',2H] torch product so autograd reaches `a`.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _lib
from ..functional import (attention_keep_mask, gat_aggregate, halo_exchange, next_attention_dropout,
                          require_partition_dtype, spmm_values)
from ..graph import CSRGraph, adj_cache
from ..partition import PartitionedGraph

# True: draw the attention dropout as an explicit [nnz, H] mask (attention_keep_mask) instead of the seeded
# in-kernel stream — the parity tests replay reference masks through this hook
EXPLICIT_DROPOUT_MASK = False

_pattern_cache = {}


def _coo_pattern(indices, shape):
    """CSR pattern + COO->CSR permutation of an `indices [2, nnz]` tensor, built once per tensor.

    The reference rebuilds `edge = adj.nonzero().t()` on every forward (GAT/models/layers.py:98) and the
    caching allocator hands the same block back, so (data_ptr, _version, shape) alone would match a
    DIFFERENT graph of equal nnz: a hit also requires that the cached entry's tensor object is still
    alive and is this very tensor (weakref identity, as graph._AdjCache does)."""
    import weakref
    key = (indices.data_ptr(), indices._version, tuple(indices.shape), tuple(shape))
    hit = _pattern_cache.get(key)
    if hit is not None:
        ref, value = hit
        if ref() is indices:
            return value
    for k in [k for k, (r, _) in _pattern_cache.items() if r() is None]:  # evict entries of dead tensors
        _pattern_cache.pop(k)
    if len(_pattern_cache) >= 16:
        _pattern_cache.pop(next(iter(_pattern_cache)))
    value = CSRGraph.from_coo(indices[0], indices[1], None, int(shape[0]), int(shape[1]), return_perm=True)
    _pattern_cache[key] = (weakref.ref(indices), value)
    return value


class SpecialSpmmFunction:
    """`SpecialSpmmFunction.apply(indices, values, shape, b)` of GAT/models/layers.py:43-64: the product
    of a sparse matrix given as COO (indices, values) with a dense matrix, differentiable in `values`
    and `b` only.  Forward = CSR SpMM; backward = edge-gradient SDDMM + transpose SpMM — the
    reference's backward goes through a dense N x N `grad_output @ b.T` (layers.py:59-61)."""

    @staticmethod
    def apply(indices, values, shape, b):
        assert not indices.requires_grad
        pattern, perm = _coo_pattern(indices, shape)
        return spmm_values(pattern, values[perm], b)


class SpecialSpmm(nn.Module):
    def forward(self, indices, values, shape, b):
        return SpecialSpmmFunction.apply(indices, values, shape, b)


def _fused_heads(x, adj, Ws, a_srcs, a_dsts, alpha, mode, elu, dropout, training, out=None):
    """All heads of one attention layer: x [N,in]; Ws list of [in,F']; a_* list of [F'].
    adj may be a partition.PartitionedGraph: x is then the rank's own rows, and so is the result."""
    if isinstance(adj, PartitionedGraph):
        return _fused_heads_partitioned(x, adj, Ws, a_srcs, a_dsts, alpha, mode, elu, dropout, training)
    g = adj_cache.get(adj)
    H = len(Ws)
    Fp = Ws[0].shape[1]
    W_cat = Ws[0] if H == 1 else torch.cat(list(Ws), dim=1)
    Wh = torch.mm(x, W_cat)  # [N, H*F']  (layers.py:23, all heads at once)
    Wh3 = Wh.view(-1, H, Fp)
    a_src = a_srcs[0].view(1, Fp) if H == 1 else torch.stack(list(a_srcs), dim=0)
    a_dst = a_dsts[0].view(1, Fp) if H == 1 else torch.stack(list(a_dsts), dim=0)
    # scores are fp32 even for bf16 features (the softmax statistics live in fp32)
    s = (Wh3.float() * a_src.float().unsqueeze(0)).sum(-1)  # [N,H] = Wh_i·a[:F']
    t = (Wh3.float() * a_dst.float().unsqueeze(0)).sum(-1)  # [N,H] = Wh_j·a[F':]
    keep = drop = None
    if training and dropout > 0.0:  # post-softmax dropout, layers.py:31
        if EXPLICIT_DROPOUT_MASK:
            keep = attention_keep_mask(g, H, dropout)
        else:
            drop = next_attention_dropout(dropout, Wh.device)  # seeded: no [nnz, H] mask is materialised
    return gat_aggregate(g, Wh, s, t, H, Fp, alpha, mode=mode, elu=elu, keep=keep, out=out, dropout=drop)


def _fused_heads_partitioned(x, pg, Ws, a_srcs, a_dsts, alpha, mode, elu, dropout, training):
    """`_fused_heads` on this rank's row block: Wh of the own rows, the halo rows' Wh from their owners
    (functional.halo_exchange), s of the own rows, t of all table rows, and the fused kernels over the block in the
    combined column space.  The backward returns d Wh of the halo rows (from the aggregation and from t) to their
    owners; d a_src / d a_dst are this rank's share, summed over the ranks by partition.allreduce_gradients.
    x has the partition's dtype (fp32 or bf16); s / t are fp32 from the same expression as `_fused_heads`, so one rank
    computes the bits of one GPU in either dtype."""
    H = len(Ws)
    Fp = Ws[0].shape[1]
    require_partition_dtype(pg, x, "GAT on a PartitionedGraph")
    if H * Fp > 256:
        raise _lib.GnnError(f"GAT on a PartitionedGraph: H*F' = {H * Fp} exceeds the 256 columns of one fused "
                            "attention call")
    g, edge_slot_base = pg.attention()
    W_cat = Ws[0] if H == 1 else torch.cat(list(Ws), dim=1)
    Wh = halo_exchange(pg, torch.mm(x, W_cat))  # [n_local + n_halo, H*F']
    Wh3 = Wh.view(-1, H, Fp)
    a_src = a_srcs[0].view(1, Fp) if H == 1 else torch.stack(list(a_srcs), dim=0)
    a_dst = a_dsts[0].view(1, Fp) if H == 1 else torch.stack(list(a_dsts), dim=0)
    s = (Wh3[:pg.n_local].float() * a_src.float().unsqueeze(0)).sum(-1)  # [n_local, H]
    t = (Wh3.float() * a_dst.float().unsqueeze(0)).sum(-1)               # [n_local + n_halo, H]
    keep = drop = None
    if training and dropout > 0.0:
        if EXPLICIT_DROPOUT_MASK:
            keep = attention_keep_mask(g, H, dropout)
        else:
            # the whole graph's mask for this block's edges
            drop = next_attention_dropout(dropout, Wh.device).with_slot_base(edge_slot_base)
    return gat_aggregate(g, Wh, s, t, H, Fp, alpha, mode=mode, elu=elu, keep=keep, dropout=drop)


class GraphAttentionLayer(nn.Module):
    """One attention head (GAT/models/layers.py:6-40 == HAN/models/NodeAttention.py:6-41)."""

    def __init__(self, in_features, out_features, dropout, alpha, concat=True, **kwargs):
        super(GraphAttentionLayer, self).__init__(**kwargs)
        self.dropout = dropout
        self.in_features = in_features
        self.out_features = out_features
        self.alpha = alpha
        self.concat = concat
        self.W = nn.Parameter(torch.empty(size=(in_features, out_features)))
        nn.init.xavier_uniform_(self.W.data, gain=1.414)
        self.a = nn.Parameter(torch.empty(size=(2 * out_features, 1)))
        nn.init.xavier_uniform_(self.a.data, gain=1.414)
        self.leakyrelu = nn.LeakyReLU(self.alpha)

    def _halves(self):
        Fp = self.out_features
        return self.a[:Fp, 0], self.a[Fp:, 0]

    def forward(self, h, adj):
        a_src, a_dst = self._halves()
        return _fused_heads(h, adj, [self.W], [a_src], [a_dst], self.alpha, _lib.GAT_SOFTMAX,
                            1 if self.concat else 0, self.dropout, self.training)

    def __repr__(self):
        return self.__class__.__name__ + ' (' + str(self.in_features) + ' -> ' + str(self.out_features) + ')'


class SpGraphAttentionLayer(nn.Module):
    """Edge-list variant (GAT/models/layers.py:72-134): att = exp(-LeakyReLU(a·[h_i||h_j]))
    normalised by its row sum, dropout on the un-normalised edge weights (layers.py:115)."""

    def __init__(self, in_features, out_features, dropout, alpha, concat=True):
        super(SpGraphAttentionLayer, self).__init__()
        self.in_features = in_features
        self.out_features = out_features
        self.alpha = alpha
        self.concat = concat
        self.W = nn.Parameter(torch.zeros(size=(in_features, out_features)))
        nn.init.xavier_normal_(self.W.data, gain=1.414)
        self.a = nn.Parameter(torch.zeros(size=(1, 2 * out_features)))
        nn.init.xavier_normal_(self.a.data, gain=1.414)
        self.dropout = nn.Dropout(dropout)
        self.leakyrelu = nn.LeakyReLU(self.alpha)

    def _halves(self):
        Fp = self.out_features
        return self.a[0, :Fp], self.a[0, Fp:]

    def forward(self, input, adj):
        a_src, a_dst = self._halves()
        return _fused_heads(input, adj, [self.W], [a_src], [a_dst], self.alpha, _lib.GAT_EXPNEG,
                            1 if self.concat else 0, self.dropout.p, self.training)

    def __repr__(self):
        return self.__class__.__name__ + ' (' + str(self.in_features) + ' -> ' + str(self.out_features) + ')'


class GATBase(nn.Module):
    """Two-layer GAT skeleton (GAT/models/GAT.py:7-18): `attentions` = the first layer's heads
    (state_dict `attentions.AttentionHead{k}.{W,a}`), `out_att` = the single-head output layer.
    `_head_cls` / `_mode` select the masked-softmax (dense) or exp(-LeakyReLU) (edge-list) scores.
    The heads never run one by one: `forward` hands all of them to one fused launch, whose
    column block k is head k — the reference's `torch.cat(..., dim=1)`."""

    _head_cls = None
    _mode = _lib.GAT_SOFTMAX

    def __init__(self, dropout, **kwargs):
        super().__init__(**kwargs)
        self.dropout = dropout
        self.attentions = nn.ModuleList()
        self.out_att = None

    def _build(self, nfeat, nhid, nclass, alpha, nheads):
        for k in range(nheads):
            self.attentions.add_module(f'AttentionHead{k}', self._head_cls(nfeat, nhid, self.dropout, alpha, True))
        self.out_att = self._head_cls(nhid * nheads, nclass, self.dropout, alpha, False)

    def forward(self, x, adj):
        # CSR of adj > 0, built once per adjacency tensor; a PartitionedGraph is passed through (x = own rows)
        graph = adj if isinstance(adj, PartitionedGraph) else adj_cache.get(adj)
        heads = list(self.attentions)
        halves = [head._halves() for head in heads]
        p_att = heads[0].dropout.p if isinstance(heads[0].dropout, nn.Dropout) else heads[0].dropout
        x = F.dropout(x, self.dropout, training=self.training)
        x = _fused_heads(x, graph, [head.W for head in heads], [h[0] for h in halves], [h[1] for h in halves],
                         heads[0].alpha, self._mode, 1 if heads[0].concat else 0, p_att, self.training)
        x = F.dropout(x, self.dropout, training=self.training)
        # `F.elu(self.out_att(x, adj))` (GAT.py:18): the ELU rides in the output layer's kernel epilogue
        oa = self.out_att
        a_src, a_dst = oa._halves()
        p_out = oa.dropout.p if isinstance(oa.dropout, nn.Dropout) else oa.dropout
        return _fused_heads(x, graph, [oa.W], [a_src], [a_dst], oa.alpha, self._mode, 1, p_out, self.training)


class GAT(GATBase):
    """Dense-adjacency GAT (GAT/models/GAT.py:21-28): `adj` is used only as the mask `adj > 0`."""

    _head_cls = GraphAttentionLayer

    def __init__(self, nfeat, nhid, nclass, dropout, alpha, nheads, **kwargs):
        super().__init__(dropout, **kwargs)
        self._build(nfeat, nhid, nclass, alpha, nheads)


class SpGAT(GATBase):
    """Edge-list GAT (GAT/models/GAT.py:31-38)."""

    _head_cls = SpGraphAttentionLayer
    _mode = _lib.GAT_EXPNEG

    def __init__(self, nfeat, nhid, nclass, dropout, alpha, nheads, **kwargs):
        super().__init__(dropout, **kwargs)
        self._build(nfeat, nhid, nclass, alpha, nheads)
