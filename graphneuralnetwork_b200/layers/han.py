"""Drop-in HAN node-level attention, semantic attention and model for /root/reference
HAN/models/NodeAttention.py:44-62, SemanticAttention.py:5-20 and HAN.py:7-41.

Fixed by the reference: class names, constructor / forward signatures and the state_dict keys
(`layers.{l}.gat_layers.meta_path_model{m}.attentions.AttentionHead{k}.{W,a}`,
`layers.{l}.semantic_attention.project.{0,2}.*`, `predict.*`).

Re-designed for the device:
  * each metapath's `GATConv` runs all its heads in ONE fused launch over the CSR of that
    metapath's float64 0/1 adjacency (`adj > 0`, converted once and cached);
  * the second `F.elu` the reference applies when `num_class is None` (NodeAttention.py:62) is
    fused into the same kernel's epilogue (double ELU) whenever no dropout sits between them;
  * without autograd the M metapath kernels write straight into their `[:, m, :]` slice of the
    `[N, M, H·F']` semantic stack — `torch.stack` (HAN.py:21) never copies;
  * semantic attention (SemanticAttention.py:15-20) keeps only its `[N·M, D]·[D, K]` product as a GEMM; tanh, the
    K→1 projection, the mean over nodes, `softmax_M` and the weighted sum are two launches forward and two backward
    (`functional.semantic_attention`), nothing of `[N, M, ·]` shape besides P is materialised (bf16 / CPU tensors
    take the plain torch formula).
"""
import torch
from torch import nn
import torch.nn.functional as F

from .. import _lib
from ..functional import (SEMANTIC_MAX_K, SEMANTIC_MAX_M, AttentionDropout, gat_aggregate, halo_exchange,
                          next_attention_dropout, require_partition_dtype, semantic_attention,
                          semantic_attention_partitioned)
from ..graph import CSRGraph, adj_cache
from ..partition import PartitionedGraph, PartitionedMetapaths
from .gat import GraphAttentionLayer, _fused_heads
from . import gat as _gat


class GATConv(nn.Module):
    """Multi-head node attention over one metapath graph (NodeAttention.py:44-62)."""

    def __init__(self, feat_size, hidden_size, dropout, num_heads, alpha=0.2, num_class=None, **kwargs):
        super().__init__(**kwargs)
        self.dropout, self.num_class = dropout, num_class
        self.attentions = nn.ModuleList()
        for k in range(num_heads):
            self.attentions.add_module(f'AttentionHead{k}', GraphAttentionLayer(feat_size, hidden_size, dropout=dropout,
                                                                                alpha=alpha, concat=True))
        if num_class is not None:
            self.out_att = GraphAttentionLayer(hidden_size * num_heads, num_class, dropout=dropout, alpha=alpha,
                                               concat=False)

    def forward(self, x, adj, out=None):
        """`out` (optional, no autograd): a `[N, H·F']` strided view the kernel fills in place."""
        graph = adj_cache.get(adj)
        heads = list(self.attentions)
        halves = [head._halves() for head in heads]
        drop_active = self.training and self.dropout > 0.0
        # heads are concat=True => ELU (NodeAttention.py:35); with num_class None the concatenation gets
        # a second ELU (NodeAttention.py:62), fused as elu=2 unless a dropout separates the two
        double_elu = self.num_class is None and not drop_active
        x = F.dropout(x, self.dropout, training=self.training)
        y = _fused_heads(x, graph, [head.W for head in heads], [h[0] for h in halves], [h[1] for h in halves],
                         heads[0].alpha, _lib.GAT_SOFTMAX, 2 if double_elu else 1, self.dropout, self.training,
                         out=out if double_elu else None)
        if double_elu:
            return y
        y = F.dropout(y, self.dropout, training=self.training)
        if self.num_class is None:
            y = F.elu(y)
        else:  # F.elu(self.out_att(y, adj)) (NodeAttention.py:61): the ELU rides in the output head's epilogue
            oa = self.out_att
            a_src, a_dst = oa._halves()
            y = _fused_heads(y, graph, [oa.W], [a_src], [a_dst], oa.alpha, _lib.GAT_SOFTMAX, 1, oa.dropout,
                             self.training)
        if out is not None:
            out.copy_(y)
            return out
        return y


class SemanticAttention(nn.Module):
    """β = softmax_M(mean_N(q·tanh(W z + b)));  out = Σ_m β_m z_m  (SemanticAttention.py:5-20)."""

    def __init__(self, in_size, hidden_size=128):
        super().__init__()
        self.project = nn.Sequential(nn.Linear(in_size, hidden_size), nn.Tanh(), nn.Linear(hidden_size, 1, bias=False))

    def forward(self, z):
        n, m, d = z.shape
        lin, proj = self.project[0], self.project[2]
        if (getattr(self, "fused", True) and z.is_cuda and z.dtype == torch.float32 and 0 < m <= SEMANTIC_MAX_M and n > 0
                and lin.out_features <= SEMANTIC_MAX_K and lin.weight.dtype == torch.float32):
            # one GEMM + two launches (tanh . q, mean over nodes, softmax over M, weighted sum: csrc/semantic.cu)
            return semantic_attention(z, lin.weight, lin.bias, proj.weight)
        scores = self.project(z.reshape(n * m, d)).view(n, m).mean(dim=0)  # [M]
        beta = torch.softmax(scores, dim=0)
        return torch.einsum('m,nmd->nd', beta, z)


class HANLayer(nn.Module):
    """M metapath GATs over the same node features + semantic attention (HAN.py:7-23)."""

    def __init__(self, num_meta_paths, in_size, out_size, layer_num_heads, dropout, **kwargs):
        super().__init__(**kwargs)
        self.gat_layers = nn.ModuleList()
        for m in range(num_meta_paths):
            self.gat_layers.add_module(f'meta_path_model{m}', GATConv(in_size, out_size, dropout, layer_num_heads))
        self.semantic_attention = SemanticAttention(in_size=out_size * layer_num_heads)
        self._width = out_size * layer_num_heads

    def _batched(self, gs, h):
        """All M metapath GATConvs (HAN.py:16-21) in ONE attention launch over the block diagonal of the M graphs:
        `z[:, m, :]` is metapath m's multi-head output — the tensor `torch.stack(semantic_embeddings, dim=1)` builds.
        Per-metapath feature dropout (NodeAttention.py:59: every GATConv draws its own mask) is kept."""
        convs = list(self.gat_layers)
        M, n = len(convs), h.shape[0]
        graphs = [adj_cache.get(g) for g in gs]
        big = CSRGraph.block_diagonal(graphs)
        heads0 = list(convs[0].attentions)
        H, Fp, alpha = len(heads0), heads0[0].out_features, heads0[0].alpha
        p, training = convs[0].dropout, self.training
        drop_active = training and p > 0.0
        Ws = [torch.cat([hd.W for hd in conv.attentions], dim=1) for conv in convs]            # M x [F_in, H*Fp]
        # one product per metapath, exactly the per-GATConv GEMM shape: Wh is then bit-identical to the unbatched path
        # (a single [F_in, M*H*Fp] product rounds differently, and LeakyReLU's kink at s_i + t_j = 0 turns a 1e-6
        # perturbation of one score into a 1e-4 change of that edge's gradient: measured on the ACM-sized golden);
        # per-metapath feature dropout draws its own mask per GATConv as the reference does
        Wh = torch.cat([torch.mm(F.dropout(h, p, training=True) if drop_active else h, W) for W in Ws], dim=1)
        a = torch.stack([torch.stack([hd.a[:, 0] for hd in conv.attentions]) for conv in convs])  # [M, H, 2*Fp]
        Wh4 = Wh.view(n, M, H, Fp).float()
        s = (Wh4 * a[None, :, :, :Fp].float()).sum(-1).permute(1, 0, 2).reshape(M * n, H)     # batched-row major
        t = (Wh4 * a[None, :, :, Fp:].float()).sum(-1).permute(1, 0, 2).reshape(M * n, H)
        keep = drop = None
        if drop_active:
            if _gat.EXPLICIT_DROPOUT_MASK:
                keep = _gat.attention_keep_mask(big, H, p)
            else:
                drop = next_attention_dropout(p, Wh.device)
        double_elu = convs[0].num_class is None and not drop_active
        z = gat_aggregate(big, Wh, s, t, H, Fp, alpha, mode=_lib.GAT_SOFTMAX, elu=2 if double_elu else 1, keep=keep,
                          dropout=drop, batch=M)                                                 # [N, M*H*Fp]
        if not double_elu:
            z = F.elu(F.dropout(z, p, training=training))  # NodeAttention.py:60-62, all metapaths at once
        return z.view(n, M, H * Fp)

    def _batched_partitioned(self, pm, h):
        """`_batched` on this rank's row block of a PartitionedMetapaths (h = the own rows): the per-metapath h·W_m on
        the own rows, ONE halo exchange of the stacked Wh, s of the own rows and t of all table rows, one batched-
        rectangular attention launch (forward and backward) and semantic attention over the global node count.
        Feature dropout (GATConv.dropout, NodeAttention.py:59-60) draws on the own rows; the attention dropout
        (the heads' GraphAttentionLayer.dropout, NodeAttention.py:31 — equal to it when built by the constructor)
        draws the whole set's mask for the block's edges.
        h has the partition's dtype (fp32 or bf16).  In bf16 the halo exchange moves bf16 rows and the node-level
        attention runs in the bf16 batched-rectangular kernels; the split semantic kernels are fp32 only, so they take
        z and the projection weights as fp32 views (autograd casts the gradients back) and the result is cast to h's
        dtype.  This differs from the 1-GPU bf16 HAN, whose semantic attention is the plain torch formula in bf16:
        the two agree to bf16 tolerance, not bit for bit."""
        convs = list(self.gat_layers)
        M = len(convs)
        heads0 = list(convs[0].attentions)
        H, Fp, alpha = len(heads0), heads0[0].out_features, heads0[0].alpha
        lin = self.semantic_attention.project[0]
        # the refusals depend on the replicated model and the features' dtype only: every rank raises together
        if M != len(pm):
            raise _lib.GnnError(f"HANLayer: {M} metapath models for {len(pm)} metapath graphs")
        require_partition_dtype(pm, h, "HANLayer on PartitionedMetapaths")
        if any(c.num_class is not None for c in convs) or H * Fp > 256 or \
                M > SEMANTIC_MAX_M or lin.out_features > SEMANTIC_MAX_K:
            raise _lib.GnnError("HANLayer on PartitionedMetapaths: needs num_class None, H*F' <= 256, "
                                f"M <= {SEMANTIC_MAX_M} and a semantic hidden width <= {SEMANTIC_MAX_K} (got "
                                f"H*F' = {H * Fp}, M = {M}, K = {lin.out_features})")
        g, shift = pm.attention()
        n = pm.n_local
        p, p_att, training = convs[0].dropout, heads0[0].dropout, self.training
        drop_active = training and p > 0.0
        Ws = [torch.cat([hd.W for hd in conv.attentions], dim=1) for conv in convs]
        Wh = torch.cat([torch.mm(F.dropout(h, p, training=True) if drop_active else h, W) for W in Ws], dim=1)
        Wh = halo_exchange(pm.union, Wh)                                                         # [n_comb, M*H*Fp]
        nc = Wh.shape[0]
        a = torch.stack([torch.stack([hd.a[:, 0] for hd in conv.attentions]) for conv in convs])  # [M, H, 2*Fp]
        Wh4 = Wh.view(nc, M, H, Fp).float()
        s = (Wh4[:n] * a[None, :, :, :Fp].float()).sum(-1).permute(1, 0, 2).reshape(M * n, H)
        t = (Wh4 * a[None, :, :, Fp:].float()).sum(-1).permute(1, 0, 2).reshape(M * nc, H)
        keep = drop = None
        if training and p_att > 0.0:
            if _gat.EXPLICIT_DROPOUT_MASK:
                keep = _gat.attention_keep_mask(g, H, p_att)
            else:
                d = next_attention_dropout(p_att, Wh.device)
                drop = AttentionDropout(d.p, d.seed, d.seed_dev, slot_shift=shift)  # the whole set's mask
        double_elu = not drop_active
        z = gat_aggregate(g, Wh, s, t, H, Fp, alpha, mode=_lib.GAT_SOFTMAX, elu=2 if double_elu else 1, keep=keep,
                          dropout=drop, batch=M)                                                 # [n, M*H*Fp]
        if not double_elu:
            z = F.elu(F.dropout(z, p, training=training))
        sem = self.semantic_attention
        b1 = None if lin.bias is None else lin.bias.float()
        out = semantic_attention_partitioned(z.view(n, M, H * Fp).float(), lin.weight.float(), b1,
                                             sem.project[2].weight.float(), pm.n_total, pm.world, pm.group)
        return out.to(h.dtype)

    def forward(self, gs, h):
        if isinstance(gs, PartitionedMetapaths):
            return self._batched_partitioned(gs, h)
        if any(isinstance(g, PartitionedGraph) for g in gs):
            raise _lib.GnnError("HANLayer: metapath graphs on a PartitionedGraph are not supported (the batched "
                                "metapath attention runs on one GPU)")
        convs = list(self.gat_layers)
        heads0 = list(convs[0].attentions)
        if (getattr(self, "batched", True) and len(convs) > 1 and all(c.num_class is None for c in convs)
                and len(heads0) * heads0[0].out_features <= 256 and h.dtype in (torch.float32, torch.bfloat16)):
            return self.semantic_attention(self._batched(gs, h))
        if torch.is_grad_enabled() and (h.requires_grad or any(p.requires_grad for p in self.parameters())):
            z = torch.stack([conv(h, g).flatten(1) for g, conv in zip(gs, convs)], dim=1)  # (N, M, H·F')
        else:
            z = h.new_empty(h.shape[0], len(convs), self._width)  # the kernels write the features' dtype (fp32 / bf16)
            for m, (g, conv) in enumerate(zip(gs, convs)):
                conv(h, g, out=z[:, m, :])
        return self.semantic_attention(z)


class HANModel(nn.Module):
    """Stack of HANLayers + linear classifier (HAN.py:26-41)."""

    def __init__(self, num_mate_paths, in_size, hidden_size, out_size, num_heads, dropout, **kwargs):
        super().__init__(**kwargs)
        widths = [in_size] + [hidden_size * k for k in num_heads]
        self.layers = nn.ModuleList(HANLayer(num_mate_paths, widths[l], hidden_size, num_heads[l], dropout)
                                    for l in range(len(num_heads)))
        self.predict = nn.Linear(widths[-1], out_size)

    def forward(self, g, h):
        """g: the M metapath adjacencies, or a PartitionedMetapaths (h = this rank's rows; so is the result)."""
        if isinstance(g, PartitionedMetapaths):
            graphs = g
        else:
            graphs = [a if isinstance(a, PartitionedGraph) else adj_cache.get(a) for a in g]  # dense float64 masks -> CSR, once per graph
        for layer in self.layers:
            h = layer(graphs, h)
        return self.predict(h)
