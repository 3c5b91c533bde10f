"""Drop-in GCN layer and model for /root/reference GCN/GCN.py:5-52.

Fixed by the reference (callers, checkpoints and its own dispatch depend on them): the class
names — `GCN_Model.forward` routes the adjacency to children whose `_get_name()` is
'Graph_conv_layer' (GCN/GCN.py:23) — the constructor / forward signatures, and the state_dict
keys `gcn_blocks.gcn{i}.dense.weight [out,in]`, `gcn_blocks.gcn{i}.bias [out]`.

Re-designed for the device:
  * `torch.spmm(adj, support) + bias` (GCN.py:43-45) is ONE launch of the row-block streaming
    CSR SpMM with the bias folded into its row flush (`functional.gcn_aggregate`);
  * the `nn.ReLU` module that follows every hidden layer (GCN.py:12,19) is folded into the same
    launch: the model walks `gcn_blocks` with one step of lookahead and, when a graph layer is
    followed by a ReLU, asks the layer for the fused activation and skips the module;
  * the COO adjacency is converted to CSR (+ transpose for the backward) once per graph;
  * `adj` may also be a `partition.PartitionedGraph` (one rank's share of a graph split over GPUs): X is then the
    rank's own rows, the aggregation is the partitioned SpMM with the same fused epilogue, and the module tree and
    state_dict are unchanged, so a checkpoint moves between 1 and N GPUs.
The dense `X·Wᵀ` stays a torch matmul (north_star): transform first, aggregate on the narrow
width.
"""
import torch
from torch import nn

from ..functional import gcn_aggregate, partitioned_gcn_aggregate
from ..graph import adj_cache
from ..partition import PartitionedGraph


def _graph(adj):
    return adj if isinstance(adj, PartitionedGraph) else adj_cache.get(adj)


class Graph_conv_layer(nn.Module):
    """Y = Â·(X Wᵀ) + b (GCN/GCN.py:41-47); `fused_relu=True` also applies the ReLU that the
    model places after the layer."""

    def __init__(self, in_features, out_features, is_bias=True, **kwargs):
        super().__init__(**kwargs)
        self.in_features, self.out_features = in_features, out_features
        self.dense = nn.Linear(in_features, out_features, bias=False)
        self.register_parameter('bias', nn.Parameter(torch.zeros(out_features)) if is_bias else None)

    def forward(self, X_input, adj, fused_relu=False):
        if isinstance(adj, PartitionedGraph):
            return partitioned_gcn_aggregate(adj, self.dense(X_input), self.bias, relu=fused_relu)
        return gcn_aggregate(adj_cache.get(adj), self.dense(X_input), self.bias, relu=fused_relu)

    def __repr__(self):
        return f'{self.__class__.__name__} ({self.in_features} -> {self.out_features})'


class GCN_Model(nn.Module):
    """num_layers graph layers; ReLU + dropout after every layer but the last (GCN/GCN.py:5-27)."""

    def __init__(self, num_features, num_hidden, num_classes, num_layers, dropout, **kwargs):
        super().__init__(**kwargs)
        widths = [num_features] + [num_hidden] * (num_layers - 1) + [num_classes]
        self.gcn_blocks = nn.Sequential()
        for i in range(num_layers):
            # GCN.py:9-19: a single-layer model is `features -> hidden` followed by ReLU + dropout
            w_out = num_hidden if i == 0 else widths[i + 1]
            self.gcn_blocks.add_module(f'gcn{i}', Graph_conv_layer(widths[i], w_out))
            if i == 0 or i < num_layers - 1:
                self.gcn_blocks.add_module(f'relu{i}', nn.ReLU())
                self.gcn_blocks.add_module(f'dropout{i}', nn.Dropout(dropout))

    def forward(self, X, adj):
        graph = _graph(adj)
        blocks = list(self.gcn_blocks)
        i = 0
        while i < len(blocks):
            block = blocks[i]
            if block._get_name() == 'Graph_conv_layer':
                fuse = i + 1 < len(blocks) and type(blocks[i + 1]) is nn.ReLU
                X = block(X, graph, fused_relu=fuse)
                i += 2 if fuse else 1
            else:
                X = block(X)
                i += 1
        return X
