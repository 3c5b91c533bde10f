"""Drop-in for the de-duplicating GraphSAGE variant of the reference
(/root/reference GraphSAGE/GraphSAGE.py:7-61; batches built by GraphSAGE/data_utils.py:82-162).

Kept from the reference because callers and checkpoints depend on it: the class names
`SageLayer` / `GraphSAGE`, their constructor and forward signatures, and the state_dict keys
`sage_blocks.sage_layer{i}.weight.weight`, `dense.{weight,bias}`.

Re-designed for the device:
  * between layers the reference materialises `torch.embedding(feats, neigh_map)` as an
    `[n, k, F]` tensor and then means it (GraphSAGE.py:47-49 + graph_utils.py:6); here the id
    map goes straight into the fused gather-mean kernel (`functional.gather_reduce`), so that
    tensor never exists;
  * `cat([self, agg]) @ Wᵀ` (GraphSAGE.py:17-21) is computed as two products against the two
    column halves of the same weight, accumulated in place (`addmm`): no `[n, 2F]` concat copy;
  * the -1 padding of the maps (data_utils.py:105-116) is resolved once per layer into row
    selections, not re-derived per use;
  * `forward_sampled` takes batches built on the device (`functional.dedup_layer_nodes`): the
    outermost neighbours are reduced straight out of the feature table, so the collate's `[n0, k, F]`
    tensor and its host-to-device copy do not exist.
"""
import torch
from torch import nn

from ..functional import gather_reduce

_REDUCE = {'MEAN': 'mean', 'MAX': 'max'}


def _reduce_name(agg_func):
    if agg_func not in _REDUCE:  # graph_utils.py:9-11 prints a hint and re-raises
        print('请选择合适的聚合函数')
        raise ValueError(agg_func)
    return _REDUCE[agg_func]


class SageLayer(nn.Module):
    """relu(W·[self ‖ agg]) — or relu(W·agg) with gcn=True (GraphSAGE.py:7-21)."""

    def __init__(self, input_size, output_size, gcn=False, **kwargs):
        super().__init__(**kwargs)
        self.input_size, self.output_size, self.gcn = input_size, output_size, gcn
        fan_in = input_size if gcn else 2 * input_size
        self.weight = nn.Linear(fan_in, output_size, bias=False)

    def forward(self, self_feats, aggregate_feats):
        w = self.weight.weight  # [out, fan_in]
        if self.gcn:
            z = aggregate_feats @ w.t()
        else:
            d = self.input_size
            z = torch.addmm(self_feats @ w[:, :d].t(), aggregate_feats, w[:, d:].t())
        return torch.relu(z)


class GraphSAGE(nn.Module):
    def __init__(self, num_layers, input_size, out_size, gcn=False, agg_func='MEAN', Unsupervised=True, class_size=None,
                 **kwargs):
        super().__init__(**kwargs)
        self.num_layers, self.gcn, self.agg_func, self.Unsupervised = num_layers, gcn, agg_func, Unsupervised
        widths = [input_size] + [out_size] * num_layers
        self.sage_blocks = nn.Sequential()
        for i, (w_in, w_out) in enumerate(zip(widths[:-1], widths[1:])):
            self.sage_blocks.add_module(f'sage_layer{i}', SageLayer(w_in, w_out, gcn=gcn))
        if not Unsupervised:
            self.dense = nn.Linear(out_size, class_size)

    # -- one tower: (features of the outermost node set, its pre-gathered neighbours, per-layer maps)
    def _encode(self, self_feats, self_maps, neigh_feats, neigh_maps):
        reduce = _reduce_name(self.agg_func)
        n, k, width = neigh_feats.shape
        # outermost layer: the collate function already gathered [n, k, F] on the host
        # (data_utils.py:154-162); reduce it in place as an identity index block
        agg = gather_reduce(neigh_feats.reshape(n * k, width), None, n, k, reduce)

        def maps(i):
            keep_self, rows = self_maps[i], neigh_maps[i]
            return keep_self[keep_self != -1], rows[rows[:, 0] != -1]  # padded rows start with -1 (GraphSAGE.py:48-49)
        return self._layers(self_feats, agg, maps, reduce)

    # -- one tower of a DedupBatch: the outermost neighbours are gathered straight from the table
    def _encode_sampled(self, table, batch):
        reduce = _reduce_name(self.agg_func)
        ids = batch.outer_neighbors
        agg = gather_reduce(table, ids.reshape(-1), ids.shape[0], ids.shape[1], reduce)

        def maps(i):
            n = batch.counts[i + 1]
            return batch.center_map[i, :n], batch.neigh_map[i, :n]
        return self._layers(table.index_select(0, batch.nodes[0]), agg, maps, reduce)

    def _layers(self, self_feats, agg, maps, reduce):
        """The layer stack: maps(i) gives layer i's kept self rows and its [n, k] neighbour rows, both unpadded."""
        last = self.num_layers - 1
        for i, layer in enumerate(self.sage_blocks):
            h = layer(self_feats, agg)
            if i == last:
                return h
            keep_self, rows = maps(i)
            self_feats = h.index_select(0, keep_self)
            agg = gather_reduce(h, rows.reshape(-1), rows.shape[0], rows.shape[1], reduce)

    def _head(self, centers, others, contexts_negatives_shape):
        if others is None:
            # supervised (GraphSAGE.py:42-53): embeddings + optional class logits
            return centers, (None if self.Unsupervised else self.dense(centers))
        # skip-gram head (GraphSAGE.py:54-61): score every centre against its contexts / negatives
        others = others.reshape(*contexts_negatives_shape, -1)
        scores = torch.einsum('bd,bcd->bc', centers, others).unsqueeze(1)
        return centers, scores

    def forward(self, center_feats_data, center_nodes_map, center_neigh_feats_data, center_neigh_nodes_map,
                contexts_negatives_feats_data, contexts_negatives_nodes_map, contexts_negatives_neigh_feats_data,
                contexts_negatives_neigh_nodes_map, contexts_negatives_shape):
        centers = self._encode(center_feats_data, center_nodes_map, center_neigh_feats_data, center_neigh_nodes_map)
        others = None if contexts_negatives_feats_data is None else self._encode(
            contexts_negatives_feats_data, contexts_negatives_nodes_map, contexts_negatives_neigh_feats_data,
            contexts_negatives_neigh_nodes_map)
        return self._head(centers, others, contexts_negatives_shape)

    def forward_sampled(self, table, batch, cn_batch=None, cn_shape=None):
        """`forward` on minibatches built on the device by `functional.dedup_layer_nodes`: no `[n, k, F]` tensor.

        table: the feature table [N, F] on the device; pad it once with `functional.pad_table` (16-byte rows take
        the TMA gather; either layout gives the same bits).  batch: the centres' DedupBatch; cn_batch / cn_shape:
        the contexts and negatives of the unsupervised head and their [B, C] shape.  The self rows of the outermost
        layer are `table[S_0]`, its aggregate reduces the outer neighbours' rows straight out of the table, and the
        inner layers cut the maps at the batch's counts.  Returns what `forward` returns on the same batch gathered
        on the host (the kernels add in the same order on both paths)."""
        centers = self._encode_sampled(table, batch)
        others = None if cn_batch is None else self._encode_sampled(table, cn_batch)
        return self._head(centers, others, cn_shape)
