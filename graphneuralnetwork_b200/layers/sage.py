"""Drop-in GraphSAGE layers (class names, ctor signatures, parameter names and forward
signatures of /root/reference GraphSAGE_Pytorch/models/{Aggregator,SageGCN,GraphSage}.py and
the `Aggregator` function of GraphSAGE/graph_utils.py).

Two ways in:
  * the reference call surface — `NeighborAggregator.forward(neighbor_feature)` with the
    pre-gathered `[n_src, fanout, F]` tensor (Aggregator.py:18): the reduce over the fanout
    axis runs in the CUDA kernel on that tensor as an identity index block;
  * the fused fast path — `GraphSage.forward_sampled(table, blocks)`: the sampled node ids
    of `multihop_sampling` (sample_utils.py:20-35) index a feature table resident in HBM and
    the gather (data_utils.py:64) is fused into the reduce, so the `[n_src, fanout, F]`
    tensor is never materialised and only the ids cross PCIe.
"""
import torch
from torch import nn
import torch.nn.functional as F

from .. import _lib
from ..functional import (_padded_empty, gather_reduce, gather_reduce_multi_raw, gather_reduce_multi_split_raw,
                          pad_table)
from ..partition import ShardedTable


class SampledBlock:
    """Neighbour features given as (table, ids): rows `ids[i*fanout:(i+1)*fanout]` of `table`
    are the neighbours of source i (the src-major layout of sample_utils.py:16)."""

    def __init__(self, table: torch.Tensor, ids: torch.Tensor, fanout: int):
        self.table, self.ids, self.fanout = table, ids, int(fanout)
        self.n_src = ids.numel() // self.fanout


class NeighborAggregator(nn.Module):
    """reduce_k(neighbours)·W (+ b) — GraphSAGE_Pytorch/models/Aggregator.py:5-37.
    state_dict: `weight [in,out]` (+ `bias [out]` with use_bias)."""

    def __init__(self, input_dim, output_dim, use_bias=False, aggr_method="mean", **kwargs):
        super().__init__(**kwargs)
        self.input_dim, self.output_dim = input_dim, output_dim
        self.use_bias, self.aggr_method = use_bias, aggr_method
        self.weight = nn.Parameter(nn.init.xavier_uniform_(torch.empty(input_dim, output_dim)))
        if use_bias:
            self.bias = nn.Parameter(torch.zeros(output_dim))

    def aggregate(self, neighbor_feature):
        """The reduce over the fanout axis, on the device: a `SampledBlock` (ids into a resident
        table: gather fused into the reduce) or the reference's pre-gathered `[n_src, fanout, F]`
        tensor (Aggregator.py:18), walked as an identity index block."""
        if self.aggr_method not in ("mean", "sum", "max"):
            raise ValueError("Unknown aggr type, expected sum, max, or mean, but got {}".format(self.aggr_method))
        if isinstance(neighbor_feature, SampledBlock):
            b = neighbor_feature
            return gather_reduce(b.table, b.ids, b.n_src, b.fanout, self.aggr_method)
        n_src, fanout, feat = neighbor_feature.shape
        # `max`: the reference's `.max(dim=1)` returns a (values, indices) tuple and the
        # following matmul raises TypeError (Aggregator.py:24,29); we implement `.values`.
        return gather_reduce(neighbor_feature.reshape(n_src * fanout, feat), None, n_src, fanout, self.aggr_method)

    def forward(self, neighbor_feature):
        # a 2-D tensor is already the aggregate (GraphSage.forward_sampled's fused multi-hop launch)
        pooled = neighbor_feature if torch.is_tensor(neighbor_feature) and neighbor_feature.dim() == 2 \
            else self.aggregate(neighbor_feature)
        return torch.addmm(self.bias, pooled, self.weight) if self.use_bias else torch.mm(pooled, self.weight)

    def extra_repr(self):
        return f'in_features={self.input_dim}, out_features={self.output_dim}, aggr_method={self.aggr_method}'


class SageGCN(nn.Module):
    """activation(src·W_self  (+ | ‖)  agg(neigh)·W_agg) — GraphSAGE_Pytorch/models/SageGCN.py:8-36.
    state_dict: `weight [in,hidden]`, `aggregator.weight [in,hidden]` (+ `aggregator.bias`)."""

    def __init__(self, input_dim, hidden_dim, activation=F.relu, aggr_neighbor_method="mean", aggr_hidden_method="sum",
                 **kwargs):
        super().__init__(**kwargs)
        assert aggr_neighbor_method in ["mean", "sum", "max"]
        assert aggr_hidden_method in ["sum", "concat"]
        self.input_dim, self.hidden_dim = input_dim, hidden_dim
        self.aggr_neighbor_method, self.aggr_hidden_method = aggr_neighbor_method, aggr_hidden_method
        self.activation = activation
        self.aggregator = NeighborAggregator(input_dim, hidden_dim, aggr_method=aggr_neighbor_method)
        self.weight = nn.Parameter(torch.empty(input_dim, hidden_dim))
        nn.init.xavier_uniform_(self.weight)

    def forward(self, src_node_features, neighbor_node_features):
        agg = self.aggregator
        # the aggregate is either handed in ([n_src, F], from the fused multi-hop launch) or reduced here
        pooled = neighbor_node_features if torch.is_tensor(neighbor_node_features) and neighbor_node_features.dim() == 2 \
            else agg.aggregate(neighbor_node_features)
        if self.aggr_hidden_method == "sum":
            # both products accumulate into one buffer: no separate add (SageGCN.py:26-27)
            hidden = torch.addmm(torch.mm(src_node_features, self.weight), pooled, agg.weight)
            if agg.use_bias:
                hidden = hidden + agg.bias
        elif self.aggr_hidden_method == "concat":
            hidden = torch.cat([torch.mm(src_node_features, self.weight), agg(pooled)], dim=1)  # SageGCN.py:28-29
        else:
            raise ValueError("Expected sum or concat, got {}".format(self.aggr_hidden_method))
        return self.activation(hidden) if self.activation else hidden

    def extra_repr(self):
        width = self.hidden_dim * (1 if self.aggr_hidden_method == "sum" else 2)
        return f'in_features={self.input_dim}, out_features={width}, aggr_hidden_method={self.aggr_hidden_method}'


class GraphSage(nn.Module):
    """GraphSAGE_Pytorch/models/GraphSage.py:6-33.  state_dict: `gcn.{l}.weight`, `gcn.{l}.aggregator.weight`."""

    def __init__(self, input_dim, hidden_dim, num_neighbors_list):
        super().__init__()
        self.input_dim, self.hidden_dim = input_dim, hidden_dim
        self.num_neighbors_list = num_neighbors_list
        self.num_layers = len(num_neighbors_list)
        widths = [input_dim] + list(hidden_dim)
        last = len(hidden_dim) - 1
        # every layer but the last ends in ReLU (GraphSage.py:13-16)
        self.gcn = nn.ModuleList(SageGCN(widths[l], widths[l + 1], **({"activation": None} if l == last else {}))
                                 for l in range(len(hidden_dim)))

    def _upper_layers(self, hidden):
        """Layers 1..L-1 (GraphSage.py:21-29): layer l turns the states of hops 0..L-l into the states of
        hops 0..L-l-1; the neighbours of hop h are the contiguous rows of hop h+1, reduced as an
        identity index block (no gather)."""
        for l in range(1, self.num_layers):
            layer = self.gcn[l]
            hidden = [layer(hidden[hop], hidden[hop + 1].view(hidden[hop].shape[0], self.num_neighbors_list[hop], -1))
                      for hop in range(self.num_layers - l)]
        return hidden[0]

    def forward(self, node_features_list):
        """Reference call surface (GraphSage.py:18-30): pre-gathered feature tensors per hop,
        `node_features_list[h]` = [B·f1·…·fh, F]."""
        layer0, fan = self.gcn[0], self.num_neighbors_list
        hidden = [layer0(node_features_list[hop],
                         node_features_list[hop + 1].view(node_features_list[hop].shape[0], fan[hop], -1))
                  for hop in range(self.num_layers)]
        return self._upper_layers(hidden)

    def forward_sampled(self, table, node_id_blocks):
        """Fused path: `table` [N,F] resident on the device (ideally `pad_table`-aligned),
        `node_id_blocks` = the id lists `multihop_sampling` returns (lengths B, B·f1, B·f1·f2, …)
        as int32/int64 device tensors.  Same arithmetic as `forward` on
        `[table[ids] for ids in node_id_blocks]`, without materialising the gathers of the
        outermost hop: layer 0 reads neighbours straight from the table.
        `table` may be a `partition.ShardedTable` (rows spread over the GPUs of a node): the
        logits and every weight gradient are then bit-identical to those over the concatenated
        tensor table (but for the sign of zero noted in `_layer0_sharded`)."""
        L, fan, layer0 = self.num_layers, self.num_neighbors_list, self.gcn[0]
        assert len(node_id_blocks) == L + 1
        fused = (not (torch.is_grad_enabled() and table.requires_grad)) and L <= 4 \
            and layer0.aggr_neighbor_method in ("mean", "sum", "max")
        no_grad = not (torch.is_grad_enabled() and (table.requires_grad or layer0.weight.requires_grad))
        if fused and no_grad and 2 * L <= 4 and layer0.aggr_hidden_method == "sum" and not layer0.aggregator.use_bias \
                and table.dtype == torch.float32:
            return self._upper_layers(self._layer0_one_launch_one_gemm(table, node_id_blocks))
        if isinstance(table, ShardedTable):
            return self._upper_layers(self._layer0_sharded(table, node_id_blocks))
        if fused:
            # every hop of layer 0 aggregates from the same table: ONE launch for all of them
            pooled = gather_reduce_multi_raw(table, [(node_id_blocks[hop + 1], node_id_blocks[hop].numel(), fan[hop])
                                                     for hop in range(L)], layer0.aggr_neighbor_method)
        else:
            pooled = [SampledBlock(table, node_id_blocks[hop + 1], fan[hop]) for hop in range(L)]
        hidden = [layer0(table.index_select(0, node_id_blocks[hop].to(torch.int64)), pooled[hop]) for hop in range(L)]
        return self._upper_layers(hidden)

    def _layer0_sharded(self, table, node_id_blocks):
        """Layer 0 over a ShardedTable outside the one-launch inference form (training, L > 2, ...): the neighbour
        reduce of every hop and, as fanout-1 blocks, the hop's own rows (what `table.index_select` gives a tensor
        table: an exact copy, but -0.0 becomes +0.0 under mean/sum) come from the shards, four blocks per launch.
        The own rows land in a contiguous [n, F] buffer and the reduces in padded ones, the shapes and strides the
        tensor path hands the products, so both paths run the same GEMMs."""
        L, fan, layer0 = self.num_layers, self.num_neighbors_list, self.gcn[0]
        F = table.shape[1]
        n_hop = [node_id_blocks[hop].numel() for hop in range(L)]
        blocks = [(node_id_blocks[hop + 1], n_hop[hop], fan[hop]) for hop in range(L)] + \
                 [(node_id_blocks[hop], n_hop[hop], 1) for hop in range(L)]
        outs = [_padded_empty(n, F, table.dtype, table.device) for n in n_hop] + \
               [torch.empty((n, F), dtype=table.dtype, device=table.device) for n in n_hop]
        for i in range(0, len(blocks), 4):
            gather_reduce_multi_raw(table, blocks[i:i + 4], layer0.aggr_neighbor_method, outs=outs[i:i + 4])
        return [layer0(outs[L + hop], outs[hop]) for hop in range(L)]

    def _layer0_one_launch_one_gemm(self, table, node_id_blocks):
        """Inference form of layer 0 for all hops at once (SageGCN.py:23-27 on every hop of GraphSage.py:24-27):
        ONE gather launch writes, for every source of every hop, its own feature row (a fanout-1 block — the
        reference's `src_node_features` gather, data_utils.py:64) and the reduce of its sampled neighbours side
        by side into one `[Σ n_hop, 2·ld]` operand, and ONE `[self ‖ pooled]·[W_self ; W_agg]` product (K = 2·F)
        replaces the two products + add per hop.  Same arithmetic, one accumulation order change: the two
        K-sums are one K-sum (fp32 re-association only)."""
        L, fan, layer0 = self.num_layers, self.num_neighbors_list, self.gcn[0]
        F_in, H = layer0.input_dim, layer0.hidden_dim
        ld = (F_in + 3) // 4 * 4
        n_hop = [node_id_blocks[hop].numel() for hop in range(L)]
        total = sum(n_hop)
        if getattr(self, "tensor_core_gemm", True) and layer0.aggr_neighbor_method in ("mean", "sum") \
                and table.stride(0) * 4 % 16 == 0 and F_in * 4 >= 256:
            try:
                return self._layer0_split_gemm(table, node_id_blocks, ld, n_hop, total)
            except _lib.GnnError:  # off the TMA path (unaligned table): the fp32 product below
                self.tensor_core_gemm = False
        key = (total, table.device)
        buf = getattr(self, "_l0_buf", None)
        if buf is None or buf[0] != key:
            # pad columns stay zero for the lifetime of the buffer: the gather writes F_in columns per row only
            Z = torch.zeros((total, 2 * ld), dtype=torch.float32, device=table.device)
            Wc = torch.zeros((2 * ld, H), dtype=torch.float32, device=table.device)
            self._l0_buf = buf = (key, Z, Wc)
        _, Z, Wc = buf
        Wc[:F_in].copy_(layer0.weight)
        Wc[ld:ld + F_in].copy_(layer0.aggregator.weight)
        blocks, outs, row = [], [], 0
        for hop in range(L):
            n = n_hop[hop]
            blocks += [(node_id_blocks[hop + 1], n, fan[hop]), (node_id_blocks[hop], n, 1)]
            outs += [Z[row:row + n, ld:ld + F_in], Z[row:row + n, :F_in]]
            row += n
        # longest block first: the short ones ride in its shadow
        order = sorted(range(len(blocks)), key=lambda i: -blocks[i][1] * blocks[i][2])
        gather_reduce_multi_raw(table, [blocks[i] for i in order], layer0.aggr_neighbor_method,
                                outs=[outs[i] for i in order])
        hidden = torch.mm(Z, Wc)
        if layer0.activation:
            hidden = layer0.activation(hidden)
        out, row = [], 0
        for n in n_hop:
            out.append(hidden[row:row + n])
            row += n
        return out

    def _table_fits_fp16(self, table):
        """max|table| < 3e4 (an aggregate of rows never exceeds it): cached per table tensor (one host read)."""
        if isinstance(table, ShardedTable):  # read-only, its max computed once at construction
            return table.abs_max < 3.0e4
        key = (table.data_ptr(), table._version, tuple(table.shape))
        hit = getattr(self, "_fp16_ok", None)
        if hit is None or hit[0] != key:
            self._fp16_ok = hit = (key, bool((table.abs().max() < 3.0e4).item()))
        return hit[1]

    def _weight_planes(self, ld, device):
        """fp16 hi / lo planes of `[W_self ; W_agg]` (rows padded to ld each), recomputed only when a weight changed
        (`_version` / storage of the two parameters): an inference loop — and a captured graph, whose runner calls
        this before every replay — pays the five small launches of the split once, not per minibatch."""
        layer0 = self.gcn[0]
        w, wa = layer0.weight, layer0.aggregator.weight
        F_in, H = layer0.input_dim, layer0.hidden_dim
        geom = (int(ld), torch.device(device))
        ver = (w._version, wa._version, w.data_ptr(), wa.data_ptr())
        planes = getattr(self, "_l0_planes", None)
        if planes is None or planes["geom"] != geom:
            planes = self._l0_planes = {
                "geom": geom, "ver": None,
                "Wc": torch.zeros((2 * ld, H), dtype=torch.float32, device=device),
                "hi": torch.zeros((2 * ld, H), dtype=torch.float16, device=device),
                "lo": torch.zeros((2 * ld, H), dtype=torch.float16, device=device)}
        if planes["ver"] != ver:
            Wc, W_hi, W_lo = planes["Wc"], planes["hi"], planes["lo"]
            with torch.no_grad():
                Wc[:F_in].copy_(w)
                Wc[ld:ld + F_in].copy_(wa)
                W_hi.copy_(Wc)
                W_lo.copy_(Wc - W_hi.float())
            planes["ver"] = ver
        return planes["hi"], planes["lo"]

    def _layer0_split_gemm(self, table, node_id_blocks, ld, n_hop, total):
        """Layer 0 with the fp32 `[self ‖ pooled]·[W_self ; W_agg]` product (K = 2·F, the largest single cost of the
        minibatch after the gather: 26,624 x 1,208 x 128 on the Reddit-shaped config runs 0.17 ms on the fp32 SIMT
        pipes) carried by the fp16 tensor cores at fp32-level accuracy: the gather's row flush writes every operand
        value as hi = fp16(x), lo = fp16(x - hi) (22 mantissa bits, the same bytes as fp32), the weights are split
        the same way, and   Z·W ~= Z_hi·W_hi + Z_lo·W_hi + Z_hi·W_lo   with fp32 accumulation — the dropped
        Z_lo·W_lo term is below 2^-22 relative.  Still a torch matmul (a library GEMM outside the hot path), on
        operands the gather kernel laid out for it.  Needs |table| within fp16 range (checked once per table)."""
        if not self._table_fits_fp16(table):
            raise _lib.GnnError("table exceeds the fp16 range: fp32 product")
        L, fan, layer0 = self.num_layers, self.num_neighbors_list, self.gcn[0]
        F_in, H = layer0.input_dim, layer0.hidden_dim
        key = (total, table.device)
        buf = getattr(self, "_l0_split", None)
        if buf is None or buf[0] != key:
            # row = [hi: self | pooled][lo: self | pooled]; pad columns stay zero for the buffer's lifetime
            Zs = torch.zeros((total, 4 * ld), dtype=torch.float16, device=table.device)
            self._l0_split = buf = (key, Zs)
        _, Zs = buf
        W_hi, W_lo = self._weight_planes(ld, table.device)
        blocks, outs, row = [], [], 0
        for hop in range(L):
            n = n_hop[hop]
            blocks += [(node_id_blocks[hop + 1], n, fan[hop]), (node_id_blocks[hop], n, 1)]
            outs += [Zs[row:row + n, ld:ld + F_in], Zs[row:row + n, :F_in]]
            row += n
        order = sorted(range(len(blocks)), key=lambda i: -blocks[i][1] * blocks[i][2])
        gather_reduce_multi_split_raw(table, [blocks[i] for i in order], layer0.aggr_neighbor_method,
                                      [outs[i] for i in order], lo_off=2 * ld)
        # three products of K = 2·ld each, added in fp32 by torch: the tensor cores' fp32 accumulation truncates, so
        # its error grows with K — one concatenated K = 4·ld product measured 5e-6 against float64, this form 2e-6
        # (the fp32 SIMT product: 0.4-1.7e-6; tools/diag_split_gemm.py)
        Z_hi, Z_lo = Zs[:, :2 * ld], Zs[:, 2 * ld:]
        hidden = torch.mm(Z_hi, W_hi, out_dtype=torch.float32)
        if getattr(self, "_addmm_out_dtype", True):
            try:  # the two fp32 adds ride in the GEMM epilogues (beta = 1) instead of two elementwise launches
                hidden = torch.addmm(hidden, Z_lo, W_hi, out_dtype=torch.float32)
                hidden = torch.addmm(hidden, Z_hi, W_lo, out_dtype=torch.float32)
            except (RuntimeError, NotImplementedError):  # settled in the warm-up call, before any graph capture
                self._addmm_out_dtype = False
                hidden = torch.mm(Z_hi, W_hi, out_dtype=torch.float32)
        if not getattr(self, "_addmm_out_dtype", True):
            hidden += torch.mm(Z_lo, W_hi, out_dtype=torch.float32)
            hidden += torch.mm(Z_hi, W_lo, out_dtype=torch.float32)
        if layer0.activation:
            hidden = layer0.activation(hidden)
        out, row = [], 0
        for n in n_hop:
            out.append(hidden[row:row + n])
            row += n
        return out

    def extra_repr(self):
        return 'in_features={}, num_neighbors_list={}'.format(self.input_dim, self.num_neighbors_list)


def Aggregator(neigh_feat, agg_func='MEAN'):
    """GraphSAGE/graph_utils.py:4-11.  'MEAN' -> fused mean over dim 1.  The reference's 'MAX'
    is `torch.argmax` (an int64 index tensor, a bug, graph_utils.py:8); we return the max
    VALUES and say so in DESIGN.md."""
    if agg_func not in ('MEAN', 'MAX'):
        print('请选择合适的聚合函数')
        raise ValueError(agg_func)
    n, k, feat = neigh_feat.shape
    return gather_reduce(neigh_feat.reshape(n * k, feat), None, n, k, 'mean' if agg_func == 'MEAN' else 'max')


def gather_mean(feats, index_map):
    """`torch.mean(torch.embedding(feats, index_map), dim=1)` fused
    (GraphSAGE/GraphSAGE.py:47-49 followed by graph_utils.py:6): `index_map` is the `[n,k]`
    int64 map of GraphSAGE/data_utils.py:105-116 with its -1-padded rows already filtered
    (GraphSAGE.py:48-49 keeps rows whose column 0 is not -1)."""
    n, k = index_map.shape
    return gather_reduce(feats, index_map.reshape(-1), n, k, 'mean')


class CapturedGraphSage:
    """Inference runner for the fused path: `GraphSage.forward_sampled` captured once into a
    CUDA graph (the aggregation kernels of libgnn_b200.so and the torch matmuls alike), then
    replayed per minibatch.  Per call only the sampled ids cross PCIe (pinned host -> static
    device buffers) and the logits come back; launch overhead is one graph launch.

        runner = CapturedGraphSage(model, table, batch=1024)
        logits_host = runner(host_id_blocks)        # list of pinned int32/int64 id tensors
    """

    def __init__(self, model: GraphSage, table: torch.Tensor, batch: int, id_dtype=torch.int32, adjacency=None,
                 seed: int = 0):
        """adjacency (a CSRGraph over the table's nodes, optional): sample the neighbour blocks on the
        device inside the captured graph (`functional.multihop_sampling`, a fresh draw per replay);
        then only the batch's node ids cross PCIe."""
        from .. import _lib
        from ..functional import multihop_sampling
        self.model, self.table, self.adjacency = model, table, adjacency
        dev = table.device
        sizes = [batch]
        for f in model.num_neighbors_list:
            sizes.append(sizes[-1] * f)
        self.ids = [torch.zeros(s, dtype=id_dtype, device=dev) for s in sizes]
        self.replays = torch.zeros(1, dtype=torch.int64, device=dev)  # per-replay RNG stream of the sampler
        self.stream = torch.cuda.Stream(device=dev)
        self.graph = torch.cuda.CUDAGraph()
        self.kernel_launches_per_replay = 0

        def body():
            if adjacency is not None:
                self.replays.add_(1)
                blocks = multihop_sampling(adjacency, self.ids[0], model.num_neighbors_list, seed, id_dtype,
                                           seed_offset=self.replays)
                for dst, src in zip(self.ids[1:], blocks[1:]):
                    dst.copy_(src)
            return model.forward_sampled(table, self.ids)

        with torch.no_grad(), torch.cuda.stream(self.stream):
            for _ in range(2):  # warm-up outside capture (allocator, cuBLAS handles, smem attributes)
                body()
            self.stream.synchronize()
            before = _lib.launch_count()
            with torch.cuda.graph(self.graph, stream=self.stream):
                self.logits = body()
            self.kernel_launches_per_replay = _lib.launch_count() - before
        # two-slot pipeline around the captured graph: ids of minibatch i+1 cross PCIe while minibatch i
        # computes, logits of minibatch i-1 travel back meanwhile (submit / collect below)
        n_in = 1 if adjacency is not None else len(self.ids)
        self._n_in = n_in
        self._h2d, self._d2h = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        self._slots = []
        for _ in range(2):
            self._slots.append({
                "stage": [torch.zeros_like(t) for t in self.ids[:n_in]],
                "out": torch.empty_like(self.logits),
                "host": torch.empty(self.logits.shape, dtype=self.logits.dtype).pin_memory(),
                "ev_in": torch.cuda.Event(), "ev_free": torch.cuda.Event(), "ev_done": torch.cuda.Event(),
                "ev_out": torch.cuda.Event(),
            })
        self._submitted = self._collected = 0
        self.logits_host = self._slots[0]["host"]

    @torch.no_grad()
    def submit(self, host_id_blocks) -> int:
        """Queue one minibatch (pinned id tensors: every hop's block, or only the batch's node ids when
        the runner samples on the device).  At most two minibatches may be in flight: call `collect`
        before the third `submit`.  Returns the ticket number."""
        if self._submitted - self._collected >= 2:
            raise RuntimeError("CapturedGraphSage: two minibatches already in flight; collect() first")
        if torch.is_tensor(host_id_blocks):
            host_id_blocks = [host_id_blocks]
        slot = self._slots[self._submitted & 1]
        with torch.cuda.stream(self._h2d):
            self._h2d.wait_event(slot["ev_free"])            # the staging buffers were consumed
            for dst, src in zip(slot["stage"], host_id_blocks[:self._n_in]):
                dst.copy_(src, non_blocking=True)            # H2D: this minibatch's ids
            slot["ev_in"].record(self._h2d)
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(slot["ev_in"])
            for dst, src in zip(self.ids[:self._n_in], slot["stage"]):
                dst.copy_(src)                               # device copy into the graph's static inputs
            slot["ev_free"].record(self.stream)
            self._refresh_model_state()                      # weight planes the graph reads, if a weight changed
            self.graph.replay()
            slot["out"].copy_(self.logits)
            slot["ev_done"].record(self.stream)
        with torch.cuda.stream(self._d2h):
            self._d2h.wait_event(slot["ev_done"])
            slot["host"].copy_(slot["out"], non_blocking=True)  # D2H: the result
            slot["ev_out"].record(self._d2h)
        self._submitted += 1
        return self._submitted - 1

    def _refresh_model_state(self):
        """Out-of-graph state the captured forward reads: the fp16 weight planes of the layer-0 product follow the
        parameters' versions (an optimiser step or load_state_dict between replays is picked up here)."""
        planes = getattr(self.model, "_l0_planes", None)
        if planes is not None:
            self.model._weight_planes(*planes["geom"])

    def collect(self) -> torch.Tensor:
        """Logits of the oldest minibatch in flight (pinned host tensor, valid until two more submits)."""
        if self._collected >= self._submitted:
            raise RuntimeError("CapturedGraphSage: nothing in flight")
        slot = self._slots[self._collected & 1]
        slot["ev_out"].synchronize()
        self._collected += 1
        self.logits_host = slot["host"]
        return slot["host"]

    def __call__(self, host_id_blocks):
        """Synchronous form: submit one minibatch and wait for its logits."""
        self.submit(host_id_blocks)
        return self.collect()
