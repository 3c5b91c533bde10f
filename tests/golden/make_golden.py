"""Generate the golden fixtures in tests/golden/*.npz from the UNMODIFIED reference.

Run with a reference checkout (kaddly/GraphNeuralNetwork):
    GNN_REFERENCE_ROOT=<checkout> python tests/golden/make_golden.py
The reference modules are imported through oracle/ref_loader.py and driven with seeded
synthetic inputs; inputs that are cheap to regenerate are stored as seeds + a checksum,
everything else (weights, index blocks, outputs, gradients) is stored verbatim.  The
fixtures pin the tests wherever the reference is absent.
"""
import hashlib
import os
import random
import sys

import numpy as np
import scipy.sparse as sp
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_loader as R  # noqa: E402
from graphneuralnetwork_b200 import synthetic as S  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def params_np(model):
    return {k: v.detach().numpy().copy() for k, v in model.state_dict().items()}


def grads_np(model):
    return {"grad." + k: p.grad.detach().numpy().copy() for k, p in model.named_parameters() if p.grad is not None}


def save(name, **arrays):
    path = os.path.join(OUT, name)
    np.savez_compressed(path, **arrays)
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB, {len(arrays)} arrays")


def make_gcn():
    gcn_mod, du = R.gcn()
    n = S.CORA["n"]
    edges = S.cora_like_edges(seed=0)
    # the reference's own pipeline: preprocess_data:35, load_cora:78, sparse_mx_to_torch_sparse_tensor:63-70
    adj = sp.coo_matrix((np.ones(edges.shape[0]), (edges[:, 0], edges[:, 1])), shape=(n, n), dtype=np.float32)
    adj = adj + adj.T.multiply(adj.T > adj) - adj.multiply(adj.T > adj)
    adj_n = du.normalize_adj(adj + sp.eye(adj.shape[0]))
    adj_t = du.sparse_mx_to_torch_sparse_tensor(adj_n)
    idx = adj_t._indices().numpy()
    val = adj_t._values().numpy()
    X = S.row_normalised_features(n, S.CORA["feats"], seed=1)
    labels = np.random.default_rng(2).integers(0, S.CORA["classes"], size=n)
    torch.manual_seed(0)
    model = gcn_mod.GCN_Model(S.CORA["feats"], S.CORA["hidden"], S.CORA["classes"], 2, 0.5)
    model.eval()
    Xt = torch.from_numpy(X)
    out = model(Xt, adj_t)
    idx_train = torch.arange(140)
    loss = torch.nn.functional.cross_entropy(out[idx_train], torch.from_numpy(labels)[idx_train])
    loss.backward()
    # one isolated layer, for the spmm check alone
    layer_out = model.gcn_blocks.gcn0(Xt, adj_t).detach().numpy()
    save("gcn_cora.npz", edges=edges, coo_row=idx[0].astype(np.int32), coo_col=idx[1].astype(np.int32), coo_val=val,
         x_seed=np.int64(1), x_sha=np.array(sha(X)), labels=labels.astype(np.int64), out=out.detach().numpy(),
         layer0_out=layer_out, loss=np.float64(loss.item()), **params_np(model), **grads_np(model))


def _gat_adj(n, pairs, seed):
    """GAT/data_utils.py:73-85: same normalisation as GCN, kept dense fp32."""
    _, du = R.gcn()
    edges = S.cora_like_edges(n=n, pairs=pairs, seed=seed)
    adj = sp.coo_matrix((np.ones(edges.shape[0]), (edges[:, 0], edges[:, 1])), shape=(n, n), dtype=np.float32)
    adj = adj + adj.T.multiply(adj.T > adj) - adj.multiply(adj.T > adj)
    adj = du.normalize_adj(adj + sp.eye(n))
    return edges, np.asarray(adj.todense(), dtype=np.float32)


def make_gat_small():
    gat_mod, _ = R.gat_models()
    n, nfeat, nhid, nheads, nclass = 300, 50, 8, 8, 7
    edges, adj = _gat_adj(n, 700, seed=3)
    adj[17, :] = 0  # one isolated row: the reference soft-maxes it to the uniform mean (layers.py:28-30)
    X = S.row_normalised_features(n, nfeat, seed=4)
    labels = np.random.default_rng(5).integers(0, nclass, size=n)
    out = {}
    for kind, cls in (("dense", gat_mod.GAT), ("sparse", gat_mod.SpGAT)):
        torch.manual_seed(1)
        model = cls(nfeat, nhid, nclass, 0.0, 0.2, nheads)  # dropout 0: train == eval, grads comparable
        model.train()
        a = torch.from_numpy(adj if kind == "dense" else np.where(np.arange(n)[:, None] == 17, np.eye(n, dtype=np.float32)[17], adj))
        o = model(torch.from_numpy(X), a)
        loss = torch.nn.functional.cross_entropy(o, torch.from_numpy(labels))
        loss.backward()
        out.update({f"{kind}.out": o.detach().numpy(), f"{kind}.loss": np.float64(loss.item())})
        out.update({f"{kind}.{k}": v for k, v in params_np(model).items()})
        out.update({f"{kind}.{k}": v for k, v in grads_np(model).items()})
    save("gat_small.npz", edges=edges, adj=adj, X=X, labels=labels.astype(np.int64), isolated_row=np.int64(17), **out)


def make_gat_cora():
    gat_mod, _ = R.gat_models()
    n = S.CORA["n"]
    edges, adj = _gat_adj(n, S.CORA["undirected_pairs"], seed=0)
    X = S.row_normalised_features(n, S.CORA["feats"], seed=1)
    torch.manual_seed(2)
    model = gat_mod.GAT(S.CORA["feats"], 8, S.CORA["classes"], 0.6, 0.2, 8)
    model.eval()
    with torch.no_grad():
        out = model(torch.from_numpy(X), torch.from_numpy(adj))
    save("gat_cora.npz", edges=edges, adj_sha=np.array(sha(adj)), x_seed=np.int64(1), x_sha=np.array(sha(X)),
         out=out.numpy(), **params_np(model))


def make_sage():
    ref = R.sage_pytorch()
    n, feat, hidden, fan, B = 500, 602, [128, 41], [5, 3], 32
    adj_lists = S.adjacency_lists(n, 8, seed=6)
    table = np.random.default_rng(7).standard_normal((n, feat), dtype=np.float32)
    random.seed(0)
    src = list(range(40, 40 + B))
    blocks = ref["sample_utils"].multihop_sampling(src, fan, adj_lists)
    feats = [torch.from_numpy(table[np.asarray(b, dtype=np.int64)]) for b in blocks]
    labels = np.random.default_rng(8).integers(0, hidden[-1], size=B)
    torch.manual_seed(3)
    model = ref["GraphSage"].GraphSage(feat, hidden, fan)
    model.train()
    out = model(feats)
    loss = torch.nn.functional.cross_entropy(out, torch.from_numpy(labels))
    loss.backward()
    extra = {}
    for method in ("mean", "sum"):
        agg = ref["Aggregator"].NeighborAggregator(feat, 16, aggr_method=method)
        with torch.no_grad():
            agg.weight.copy_(torch.eye(feat)[:, :16])
            neigh = feats[1].view(B, fan[0], -1)
            extra[f"agg.{method}"] = agg(neigh).numpy()  # == reduce(neigh)[:, :16]
    adj_flat = np.concatenate([np.asarray(sorted(adj_lists[i]), dtype=np.int32) for i in range(n)])
    adj_ptr = np.cumsum([0] + [len(adj_lists[i]) for i in range(n)]).astype(np.int64)
    save("sage_small.npz", table_seed=np.int64(7), table_sha=np.array(sha(table)), adj_ptr=adj_ptr, adj_flat=adj_flat,
         block0=np.asarray(blocks[0], np.int64), block1=np.asarray(blocks[1], np.int64),
         block2=np.asarray(blocks[2], np.int64), labels=labels.astype(np.int64), out=out.detach().numpy(),
         loss=np.float64(loss.item()), **params_np(model), **grads_np(model), **extra)


def make_sage_v2():
    ref = R.sage_v2()
    n, feat, out_size, B, k, L = 300, 64, 32, 8, 4, 2
    adj_lists = S.adjacency_lists(n, 6, seed=9)
    table = np.random.default_rng(10).standard_normal((n, feat), dtype=np.float32)
    random.seed(1)
    collate = ref["data_utils"].collate_fn(adj_lists, table.tolist(), L, k, False, False)
    data = [(i, int(i % 3)) for i in range(20, 20 + B)]
    (center_feats, center_map, neigh_feats, neigh_map), labels = collate(data)
    torch.manual_seed(4)
    model = ref["GraphSAGE"].GraphSAGE(L, feat, out_size, gcn=False, agg_func='MEAN', Unsupervised=False, class_size=3)
    model.train()
    feats_out, classes = model(center_feats, center_map, neigh_feats, neigh_map, None, None, None, None, None)
    loss = torch.nn.functional.cross_entropy(classes, labels)
    loss.backward()
    save("sage_v2_small.npz", center_feats=center_feats.numpy(), center_map=center_map.numpy(),
         neigh_feats=neigh_feats.numpy(), neigh_map=neigh_map.numpy(), labels=labels.numpy(),
         feats_out=feats_out.detach().numpy(), classes=classes.detach().numpy(), loss=np.float64(loss.item()),
         **params_np(model), **grads_np(model))


def make_han():
    ref = R.han()
    n, fin, M, heads, hid, ncls = 150, 40, 3, [8], 8, 3
    gs = [S.symmetric_mask(n, t, seed=11 + i) for i, t in enumerate((400, 6000, 1500))]
    X = np.random.default_rng(14).standard_normal((n, fin), dtype=np.float32)
    labels = np.random.default_rng(15).integers(0, ncls, size=n)
    torch.manual_seed(5)
    model = ref["HAN"].HANModel(M, fin, hid, ncls, heads, 0.0)
    model.train()
    out = model([torch.from_numpy(g) for g in gs], torch.from_numpy(X))
    loss = torch.nn.functional.cross_entropy(out, torch.from_numpy(labels))
    loss.backward()
    packed = np.stack([np.packbits(g.astype(np.uint8), axis=1) for g in gs])
    save("han_small.npz", masks_packed=packed, n=np.int64(n), X=X, labels=labels.astype(np.int64),
         out=out.detach().numpy(), loss=np.float64(loss.item()), **params_np(model), **grads_np(model))


def make_gatne():
    """GATNE per-edge-type neighbour aggregation (SURVEY.md §8f rank 3): both reference variants, with
    learned embeddings (GATNE-T) and with node features (GATNE-I), forward + gradients."""
    ref_pt, ref_v1 = R.gatne()
    N, T, K, B, E, U, A, Fd = 300, 3, 10, 64, 32, 10, 20, 24
    rng = np.random.default_rng(21)
    inputs = torch.from_numpy(rng.integers(0, N, B))
    types = torch.from_numpy(rng.integers(0, T, B))
    neigh = torch.from_numpy(rng.integers(0, N, (B, T, K)))
    feats = torch.from_numpy(rng.standard_normal((N, Fd)).astype(np.float32))
    target = torch.from_numpy(rng.standard_normal((B, E)).astype(np.float32))
    out = {"inputs": inputs.numpy(), "types": types.numpy(), "neigh": neigh.numpy(), "features": feats.numpy(),
           "target": target.numpy()}
    for tag, ctor in (("pt_t_sum", lambda: ref_pt.GraphEncoder(N, E, U, T, A, None, agg_func="SUM")),
                      ("pt_t_mean", lambda: ref_pt.GraphEncoder(N, E, U, T, A, None, agg_func="MEAN")),
                      ("pt_i_sum", lambda: ref_pt.GraphEncoder(N, E, U, T, A, feats, agg_func="SUM")),
                      ("v1_t", lambda: ref_v1.GATNEModel(N, E, U, T, A, None)),
                      ("v1_i", lambda: ref_v1.GATNEModel(N, E, U, T, A, feats))):
        torch.manual_seed(7)
        model = ctor()
        emb = model(inputs, types, neigh)
        loss = ((emb - target) ** 2).sum()
        loss.backward()
        out[f"{tag}.out"] = emb.detach().numpy()
        out[f"{tag}.loss"] = np.float64(loss.item())
        out.update({f"{tag}.{k}": v for k, v in params_np(model).items()})
        out.update({f"{tag}.{k}": v for k, v in grads_np(model).items()})
    save("gatne_small.npz", **out)


def make_special_spmm():
    """GAT/models/layers.py:43-64 SpecialSpmmFunction on an UNSORTED COO pattern with one duplicated
    entry: output, gradient w.r.t. the values (the edge-gradient SDDMM contract) and w.r.t. b."""
    layers = R.gat_layers()
    rng = np.random.default_rng(31)
    n, m, F, nnz = 90, 90, 24, 900  # square: the reference indexes its dense gradient with row*N+col (layers.py:60)
    rows, cols = rng.integers(0, n, nnz), rng.integers(0, m, nnz)
    rows[-1], cols[-1] = rows[0], cols[0]  # a duplicate: two separate values on the same position
    indices = torch.from_numpy(np.vstack((rows, cols)).astype(np.int64))
    values = torch.from_numpy(rng.standard_normal(nnz).astype(np.float32)).requires_grad_(True)
    b = torch.from_numpy(rng.standard_normal((m, F)).astype(np.float32)).requires_grad_(True)
    G = torch.from_numpy(rng.standard_normal((n, F)).astype(np.float32))
    out = layers.SpecialSpmmFunction.apply(indices, values, torch.Size([n, m]), b)
    out.backward(G)
    save("special_spmm.npz", indices=indices.numpy(), values=values.detach().numpy(), b=b.detach().numpy(), G=G.numpy(),
         out=out.detach().numpy(), grad_values=values.grad.numpy(), grad_b=b.grad.numpy(), shape=np.array([n, m]))


def make_gat_cora_train():
    """Cora-sized GAT in TRAIN mode, dropout 0.6 (GAT/run.py:9) on features and on the attention matrices
    (layers.py:31), forward + every gradient, with the dropout masks replayed from seeds on both sides."""
    gat_mod, _ = R.gat_models()
    n = S.CORA["n"]
    edges, adj = _gat_adj(n, S.CORA["undirected_pairs"], seed=0)
    X = S.row_normalised_features(n, S.CORA["feats"], seed=1)
    labels = np.random.default_rng(2).integers(0, S.CORA["classes"], size=n)
    torch.manual_seed(2)
    model = gat_mod.GAT(S.CORA["feats"], 8, S.CORA["classes"], 0.6, 0.2, 8)
    model.train()
    import torch.nn.functional as Fnn
    from oracle.gat import replay_dropout
    orig, Fnn.dropout = Fnn.dropout, replay_dropout(1000)
    try:
        out = model(torch.from_numpy(X), torch.from_numpy(adj))
        calls = Fnn.dropout.k
    finally:
        Fnn.dropout = orig
    loss = torch.nn.functional.cross_entropy(out[:140], torch.from_numpy(labels)[:140])
    loss.backward()
    save("gat_cora_train.npz", edges=edges, adj_sha=np.array(sha(adj)), x_seed=np.int64(1), x_sha=np.array(sha(X)),
         labels=labels.astype(np.int64), dropout_base_seed=np.int64(1000), dropout_calls=np.int64(calls),
         out=out.detach().numpy(), loss=np.float64(loss.item()), **params_np(model), **grads_np(model))


def make_han_acm():
    """ACM-sized HAN (N=3025, 1870 features, 3 metapaths incl. a 24 %-dense one, 8 heads x 8), forward + every
    gradient, dropout 0: the CTA-per-row schedule of the attention kernels at the size BASELINE configs[3] names.
    Inputs are regenerated from seeds on the test side (checksums stored)."""
    ref = R.han()
    n, fin, M = S.ACM["n"], S.ACM["feats"], 3
    gs = [S.symmetric_mask(n, t, seed=11 + i) for i, t in enumerate(S.ACM["metapath_nnz"])]
    X = np.random.default_rng(14).standard_normal((n, fin), dtype=np.float32)
    labels = np.random.default_rng(15).integers(0, S.ACM["classes"], size=n)
    torch.manual_seed(5)
    model = ref["HAN"].HANModel(M, fin, 8, S.ACM["classes"], [8], 0.0)
    model.train()
    out = model([torch.from_numpy(g) for g in gs], torch.from_numpy(X))
    loss = torch.nn.functional.cross_entropy(out, torch.from_numpy(labels))
    loss.backward()
    save("han_acm.npz", mask_sha=np.array([sha(g) for g in gs]), x_sha=np.array(sha(X)), labels=labels.astype(np.int64),
         out=out.detach().numpy(), loss=np.float64(loss.item()), **params_np(model), **grads_np(model))


def make_gtn():
    """GTN_Model forward + backward (GTN/models/GTN.py) on a small 4-edge-type graph: the learned adjacency the final
    gcn_conv aggregates over is the output of two dense metapath compositions."""
    g = R.gtn()
    n, E, C, w_in, w_out, classes = 60, 4, 2, 12, 8, 3
    rng = np.random.default_rng(21)
    A = (rng.random((n, n, E)) < 0.08).astype(np.float32)
    A[:, :, E - 1] = np.eye(n, dtype=np.float32)  # the identity edge type GTN appends
    X = rng.standard_normal((n, w_in)).astype(np.float32)
    target = rng.choice(n, size=20, replace=False).astype(np.int64)
    labels = rng.integers(0, classes, size=20)
    torch.manual_seed(5)
    model = g["GTN"].GTN_Model(E, C, w_in, w_out, classes, 2, True)
    for m in model.modules():
        if isinstance(m, g["GTConv"].GTConv):
            torch.nn.init.normal_(m.weight, std=0.5)  # the reference leaves GTConv.weight uninitialised (GTConv.py:11)
    y, _ = model(torch.from_numpy(A), torch.from_numpy(X), torch.from_numpy(target))
    torch.nn.functional.cross_entropy(y, torch.from_numpy(labels)).backward()
    H_in = torch.rand(n, n, generator=torch.Generator().manual_seed(3)) * (torch.rand(n, n, generator=torch.Generator().manual_seed(4)) < 0.2)
    H_in.requires_grad_(True)
    out = model.gcn_conv(torch.from_numpy(X), H_in)
    Gout = torch.from_numpy(rng.standard_normal(out.shape).astype(np.float32))
    (dH,) = torch.autograd.grad((out * Gout).sum(), H_in)
    save("gtn_small.npz", A=A, X=X, target=target, labels=labels, y=y.detach().numpy(),
         norm_false=g["GTN"].norm(H_in.detach(), False).numpy(), norm_true=g["GTN"].norm(H_in.detach(), True).numpy(),
         H_in=H_in.detach().numpy(), conv_out=out.detach().numpy(), conv_gout=Gout.numpy(), conv_dH=dH.numpy(),
         **{"param." + k: v for k, v in params_np(model).items()}, **grads_np(model))


if __name__ == "__main__":
    assert R.available(), "reference not found"
    torch.set_num_threads(8)
    makers = {"gcn": make_gcn, "gat_small": make_gat_small, "gat_cora": make_gat_cora, "sage": make_sage,
              "sage_v2": make_sage_v2, "han": make_han, "gatne": make_gatne, "special_spmm": make_special_spmm,
              "gtn": make_gtn, "gat_cora_train": make_gat_cora_train, "han_acm": make_han_acm}
    # `python make_golden.py [name ...]`: only the named fixtures (the committed ones are not rewritten otherwise)
    for name in (sys.argv[1:] or list(makers)):
        makers[name]()
