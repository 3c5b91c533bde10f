"""The oracle against the reference: every oracle function that a GPU parity test leans on is re-pinned here.
Where the reference modules are available (oracle/ref_loader.py: $GNN_REFERENCE_ROOT or the oracle/_ref
snapshot) each test runs them LIVE on fresh seeded inputs; elsewhere it compares with the outputs the
unmodified reference stored in tests/golden/ (tests/golden/make_golden.py)."""
import random

import numpy as np
import pytest
import torch

from conftest import load_golden
from graphneuralnetwork_b200 import synthetic as S
from oracle import gat as ogat, gatne as ogatne, gcn as ogcn, ref_loader as R, sage as osage

LIVE = R.available()
TOL = 1e-5


def _params(g, prefix=""):
    """The reference state_dict a fixture stored (float32 arrays; gradients excluded)."""
    return {k[len(prefix):]: torch.from_numpy(v) for k, v in g.items()
            if k.startswith(prefix) and not k[len(prefix):].startswith("grad.") and v.dtype == np.float32 and v.ndim >= 1}


def _rel(a, b):
    a, b = torch.as_tensor(a, dtype=torch.float64), torch.as_tensor(b, dtype=torch.float64)
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_gcn_adjacency_pipeline_bit_exact(seed):
    """GCN/data_utils.py:35,54-70 on random directed edge lists with duplicates and both directions."""
    import scipy.sparse as sp
    if not LIVE:
        return _adjacency_vs_fixture(seed)
    _, du = R.gcn()
    rng = np.random.default_rng(seed)
    n = 300
    edges = rng.integers(0, n, (1500, 2)).astype(np.int32)
    edges = edges[edges[:, 0] != edges[:, 1]]
    edges = np.unique(edges, axis=0)  # load_cora's edge list has no duplicate rows
    adj = sp.coo_matrix((np.ones(edges.shape[0]), (edges[:, 0], edges[:, 1])), shape=(n, n), dtype=np.float32)
    adj = adj + adj.T.multiply(adj.T > adj) - adj.multiply(adj.T > adj)
    ref = du.sparse_mx_to_torch_sparse_tensor(du.normalize_adj(adj + sp.eye(n)))
    row, col, val = ogcn.build_adjacency(edges, n)
    idx = ref._indices().numpy()
    assert np.array_equal(idx[0], row) and np.array_equal(idx[1], col)
    assert np.array_equal(ref._values().numpy().view(np.uint32), val.view(np.uint32))


def _adjacency_vs_fixture(seed):
    """One reference-normalised adjacency per seed: the GCN Cora-shaped COO (exact arrays), the 300-node GAT
    dense matrix (exact, row 17 emptied by the fixture) and the Cora-shaped GAT dense matrix (sha256)."""
    import hashlib
    name = ("gcn_cora.npz", "gat_small.npz", "gat_cora.npz")[seed]
    g = load_golden(name)
    n = 300 if name == "gat_small.npz" else S.CORA["n"]
    row, col, val = ogcn.build_adjacency(g["edges"], n)
    if name == "gcn_cora.npz":
        assert np.array_equal(row, g["coo_row"]) and np.array_equal(col, g["coo_col"])
        assert np.array_equal(val.view(np.uint32), g["coo_val"].view(np.uint32))
        return
    dense = np.zeros((n, n), np.float32)
    dense[row, col] = val
    if name == "gat_small.npz":
        dense[int(g["isolated_row"]), :] = 0
        assert np.array_equal(dense.view(np.uint32), g["adj"].view(np.uint32))
    else:
        assert hashlib.sha256(dense.tobytes()).hexdigest() == str(g["adj_sha"])


@pytest.mark.parametrize("seed", [0, 1])
@pytest.mark.parametrize("sparse", [False, True])
def test_gat_heads(seed, sparse):
    if not LIVE:  # the 8-head + output-head model the fixture stored, dense and sparse layers
        g = load_golden("gat_small.npz")
        X, adj = torch.from_numpy(g["X"]), torch.from_numpy(g["adj"])
        kind = "sparse" if sparse else "dense"
        if sparse:  # the fixture's SpGAT input keeps a self-loop on the isolated row
            adj = adj.clone()
            adj[int(g["isolated_row"]), int(g["isolated_row"])] = 1.0
        assert _rel(ogat.gat_model(X, _params(g, kind + "."), adj, 0.2, 8, sparse=sparse), g[kind + ".out"]) < TOL
        if not sparse:
            W, a = _params(g, "dense.")[f"attentions.AttentionHead{seed}.W"], _params(g, "dense.")[f"attentions.AttentionHead{seed}.a"]
            lit = ogat.dense_head(X, W, a, adj, 0.2, True, materialise_pairs=True)
            assert _rel(ogat.dense_head(X, W, a, adj, 0.2, True, materialise_pairs=False), lit) < TOL
        return
    layers = R.gat_layers()
    torch.manual_seed(seed)
    n, fin, fout = 60, 20, 8
    adj = (torch.rand(n, n) < 0.1).float()
    adj = ((adj + adj.t() + torch.eye(n)) > 0).float()
    x = torch.randn(n, fin)
    cls = layers.SpGraphAttentionLayer if sparse else layers.GraphAttentionLayer
    for concat in (True, False):
        head = cls(fin, fout, dropout=0.0, alpha=0.2, concat=concat).eval()
        fn = ogat.sparse_head if sparse else ogat.dense_head
        out = fn(x, head.W.detach(), head.a.detach(), adj, 0.2, concat)
        assert _rel(out, head(x, adj).detach()) < TOL
    if not sparse:  # the literal [N,N,2F'] materialisation agrees with the decomposed score
        head = cls(fin, fout, dropout=0.0, alpha=0.2, concat=True).eval()
        a = ogat.dense_head(x, head.W.detach(), head.a.detach(), adj, 0.2, True, materialise_pairs=True)
        b = ogat.dense_head(x, head.W.detach(), head.a.detach(), adj, 0.2, True, materialise_pairs=False)
        assert _rel(a, b) < TOL


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_graphsage_forward_and_sampler(seed):
    if not LIVE:  # the fixture's forward and its sampled blocks (Python's RNG seeded 0 before the sampler)
        g = load_golden("sage_small.npz")
        table = torch.from_numpy(np.random.default_rng(int(g["table_seed"])).standard_normal((500, 602), dtype=np.float32))
        feats = [osage.gather_features(table, g[f"block{i}"]) for i in range(3)]
        assert _rel(osage.graphsage_forward(feats, _params(g), [5, 3]), g["out"]) < TOL
        adj = S.adjacency_lists(500, 8, seed=6)
        random.seed(0)
        blocks = osage.multihop_sampling(list(range(40, 72)), [5, 3], adj)
        assert all(np.array_equal(np.asarray(blocks[i], np.int64), g[f"block{i}"]) for i in range(3))
        return
    ref = R.sage_pytorch()
    torch.manual_seed(seed)
    model = ref["GraphSage"].GraphSage(30, [16, 5], [4, 3]).eval()
    feats = [torch.randn(8, 30), torch.randn(32, 30), torch.randn(96, 30)]
    params = {k: v.detach() for k, v in model.state_dict().items()}
    assert _rel(osage.graphsage_forward(feats, params, [4, 3]), model(feats).detach()) < TOL
    # the sampler consumes Python's global RNG exactly like the reference's
    table = {i: set(np.random.default_rng(seed + i).integers(0, 50, 1 + i % 9).tolist()) for i in range(50)}
    random.seed(seed)
    theirs = ref["sample_utils"].multihop_sampling([1, 2, 3], [4, 3], table)
    random.seed(seed)
    ours = osage.multihop_sampling([1, 2, 3], [4, 3], table)
    assert [list(map(int, a)) for a in theirs] == [list(map(int, b)) for b in ours]


@pytest.mark.parametrize("seed", [0, 1])
def test_han_model(seed):
    if not LIVE:  # seed 0: the 150-node fixture, seed 1: the ACM-sized one
        if seed == 0:
            g = load_golden("han_small.npz")
            n = int(g["n"])
            gs = [torch.from_numpy(np.unpackbits(m, axis=1)[:, :n].astype(np.float64)) for m in g["masks_packed"]]
            h = torch.from_numpy(g["X"])
        else:
            g = load_golden("han_acm.npz")
            n = S.ACM["n"]
            gs = [torch.from_numpy(S.symmetric_mask(n, t, seed=11 + i)) for i, t in enumerate(S.ACM["metapath_nnz"])]
            h = torch.from_numpy(np.random.default_rng(14).standard_normal((n, S.ACM["feats"]), dtype=np.float32))
        assert _rel(ogat.han_model(gs, h, _params(g), [8]), g["out"]) < TOL
        return
    ref = R.han()
    torch.manual_seed(seed)
    n, fin = 40, 12
    model = ref["HAN"].HANModel(2, fin, 4, 3, [2], 0.0).eval()
    gs = []
    for k in range(2):
        m = (torch.rand(n, n) < 0.15)
        gs.append(((m | m.t() | torch.eye(n, dtype=torch.bool))).double())
    h = torch.randn(n, fin)
    params = {k: v.detach() for k, v in model.state_dict().items()}
    assert _rel(ogat.han_model(gs, h, params, [2]), model(gs, h).detach()) < TOL


@pytest.mark.parametrize("seed", [0, 1])
def test_gatne_encoders(seed):
    if not LIVE:  # both reference variants, with learned embeddings and with node features
        g = load_golden("gatne_small.npz")
        inputs, types, neigh = (torch.from_numpy(g[k]) for k in ("inputs", "types", "neigh"))
        feats = torch.from_numpy(g["features"])
        for tag, f, agg in (("pt_t_sum", None, "SUM"), ("pt_t_mean", None, "MEAN"), ("pt_i_sum", feats, "SUM"),
                            ("v1_t", None, "SUM"), ("v1_i", feats, "SUM")):
            out = ogatne.encoder_forward(_params(g, tag + "."), inputs, types, neigh, f, agg)
            assert _rel(out, g[f"{tag}.out"]) < TOL, tag
        return
    ref_pt, ref_v1 = R.gatne()
    rng = np.random.default_rng(seed)
    N, T, K, B, E, U, A, Fd = 80, 2, 5, 16, 12, 6, 7, 9
    inputs, types = torch.from_numpy(rng.integers(0, N, B)), torch.from_numpy(rng.integers(0, T, B))
    neigh = torch.from_numpy(rng.integers(0, N, (B, T, K)))
    feats = torch.from_numpy(rng.standard_normal((N, Fd)).astype(np.float32))
    for ctor, f, agg in ((lambda: ref_pt.GraphEncoder(N, E, U, T, A, None, agg_func="MEAN"), None, "MEAN"),
                         (lambda: ref_pt.GraphEncoder(N, E, U, T, A, feats, agg_func="SUM"), feats, "SUM"),
                         (lambda: ref_v1.GATNEModel(N, E, U, T, A, None), None, "SUM"),
                         (lambda: ref_v1.GATNEModel(N, E, U, T, A, feats), feats, "SUM")):
        torch.manual_seed(seed)
        model = ctor()
        params = {k: v.detach() for k, v in model.state_dict().items()}
        assert _rel(ogatne.encoder_forward(params, inputs, types, neigh, f, agg), model(inputs, types, neigh).detach()) < TOL


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_gtn_norm_and_gcn_conv(seed):
    """GTN/models/GTN.py:7-19 (norm, both modes, bit-exact) and :49-52 (gcn_conv) on fresh learned adjacencies,
    including empty columns (deg 0 -> inf -> 0); the drop-in's element-wise `norm` is bit-identical too."""
    from oracle import gtn as ogtn
    from graphneuralnetwork_b200.layers import gtn as lgtn
    if not LIVE:  # the fixture's learned adjacency (norm of both modes) and gcn_conv output
        g = load_golden("gtn_small.npz")
        H = torch.from_numpy(g["H_in"])
        for add, key in ((False, "norm_false"), (True, "norm_true")):
            assert np.array_equal(ogtn.norm(H, add).numpy(), g[key]) and np.array_equal(lgtn.norm(H, add).numpy(), g[key])
        conv = ogtn.gcn_conv(torch.from_numpy(g["X"]), H, torch.from_numpy(g["param.weight"]))
        assert _rel(conv, g["conv_out"]) < 1e-6
        return
    ref = R.gtn()["GTN"]
    g = torch.Generator().manual_seed(seed)
    n = 50 + 7 * seed
    H = torch.rand(n, n, generator=g) * (torch.rand(n, n, generator=g) < 0.15)
    H[:, 3] = 0  # an empty column
    for add in (False, True):
        want = ref.norm(H, add)
        assert torch.equal(ogtn.norm(H, add), want)
        assert torch.equal(lgtn.norm(H, add), want)
    torch.manual_seed(seed)
    model = ref.GTN_Model(3, 2, 10, 6, 3, 1, True)
    X = torch.randn(n, 10, generator=g)
    assert _rel(ogtn.gcn_conv(X, H, model.weight.detach()), model.gcn_conv(X, H).detach()) < 1e-6
