"""The torch-only pieces of the drop-in layers against the UNMODIFIED reference classes, on the CPU.
Where the reference is available (oracle/ref_loader.py: $GNN_REFERENCE_ROOT or the oracle/_ref snapshot) the
tests run its classes live on fresh inputs; elsewhere they compare with the reference outputs and weights stored
in tests/golden/, and skip the configurations no fixture stored.  The CUDA-backed pieces are covered by tests/test_gpu_parity.py against
fixtures generated from the same classes."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from graphneuralnetwork_b200 import layers
from oracle import ref_loader as R

needs_reference = pytest.mark.skipif(not R.available(), reason="reference tree not present")
TOL = 1e-5


def _rel(a, b):
    return float(((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).detach())


def _copy_state(dst, src):
    dst.load_state_dict(src.state_dict(), strict=True)


@pytest.mark.parametrize("hidden_method", ["sum", "concat"])
@pytest.mark.parametrize("activation", ["relu", None])
def test_sagegcn_combination_matches_reference(hidden_method, activation):
    """SageGCN.py:23-36: self/neighbour products, sum | concat, optional activation.  Ours receives the
    already-aggregated neighbours (what the kernel returns); the reference aggregates its 3-D input itself."""
    if not R.available():
        if hidden_method == "concat":
            pytest.skip("no stored reference output for aggr_hidden_method='concat'")
        # the stored reference GraphSage forward (GraphSage.py:18-30): layer 0 relu, layer 1 no activation
        from oracle import sage as osage
        g = load_golden("sage_small.npz")
        table = torch.from_numpy(np.random.default_rng(int(g["table_seed"])).standard_normal((500, 602), dtype=np.float32))
        hidden = [osage.gather_features(table, g[f"block{i}"]) for i in range(3)]
        for l, (fin, fout, act) in enumerate(((602, 128, torch.nn.functional.relu), (128, 41, None))):
            ours = layers.SageGCN(fin, fout, activation=act, aggr_neighbor_method="mean", aggr_hidden_method="sum")
            ours.load_state_dict({k: torch.from_numpy(g[f"gcn.{l}.{k}"]) for k in ("weight", "aggregator.weight")})
            hidden = [ours(hidden[hop], hidden[hop + 1].view(hidden[hop].shape[0], (5, 3)[hop], -1).mean(dim=1))
                      for hop in range(len(hidden) - 1)]
        assert _rel(hidden[0], torch.from_numpy(g["out"])) < TOL
        return
    ref = R.sage_pytorch()
    act = torch.nn.functional.relu if activation else None
    torch.manual_seed(0)
    theirs = ref["SageGCN"].SageGCN(24, 16, activation=act, aggr_neighbor_method="mean", aggr_hidden_method=hidden_method)
    ours = layers.SageGCN(24, 16, activation=act, aggr_neighbor_method="mean", aggr_hidden_method=hidden_method)
    _copy_state(ours, theirs)
    src, neigh = torch.randn(50, 24), torch.randn(50, 7, 24)
    assert _rel(ours(src, neigh.mean(dim=1)), theirs(src, neigh)) < TOL


def test_neighbor_aggregator_bias_matches_reference():
    if not R.available():  # the stored reference aggregator (identity weight, no bias) on the fixture's hop-1 block
        from oracle import sage as osage
        g = load_golden("sage_small.npz")
        table = torch.from_numpy(np.random.default_rng(int(g["table_seed"])).standard_normal((500, 602), dtype=np.float32))
        neigh = osage.gather_features(table, g["block1"]).view(32, 5, -1)
        for method in ("mean", "sum"):
            ours = layers.NeighborAggregator(602, 16, aggr_method=method)
            ours.load_state_dict({"weight": torch.eye(602)[:, :16]})
            reduced = neigh.mean(dim=1) if method == "mean" else neigh.sum(dim=1)
            assert _rel(ours(reduced).detach(), torch.from_numpy(g[f"agg.{method}"])) < TOL, method
        return
    ref = R.sage_pytorch()
    torch.manual_seed(1)
    theirs = ref["Aggregator"].NeighborAggregator(24, 16, use_bias=True, aggr_method="sum")
    theirs.bias.data.normal_()
    ours = layers.NeighborAggregator(24, 16, use_bias=True, aggr_method="sum")
    _copy_state(ours, theirs)
    neigh = torch.randn(40, 5, 24)
    assert _rel(ours(neigh.sum(dim=1)), theirs(neigh)) < TOL


@pytest.mark.parametrize("gcn", [False, True])
def test_sage_v2_layer_split_weight_matches_reference(gcn):
    """GraphSAGE/GraphSAGE.py:7-21: relu(W [self ‖ agg]) computed without the concat copy."""
    if not R.available():
        if gcn:
            pytest.skip("no stored reference output for SageLayer(gcn=True)")
        # the stored reference GraphSAGE forward (GraphSAGE.py:43-49), both layers through our SageLayer
        from oracle import sage as osage
        g = load_golden("sage_v2_small.npz")
        center, neigh = torch.from_numpy(g["center_feats"]), torch.from_numpy(g["neigh_feats"])
        cmap, nmap = torch.from_numpy(g["center_map"]), torch.from_numpy(g["neigh_map"])
        l0, l1 = layers.SageLayer(64, 32), layers.SageLayer(32, 32)
        for l, layer in enumerate((l0, l1)):
            layer.load_state_dict({"weight.weight": torch.from_numpy(g[f"sage_blocks.sage_layer{l}.weight.weight"])})
        h = l0(center, osage.aggregator_v2(neigh))
        h2 = l1(torch.embedding(h, cmap[0][cmap[0] != -1]), osage.embed_mean_v2(h, nmap[0]))
        assert _rel(h2.detach(), torch.from_numpy(g["feats_out"])) < TOL
        return
    ref = R.sage_v2()
    torch.manual_seed(2)
    theirs = ref["GraphSAGE"].SageLayer(20, 12, gcn=gcn)
    ours = layers.SageLayer(20, 12, gcn=gcn)
    _copy_state(ours, theirs)
    a, b = torch.randn(33, 20), torch.randn(33, 20)
    assert _rel(ours(a, b), theirs(a, b)) < TOL


@needs_reference
def test_semantic_attention_matches_reference():
    ref = R.han()
    torch.manual_seed(3)
    theirs = ref["SemanticAttention"].SemanticAttention(in_size=64, hidden_size=128)
    ours = layers.SemanticAttention(in_size=64, hidden_size=128)
    _copy_state(ours, theirs)
    z = torch.randn(300, 3, 64)
    assert _rel(ours(z), theirs(z)) < TOL
    z.requires_grad_(True)
    go = torch.randn(300, 64)
    g1, = torch.autograd.grad(ours(z), z, go)
    g2, = torch.autograd.grad(theirs(z), z, go)
    assert _rel(g1, g2) < TOL


@needs_reference
def test_gatne_decoder_matches_reference():
    ref_pt, _ = R.gatne()
    torch.manual_seed(4)
    theirs = ref_pt.GraphDecoder(100, 32)
    ours = layers.GraphDecoder(100, 32)
    _copy_state(ours, theirs)
    emb, cn = torch.randn(16, 32), torch.randint(0, 100, (16, 6))
    assert _rel(ours(emb, cn), theirs(emb, cn)) < TOL


# what tests/golden/make_golden.py stores beside a reference state_dict (inputs, outputs, checksums); every
# other key of a fixture, gradients aside, is a reference parameter in state_dict order
_FIXTURE_DATA = {"edges", "coo_row", "coo_col", "coo_val", "x_seed", "x_sha", "labels", "out", "layer0_out", "loss",
                 "adj", "X", "isolated_row", "adj_sha", "table_seed", "table_sha", "adj_ptr", "adj_flat", "block0",
                 "block1", "block2", "agg.mean", "agg.sum", "center_feats", "center_map", "neigh_feats", "neigh_map",
                 "feats_out", "classes", "masks_packed", "n", "inputs", "types", "neigh", "features", "target"}


def test_model_constructors_consume_the_same_rng_stream():
    """Same seed => same initial weights as the reference constructors (parameter creation order and
    initialisers match), so a run seeded like the reference starts from the reference's weights.  The
    reference side is the initial state_dict each fixture stored (tests/golden/make_golden.py: the seed set
    right before the reference constructor ran, no optimiser step after it)."""
    gatne_feats = torch.from_numpy(load_golden("gatne_small.npz")["features"])
    for fixture, prefix, seed, build_ours in (
            ("gcn_cora.npz", "", 0, lambda: layers.GCN_Model(1433, 16, 7, 2, 0.5)),
            ("gat_small.npz", "dense.", 1, lambda: layers.GAT(50, 8, 7, 0.0, 0.2, 8)),
            ("gat_small.npz", "sparse.", 1, lambda: layers.SpGAT(50, 8, 7, 0.0, 0.2, 8)),
            ("gat_cora.npz", "", 2, lambda: layers.GAT(1433, 8, 7, 0.6, 0.2, 8)),
            ("sage_small.npz", "", 3, lambda: layers.GraphSage(602, [128, 41], [5, 3])),
            ("sage_v2_small.npz", "", 4, lambda: layers.GraphSAGE(2, 64, 32, gcn=False, agg_func='MEAN',
                                                                 Unsupervised=False, class_size=3)),
            ("han_small.npz", "", 5, lambda: layers.HANModel(3, 40, 8, 3, [8], 0.0)),
            ("gatne_small.npz", "pt_t_sum.", 7, lambda: layers.GraphEncoder(300, 32, 10, 3, 20, None, agg_func="SUM")),
            ("gatne_small.npz", "pt_i_sum.", 7, lambda: layers.GraphEncoder(300, 32, 10, 3, 20, gatne_feats,
                                                                            agg_func="SUM")),
            ("gatne_small.npz", "v1_t.", 7, lambda: layers.GATNEModelV1(300, 32, 10, 3, 20, None)),
            ("gatne_small.npz", "v1_i.", 7, lambda: layers.GATNEModelV1(300, 32, 10, 3, 20, gatne_feats)),
    ):
        g = load_golden(fixture)
        torch.manual_seed(seed)
        b = build_ours().state_dict()
        # exactly the reference state_dict's parameter names, in its order, and the same values
        ref_keys = [k[len(prefix):] for k in g if k.startswith(prefix) and not k[len(prefix):].startswith("grad.")
                    and k[len(prefix):] not in _FIXTURE_DATA]
        assert ref_keys == list(b), fixture + prefix
        for k, v in b.items():
            assert g[prefix + k].shape == tuple(v.shape) and np.array_equal(g[prefix + k], v.numpy()), fixture + prefix + k
