"""The drop-in claim, executed: the reference's OWN model classes and training loop, with the layers on the hot
path substituted by import path (SURVEY.md §8b "installed by import-path substitution"), run on the GPU and
are compared with the unmodified reference run on the CPU from the same seed.

The reference modules come from the checkout $GNN_REFERENCE_ROOT names or from the verbatim snapshot in the
git-ignored oracle/_ref/ (tools/make_ref_snapshot.py, made by __graft_entry__.build()).  Skipped when neither exists.
  * GCN   GCN/GCN.py:21-27 `GCN_Model` (dispatch on `_get_name() == 'Graph_conv_layer'`) built from the reference
          class with `Graph_conv_layer` replaced, trained by the reference's `train` (GCN/train_eval.py:20-66);
  * SAGE  GraphSAGE_Pytorch `GraphSage` / `SageGCN` with `NeighborAggregator` replaced, fed by the reference's own
          `collate_fn` (data_utils.py:52-65: python sampler + list gather);
  * HAN   HAN/models/HAN.py `HANModel` with `GATConv` replaced, forward + backward."""
import copy
import os
import random

import numpy as np
import pytest
import torch

from conftest import rel_err
from graphneuralnetwork_b200 import layers, synthetic as S
from oracle import gcn as ogcn
from oracle import ref_loader

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not ref_loader.available(), reason="no reference snapshot (oracle/_ref)")]
DEV = "cuda"


def _cora_like(n=600, pairs=1500, feats=64, classes=7, seed=0):
    edges = S.cora_like_edges(n, pairs, seed)
    row, col, val = ogcn.build_adjacency(edges, n)
    adj = torch.sparse_coo_tensor(torch.from_numpy(np.vstack((row, col))), torch.from_numpy(val), (n, n))
    X = torch.from_numpy(S.row_normalised_features(n, feats, seed + 1))
    y = torch.from_numpy(np.random.default_rng(seed + 2).integers(0, classes, n))
    idx = torch.arange(n)
    return adj, X, y, idx[:140], idx[140:300], idx[300:]


def test_reference_gcn_train_loop_with_dropin_layer(lib, tmp_path, monkeypatch, capsys):
    ref_gcn, _ = ref_loader.gcn()
    train_eval = ref_loader.gcn_train_eval()
    data = _cora_like()
    monkeypatch.chdir(tmp_path)
    os.mkdir("saved_dict")  # the reference loop saves checkpoints under ./saved_dict/GCN (train_eval.py:35-39)

    def run(layer_cls, device):
        monkeypatch.setattr(ref_gcn, "Graph_conv_layer", layer_cls)
        torch.manual_seed(7)
        model = ref_gcn.GCN_Model(64, 16, 7, 2, 0.0)  # dropout 0: the CPU and CUDA generators differ
        torch.manual_seed(8)                           # `train` re-initialises every nn.Linear (train_eval.py:21-25)
        train_eval.train(model, data, 0.01, 3, torch.device(device))
        return {k: v.detach().cpu() for k, v in model.state_dict().items()}

    want = run(ref_gcn.Graph_conv_layer, "cpu")        # the unmodified reference, CPU
    got = run(layers.Graph_conv_layer, DEV)            # same reference model + loop, our layer, GPU
    assert "Epoch [1/3]" in capsys.readouterr().out    # the reference loop really ran (its own log line)
    assert os.path.exists("saved_dict/GCN/GCN.ckpt")
    assert want.keys() == got.keys()                   # identical state_dict keys: checkpoints interchange
    for k in want:
        assert rel_err(got[k].numpy(), want[k].numpy()) < 1e-4, k  # 3 Adam steps apart from fp32 re-association


def test_reference_graphsage_with_dropin_aggregator_on_reference_collate(lib, monkeypatch):
    mods = ref_loader.sage_pytorch()
    du = ref_loader.sage_data_utils()
    n, F_in, fan = 400, 48, [5, 3]
    adj_lists = S.adjacency_lists(n, 6, seed=1)
    rng = np.random.default_rng(2)
    feat = rng.standard_normal((n, F_in)).astype(np.float32)
    collate = du.collate_fn(adj_lists, feat.tolist(), fan)   # the reference's sampler + python-list gather
    random.seed(0)
    feats, labels = collate([(i, int(i % 3)) for i in range(32)])
    assert [f.shape[0] for f in feats] == [32, 160, 480]
    torch.manual_seed(3)
    ref_model = mods["GraphSage"].GraphSage(F_in, [32, 3], fan)
    want = ref_model(feats)
    torch.nn.functional.cross_entropy(want, labels).backward()
    monkeypatch.setattr(mods["SageGCN"], "NeighborAggregator", layers.NeighborAggregator)
    torch.manual_seed(3)
    model = mods["GraphSage"].GraphSage(F_in, [32, 3], fan)  # the reference GraphSage/SageGCN around OUR aggregator
    assert type(model.gcn[0].aggregator) is layers.NeighborAggregator
    model.load_state_dict(ref_model.state_dict(), strict=True)
    model = model.to(DEV)
    got = model([f.to(DEV) for f in feats])
    torch.nn.functional.cross_entropy(got, labels.to(DEV)).backward()
    assert rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < 1e-5
    for (name, p), (_, q) in zip(model.named_parameters(), ref_model.named_parameters()):
        assert rel_err(p.grad.cpu().numpy(), q.grad.numpy()) < 2e-5, name


def test_reference_han_model_with_dropin_gatconv(lib, monkeypatch):
    mods = ref_loader.han()
    n, F_in = 150, 20
    gs = [torch.from_numpy(S.symmetric_mask(n, t, seed=5 + i)) for i, t in enumerate((400, 4000))]
    X = torch.from_numpy(np.random.default_rng(6).standard_normal((n, F_in)).astype(np.float32))
    y = torch.from_numpy(np.random.default_rng(7).integers(0, 3, n))
    torch.manual_seed(1)
    ref_model = mods["HAN"].HANModel(2, F_in, 8, 3, [4], 0.0)
    want = ref_model(gs, X)
    torch.nn.functional.cross_entropy(want, y).backward()
    monkeypatch.setattr(mods["HAN"], "GATConv", layers.GATConv)
    torch.manual_seed(1)
    model = mods["HAN"].HANModel(2, F_in, 8, 3, [4], 0.0)   # reference HANModel / HANLayer / SemanticAttention
    assert type(list(model.layers[0].gat_layers)[0]) is layers.GATConv
    model.load_state_dict(copy.deepcopy(ref_model.state_dict()), strict=True)
    model = model.to(DEV)
    got = model([g.to(DEV) for g in gs], X.to(DEV))
    torch.nn.functional.cross_entropy(got, y.to(DEV)).backward()
    assert rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < 1e-5
    for (name, p), (_, q) in zip(model.named_parameters(), ref_model.named_parameters()):
        assert rel_err(p.grad.cpu().numpy(), q.grad.numpy()) < 2e-5, name


def test_reference_semantic_attention_state_dict_and_gradients(lib):
    """The reference's own SemanticAttention (HAN/models/SemanticAttention.py:5-20) on the CPU against the fused
    drop-in on the GPU: identical state_dict keys (strict load), forward and every gradient."""
    mods = ref_loader.han()
    n, m, d = 300, 3, 64
    torch.manual_seed(2)
    ref = mods["SemanticAttention"].SemanticAttention(in_size=d)
    z = torch.randn(n, m, d)
    gy = torch.randn(n, d)
    zr = z.clone().requires_grad_(True)
    want = ref(zr)
    want.backward(gy)
    ours = layers.SemanticAttention(in_size=d)
    ours.load_state_dict(copy.deepcopy(ref.state_dict()), strict=True)
    ours = ours.to(DEV)
    zg = z.to(DEV).requires_grad_(True)
    got = ours(zg)
    got.backward(gy.to(DEV))
    assert got.shape == want.shape and rel_err(got.detach().cpu().numpy(), want.detach().numpy()) < 1e-5
    assert rel_err(zg.grad.cpu().numpy(), zr.grad.numpy()) < 2e-5
    for (name, p), (_, q) in zip(ours.named_parameters(), ref.named_parameters()):
        assert rel_err(p.grad.cpu().numpy(), q.grad.numpy()) < 1e-4, name  # fp32 reference on the other side
