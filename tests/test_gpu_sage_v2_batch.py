"""De-duplicating GraphSAGE minibatches built on the device (`functional.dedup_layer_nodes`) against the oracle fed
with the same device draws, and `GraphSAGE.forward_sampled` against `forward` on the same batch gathered on the
host: logits and weight gradients bit for bit (the gather kernels add in the same order on the identity-block and
id-map paths, DESIGN §4.2)."""
import copy

import numpy as np
import pytest
import torch

from conftest import load_golden
from graphneuralnetwork_b200 import _lib, functional as Fn, layers
from graphneuralnetwork_b200 import synthetic as S
from graphneuralnetwork_b200.graph import CSRGraph
from oracle.sage_dedup import layer_adj_nodes_v2

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _graph(n=300, deg=6, seed=9):
    adj = S.adjacency_lists(n, deg, seed=seed)
    ptr = np.cumsum([0] + [len(adj[i]) for i in range(n)]).astype(np.int64)
    flat = np.concatenate([np.asarray(sorted(adj[i]), dtype=np.int32) for i in range(n)])
    return adj, CSRGraph(cuda(ptr), cuda(flat), None, n, n)


def _host_collate(table, b):
    """What the reference collate hands `forward`: X[S_0], the maps, and X[outer draws] as [n0, k, F]."""
    t = table.cpu()
    s0 = b.nodes[0].cpu()
    ids = b.outer_neighbors.cpu()
    return (t[s0].to(DEV), b.center_map, t[ids.reshape(-1)].reshape(*ids.shape, -1).to(DEV), b.neigh_map)


@pytest.mark.parametrize("L", [1, 2, 3])
def test_dedup_layer_nodes_matches_oracle(lib, L):
    adj, g = _graph()
    k, seed = 4, 77
    batch = [131, 20, 7, 299, 42, 0, 58, 21, 200, 150]
    b = Fn.dedup_layer_nodes(g, batch, L, k, seed)

    def draws(level, nodes):
        d = Fn.sample_neighbors(g, cuda(np.asarray(nodes, np.int64)), k, seed + 0x9E3779B9 * (L - level), torch.int64)
        assert torch.equal(d.view(-1, k), b.neighbors[level])  # the batch carries exactly these draws
        return d.cpu().numpy()

    nodes, cm, nm, outer = layer_adj_nodes_v2(adj, batch, L, k, draws)
    assert b.counts == [len(x) for x in nodes]
    for got, want in zip(b.nodes, nodes):
        assert got.dtype == torch.int64 and np.array_equal(got.cpu().numpy(), want)
    assert np.array_equal(b.center_map.cpu().numpy(), cm)
    assert np.array_equal(b.neigh_map.cpu().numpy(), nm)
    assert np.array_equal(b.outer_neighbors.cpu().numpy(), outer)
    again = Fn.dedup_layer_nodes(g, batch, L, k, seed)
    assert again.counts == b.counts
    for x, y in zip(again.nodes + again.neighbors + [again.center_map, again.neigh_map],
                    b.nodes + b.neighbors + [b.center_map, b.neigh_map]):
        assert torch.equal(x, y)


def _pair(L, F, gcn, agg, classes=5, unsupervised=False):
    torch.manual_seed(5)
    m = layers.GraphSAGE(L, F, 32, gcn=gcn, agg_func=agg, Unsupervised=unsupervised, class_size=classes).to(DEV)
    return m, copy.deepcopy(m)


@pytest.mark.parametrize("F", [64, 602])
@pytest.mark.parametrize("agg,gcn,L,grads", [("MEAN", False, 2, True), ("MEAN", True, 2, True), ("MEAN", False, 3, True),
                                             ("MAX", False, 1, True), ("MAX", True, 1, True), ("MAX", False, 2, False),
                                             ("MAX", True, 3, False)])
def test_forward_sampled_is_forward_bit_for_bit(lib, F, agg, gcn, L, grads):
    """MAX runs its gradients at L = 1 only: `forward` has no max backward into a gathered layer output."""
    _, g = _graph()
    table = torch.from_numpy(np.random.default_rng(1).standard_normal((300, F), dtype=np.float32)).to(DEV)
    padded = Fn.pad_table(table)
    b = Fn.dedup_layer_nodes(g, list(range(40, 56)), L, 5, seed=3)
    labels = cuda(np.random.default_rng(2).integers(0, 5, 16))
    m_host, m_dev = _pair(L, F, gcn, agg)
    with torch.set_grad_enabled(grads):
        e1, y1 = m_host(*_host_collate(table, b), None, None, None, None, None)
        e2, y2 = m_dev.forward_sampled(padded, b)
    assert torch.equal(e1, e2) and torch.equal(y1, y2)
    if grads:
        torch.nn.functional.cross_entropy(y1, labels).backward()
        torch.nn.functional.cross_entropy(y2, labels).backward()
        for (name, p1), (_, p2) in zip(m_host.named_parameters(), m_dev.named_parameters()):
            assert torch.equal(p1.grad, p2.grad), name


def test_forward_sampled_unsupervised_head(lib):
    _, g = _graph()
    table = torch.from_numpy(np.random.default_rng(4).standard_normal((300, 64), dtype=np.float32)).to(DEV)
    B, C = 6, 3
    centers = Fn.dedup_layer_nodes(g, list(range(100, 100 + B)), 2, 4, seed=8)
    others = Fn.dedup_layer_nodes(g, np.random.default_rng(5).integers(0, 300, B * C), 2, 4, seed=9)
    m_host, m_dev = _pair(2, 64, False, "MEAN", unsupervised=True)
    e1, s1 = m_host(*_host_collate(table, centers), *_host_collate(table, others), (B, C))
    e2, s2 = m_dev.forward_sampled(Fn.pad_table(table), centers, others, (B, C))
    assert s1.shape == s2.shape == (B, 1, C)
    for a, b in ((e1, e2), (s1, s2)):
        assert (a - b).abs().max().item() <= 1e-5 * max(b.abs().max().item(), 1.0)
    s2.sum().backward()
    assert all(p.grad is not None for p in m_dev.parameters())


def test_dedup_refuses_a_graph_with_an_empty_row(lib):
    ptr = cuda(np.array([0, 1, 1, 2], np.int64))  # row 1 has no edges
    g = CSRGraph(ptr, cuda(np.array([1, 0], np.int32)), None, 3, 3)
    with pytest.raises(_lib.GnnError, match="without edges"):
        Fn.dedup_layer_nodes(g, [0], 2, 2, seed=0)
    _, g = _graph()
    with pytest.raises(IndexError):
        Fn.dedup_layer_nodes(g, [0, 300], 2, 2, seed=0)


def test_drop_in_trains_on_golden_parameters(lib):
    """The golden's model (tests/golden/sage_v2_small.npz) trains three Adam steps on device-built batches."""
    gd = load_golden("sage_v2_small.npz")
    _, g = _graph()
    table = Fn.pad_table(torch.from_numpy(np.random.default_rng(10).standard_normal((300, 64), dtype=np.float32)).to(DEV))
    model = layers.GraphSAGE(2, 64, 32, gcn=False, agg_func='MEAN', Unsupervised=False, class_size=3).to(DEV)
    model.load_state_dict({k: torch.from_numpy(gd[k]) for k in model.state_dict()})
    before = {k: v.clone() for k, v in model.state_dict().items()}
    opt = torch.optim.Adam(model.parameters(), lr=1e-2)
    labels = cuda(gd["labels"])
    for step in range(3):
        b = Fn.dedup_layer_nodes(g, list(range(20, 28)), 2, 4, seed=100 + step)
        opt.zero_grad()
        _, logits = model.forward_sampled(table, b)
        loss = torch.nn.functional.cross_entropy(logits, labels)
        loss.backward()
        opt.step()
        assert np.isfinite(loss.item())
    for k, v in model.state_dict().items():
        assert torch.isfinite(v).all() and not torch.equal(v, before[k]), k
