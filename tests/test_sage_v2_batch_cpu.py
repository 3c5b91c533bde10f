"""The de-duplicating GraphSAGE batch layout (GraphSAGE/data_utils.py:82-162) restated by
`oracle.sage_dedup.layer_adj_nodes_v2`, held to the reference collate's own batch in tests/golden/sage_v2_small.npz:
the node ids behind that batch are recovered by matching feature rows against the table, the golden's draws are
replayed, and the maps must agree up to the order of each node set (ascending here, CPython set order there)."""
import numpy as np
import pytest

from conftest import load_golden
from graphneuralnetwork_b200 import synthetic as S
from oracle.sage_dedup import layer_adj_nodes_v2

N, FEAT, L, K = 300, 64, 2, 4
BATCH = list(range(20, 28))


def _ids_of(rows, table):
    """Node id of every feature row (the table's rows are distinct standard-normal draws)."""
    lookup = {table[i].tobytes(): i for i in range(table.shape[0])}
    return np.asarray([lookup[r.tobytes()] for r in np.ascontiguousarray(rows)], np.int64)


@pytest.fixture(scope="module")
def recovered():
    g = load_golden("sage_v2_small.npz")
    table = np.random.default_rng(10).standard_normal((N, FEAT), dtype=np.float32)
    s0 = _ids_of(g["center_feats"], table)
    outer = _ids_of(g["neigh_feats"].reshape(-1, FEAT), table).reshape(len(s0), K)
    return g, s0, outer


def test_golden_ids_are_recovered(recovered):
    g, s0, outer = recovered
    assert len(s0) == len(set(s0.tolist())) == g["center_map"].shape[1] == 37
    n1 = int((g["center_map"][0] != -1).sum())
    assert n1 == len(BATCH) and s0[g["center_map"][0][:n1]].tolist() == BATCH  # the batch keeps its order
    adj = S.adjacency_lists(N, 6, seed=9)
    for v, row in zip(s0.tolist(), outer.tolist()):
        assert set(row) <= adj[v]


def test_oracle_reproduces_golden_maps_up_to_set_order(recovered):
    g, s0, outer = recovered
    adj = S.adjacency_lists(N, 6, seed=9)
    cmap, nmap = g["center_map"], g["neigh_map"]
    n1 = len(BATCH)
    inner = {v: s0[nmap[0][r]] for r, v in enumerate(BATCH)}  # the golden's draws for S_1, in draw order
    outer_of = dict(zip(s0.tolist(), outer))

    def draws(level, nodes):
        return [(inner if level == 1 else outer_of)[v] for v in nodes]

    nodes, cm, nm, out = layer_adj_nodes_v2(adj, BATCH, L, K, draws)
    assert nodes[1].tolist() == BATCH
    assert sorted(s0.tolist()) == nodes[0].tolist()  # same set, ascending
    assert cm.shape == cmap.shape and nm.shape == nmap.shape
    # the same -1 padding shape
    assert np.array_equal(cm == -1, cmap == -1) and np.array_equal(nm == -1, nmap == -1)
    # the same id behind every map entry
    assert np.array_equal(nodes[0][cm[0][:n1]], s0[cmap[0][:n1]])
    assert np.array_equal(nodes[0][nm[0][:n1]], s0[nmap[0][:n1]])
    # the outermost draws follow the set's order
    assert np.array_equal(out, np.stack([outer_of[v] for v in nodes[0].tolist()]))


def _adj(n):
    return {i: {(i + 1) % n, (i + 2) % n} for i in range(n)}


def test_oracle_single_node():
    adj = _adj(5)
    nodes, cm, nm, out = layer_adj_nodes_v2(adj, [3], 1, 2, lambda l, v: [[4, 0] for _ in v])
    assert [x.tolist() for x in nodes] == [[3]] and cm.shape == (0, 1) and nm.shape == (0, 1, 2)
    assert out.tolist() == [[4, 0]]
    nodes, cm, nm, out = layer_adj_nodes_v2(adj, [3], 2, 2, lambda l, v: [sorted(adj[x]) for x in v])
    assert [x.tolist() for x in nodes] == [[0, 3, 4], [3]]
    assert cm.tolist() == [[1, -1, -1]]
    assert nm.tolist() == [[[0, 2], [-1, -1], [-1, -1]]]
    assert out.tolist() == [[1, 2], [0, 4], [0, 1]]


def test_oracle_k_larger_than_degree_and_duplicate_draws():
    """k above the degree draws with replacement (the device sampler's rule): repeats stay in the map rows, once in
    the set; a draw that is already in the batch maps onto the batch's own position."""
    adj = _adj(6)
    d = {0: [1, 1, 2, 1], 1: [2, 3, 3, 2]}
    nodes, cm, nm, out = layer_adj_nodes_v2(adj, [1, 0], 2, 4, lambda l, v: [d[x] if l == 1 else [adj[x].copy().pop()] * 4
                                                                               for x in v])
    assert nodes[0].tolist() == [0, 1, 2, 3] and nodes[1].tolist() == [1, 0]
    assert cm.tolist() == [[1, 0, -1, -1]]
    assert nm[0, :2].tolist() == [[2, 3, 3, 2], [1, 1, 2, 1]]
    assert (nm[0, 2:] == -1).all()
    assert out.shape == (4, 4)


def test_oracle_refuses_draws_that_are_not_neighbours():
    with pytest.raises(ValueError):
        layer_adj_nodes_v2(_adj(4), [0], 2, 1, lambda l, v: [[3] for _ in v])
