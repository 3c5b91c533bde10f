"""Oracle: the per-layer node sets and index maps of the de-duplicating GraphSAGE collate
(GraphSAGE/data_utils.py:82-117 `get_layer_adj_nodes`, and the outermost draws of its collate_fn :154-162;
SURVEY.md §3.4)."""
import numpy as np


def layer_adj_nodes_v2(adj_lists, batch, num_layers, k, draws):
    """get_layer_adj_nodes with the sampled draws passed in: draws(l, nodes) returns the k neighbour ids drawn for
    every node of S_l (a [len(nodes), k] array-like, draw order), so the device sampler's draws can be replayed.
    The single deviation from the reference: every union S_i = S_{i+1} ∪ draws(i+1, S_{i+1}) is sorted ascending,
    where the reference iterates a CPython set (hash order).  The batch S_{L-1} keeps its order.

    Returns (nodes, center_map, neigh_map, outer): nodes[l] the ids of S_l; center_map int64 [L-1, n0] and
    neigh_map int64 [L-1, n0, k] in the reference's layout (positions in S_i of S_{i+1} and of its draws, rows past
    |S_{i+1}| all -1); outer int64 [n0, k] = draws(0, S_0), the neighbours whose features the collate gathers."""
    nodes = [[int(v) for v in batch]]
    samples = []
    for level in range(num_layers - 1, 0, -1):
        d = _checked(adj_lists, nodes[0], k, draws(level, nodes[0]))
        samples.insert(0, d)
        nodes.insert(0, sorted(set(nodes[0]) | set(d.reshape(-1).tolist())))
    n0 = len(nodes[0])
    center_map = np.full((num_layers - 1, n0), -1, np.int64)
    neigh_map = np.full((num_layers - 1, n0, k), -1, np.int64)
    for i in range(num_layers - 1):
        pos = {v: p for p, v in enumerate(nodes[i])}
        for r, v in enumerate(nodes[i + 1]):
            center_map[i, r] = pos[v]
            neigh_map[i, r] = [pos[u] for u in samples[i][r].tolist()]
    outer = _checked(adj_lists, nodes[0], k, draws(0, nodes[0]))
    return [np.asarray(s, np.int64) for s in nodes], center_map, neigh_map, outer


def _checked(adj_lists, nodes, k, d):
    """The draws as int64 [len(nodes), k]; each must be a neighbour of its node (data_utils.py:91-94)."""
    d = np.asarray(d, np.int64).reshape(len(nodes), k)
    for v, row in zip(nodes, d.tolist()):
        if not set(row) <= set(adj_lists[v]):
            raise ValueError(f"draws of node {v} are not all its neighbours: {row}")
    return d
