"""GTN over a row partition on the device: the ordered row reduction (gnn_peer_reduce_rows_f32) against sequential
fp32 adds in rank order, bit for bit, with its untouched columns and rows; a PartitionedRelationStack of one rank
against GTN_Model on the whole RelationStack (logits, every gradient and 3 Adam steps bit-identical); the refusals;
and two real ranks through tools/gtn_dist_train.py --check."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from graphneuralnetwork_b200 import _lib, layers
from graphneuralnetwork_b200.functional import peer_reduce_rows_raw
from graphneuralnetwork_b200.layers.gtn import RelationStack
from graphneuralnetwork_b200.partition import PartitionedRelationStack

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
SENTINEL = -12345.5


@pytest.mark.parametrize("P", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("F, ld, ld_out", [(8, 8, 8), (13, 16, 20), (7, 9, 7), (6, 7, 11), (1, 1, 3)])
@pytest.mark.parametrize("relu", [False, True])
def test_reduce_rows_matches_sequential_fp32_adds(P, F, ld, ld_out, relu):
    rows = 97
    g = torch.Generator(device=DEV).manual_seed(P * 100 + F)
    srcs = [torch.randn(rows, ld, device=DEV, generator=g) * (q + 1) for q in range(P)]
    for lo, hi in ((0, rows), (13, 58), (96, 97), (40, 40)):
        ref = srcs[0][lo:hi, :F].clone()
        for s in srcs[1:]:
            ref = ref + s[lo:hi, :F]  # ((s0 + s1) + s2) + ...
        if relu:
            ref = torch.relu(ref)
        out = torch.full((hi - lo + 3, ld_out), SENTINEL, device=DEV)
        peer_reduce_rows_raw([s.data_ptr() for s in srcs], ld, F, lo, hi, out, relu)
        assert torch.equal(out[:hi - lo, :F], ref)
        assert bool((out[:hi - lo, F:] == SENTINEL).all()) and bool((out[hi - lo:] == SENTINEL).all())


def test_reduce_rows_unaligned_sources_take_the_scalar_path():
    base = torch.randn(4 * 65 + 1, device=DEV)
    a, b = base[1:].view(65, 4), torch.randn(65, 4, device=DEV)  # a starts 4 bytes past a 16-byte boundary
    out = torch.full((65, 4), SENTINEL, device=DEV)
    peer_reduce_rows_raw([a.data_ptr(), b.data_ptr()], 4, 4, 0, 65, out)
    assert torch.equal(out, a + b)


def _golden_stack():
    g = load_golden("gtn_small.npz")
    return (RelationStack.from_dense(torch.from_numpy(g["A"]).to(DEV)), torch.from_numpy(g["X"]).to(DEV),
            torch.from_numpy(g["target"]).to(DEV), torch.from_numpy(g["labels"]).to(DEV), 4, 3)


def _random_stack(seed, n=1500, K=5):
    """Power-law relations with a cycle each (no empty column of an off-diagonal H) plus the identity."""
    rng = np.random.default_rng(seed)
    A = np.zeros((n, n, K), np.float32)
    for k in range(K - 1):
        deg = np.minimum((rng.pareto(2.0, n) * 1.5).astype(int), 150)
        r = np.repeat(np.arange(n), deg)
        A[r, rng.integers(0, n, len(r)), k] = rng.uniform(0.2, 1.0, len(r))
        perm = rng.permutation(n)
        A[perm, np.roll(perm, 1), k] = rng.uniform(0.2, 1.0, n)
    A[:, :, K - 1] = np.eye(n, dtype=np.float32)
    X = torch.randn(n, 12, generator=torch.Generator().manual_seed(seed)).to(DEV)
    target = torch.arange(0, n, 5, device=DEV)
    labels = torch.randint(0, 3, (target.numel(),), generator=torch.Generator().manual_seed(seed + 1)).to(DEV)
    return RelationStack.from_dense(torch.from_numpy(A).to(DEV)), X, target, labels, K, 3


def _models(K, L, w_in, classes, seed):
    torch.manual_seed(seed)
    a = layers.GTN_Model(K, 2, w_in, 8, classes, L, True)
    for m in a.modules():
        if isinstance(m, layers.GTConv):
            torch.nn.init.normal_(m.weight, std=0.5)
    b = layers.GTN_Model(K, 2, w_in, 8, classes, L, True)
    b.load_state_dict(a.state_dict())
    return a.to(DEV), b.to(DEV)


def _train(model, adj, X, target, labels, steps=3):
    opt = torch.optim.Adam(model.parameters(), lr=0.005, weight_decay=1e-3)
    first = None
    for s in range(steps):
        opt.zero_grad(set_to_none=True)
        y, Ws = model(adj, X, target)
        torch.nn.functional.cross_entropy(y, labels).backward()
        if s == 0:
            first = (y.detach().clone(), {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None},
                     [[w.clone() for w in W] for W in Ws])
        opt.step()
    return first, {k: v.detach().clone() for k, v in model.state_dict().items()}


@pytest.mark.parametrize("which", ["golden", "random"])
@pytest.mark.parametrize("L", [1, 2, 3])
def test_world_one_is_bit_identical_to_the_whole_stack(which, L):
    stack, X, target, labels, K, classes = _golden_stack() if which == "golden" else _random_stack(L)
    whole, part = _models(K, L, X.shape[1], classes, 7 + L)
    ps = PartitionedRelationStack(stack, 0, 1, L, 2 * 8)
    assert ps.bounds == [0, stack.n] and ps.n_local == stack.n and ps.row_range == (0, stack.n)
    assert ps.nnz_per_layer == [P.nnz for P in stack.patterns(L)[0]]
    (y1, g1, W1), w1 = _train(whole, stack, X, target, labels)
    (y2, g2, W2), w2 = _train(part, ps, X, target, labels)
    assert torch.equal(y1, y2)
    assert g1.keys() == g2.keys()
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k
    for k in w1:
        assert torch.equal(w1[k], w2[k]), k
    assert all(torch.equal(a, b) for A, B in zip(W1, W2) for a, b in zip(A, B))
    ps.check_status()
    ps.close()


def test_world_one_step_reads_nothing_back():
    stack, X, target, labels, K, classes = _golden_stack()
    _, model = _models(K, 2, X.shape[1], classes, 3)
    ps = PartitionedRelationStack(stack, 0, 1, 2, 16)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        y, _ = model(ps, X, target)
        torch.nn.functional.cross_entropy(y, labels).backward()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()


@pytest.mark.parametrize("C", [1, 2])
def test_empty_block_gcn_tail_takes_part_in_the_reduce(C):
    """A rank whose row block is empty: its gcn_conv pattern is [n, 0] with [0, C] values.  The normalise-and-aggregate
    tail still hands its (zero) partial degrees to the reduce, as every rank must, and returns a zero partial output;
    the backward gives empty value and XW gradients.  norm's column sums over the empty D_l reach the reduce too."""
    from graphneuralnetwork_b200.functional import column_normalize
    from graphneuralnetwork_b200.graph import CSRGraph
    from graphneuralnetwork_b200.layers.gtn import _gcn_pattern, _normalized_aggregate
    n, w = 50, 8
    D = CSRGraph(torch.zeros(1, dtype=torch.int64, device=DEV), torch.zeros(0, dtype=torch.int32, device=DEV), None,
                 0, n)
    g, src, diag = _gcn_pattern(D, torch.zeros(0, dtype=torch.int64, device=DEV), n, n)
    assert (g.n_rows, g.n_cols, g.nnz, src.numel(), diag.numel()) == (n, 0, 0, 0, 0)
    vals = torch.zeros((0, C), device=DEV, requires_grad=True)
    XW = torch.zeros((0, w), device=DEV, requires_grad=True)
    seen = []

    def reduce(x):
        seen.append(x.detach().clone())
        return x

    Y = _normalized_aggregate(g, vals, XW, reduce=reduce)
    assert len(seen) == 1 and seen[0].shape == (n, C) and not seen[0].any()
    assert Y.shape == (n, C * w) and not Y.any()
    dv, dx = torch.autograd.grad(Y, (vals, XW), torch.randn_like(Y))
    assert dv.shape == (0, C) and dx.shape == (0, w)
    Hn = column_normalize(D, vals, reduce=reduce)
    assert len(seen) == 2 and seen[1].shape == (n, C) and not seen[1].any() and Hn.shape == (0, C)
    assert torch.autograd.grad(Hn.sum(), vals)[0].shape == (0, C)


def test_refusals():
    stack, X, target, _, K, classes = _golden_stack()
    ps = PartitionedRelationStack(stack, 0, 1, 2, 16)
    with pytest.raises(ValueError, match="layers"):
        _models(K, 1, X.shape[1], classes, 0)[1](ps, X, target)        # 1 layer, the stack has 2
    with pytest.raises(ValueError, match="edge types"):
        _models(K + 1, 2, X.shape[1], classes, 0)[1](ps, X, target)
    wide = layers.GTN_Model(K, 2, X.shape[1], 16, classes, 2, True).to(DEV)  # width 32, the stack 16
    with pytest.raises(ValueError, match="width"):
        wide(ps, X, target)
    with pytest.raises(ValueError, match="X_local"):
        _models(K, 2, X.shape[1], classes, 0)[1](ps, X[1:], target)
    with pytest.raises(ValueError):
        PartitionedRelationStack(stack, 0, 1, 0, 16)
    nnz = sum(P.nnz for P in stack.patterns(2)[0])
    PartitionedRelationStack(stack, 0, 1, 2, 16, max_nnz_per_rank=nnz).close()
    with pytest.raises(_lib.GnnError, match="PartitionedRelationStack: .*max_nnz_per_rank"):
        PartitionedRelationStack(stack, 0, 1, 2, 16, max_nnz_per_rank=nnz - 1)
    ps.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one node")
def test_two_rank_gtn_training_check():
    """Two real ranks train GTN on a PartitionedRelationStack (DBLP-shaped stack at 1/20 scale, C = 2, 1 to 3 layers);
    every rank compares its rows of the logits, the step-1 gradients and the weights after 3 Adam steps with the same
    model trained on the whole stack on one GPU, repeats the run bit for bit, and runs one step without host reads."""
    import json
    import os
    import socket
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(root, "tools", "gtn_dist_train.py"), "--check"]
    out = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 2 * 3, out.stdout[-2000:]  # ranks x layer counts
    for d in lines:
        tag = (d["layers"], d["rank"])
        assert d["logits_rel_err"] <= 1e-5 and d["grad_rel_err"] <= 5e-5, (tag, d)
        assert d["weights_rel_err"] <= 1e-4 and d["bitwise_repeat"] and d["step_without_host_reads"], (tag, d)
