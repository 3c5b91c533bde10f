"""GTN_Model on a RelationStack (sparse learned metapath composition) against the reference's golden and against the
dense drop-in on the device: logits, every parameter gradient, Adam steps; stack construction; no host reads in a
step once the stack's patterns are cached."""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_err
from graphneuralnetwork_b200 import _lib, layers
from graphneuralnetwork_b200.graph import CSRGraph
from graphneuralnetwork_b200.layers.gtn import RelationStack

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
TOL32 = 1e-5
TOL_GRAD = 2e-5  # the gradient tolerance of test_gpu_parity.py::test_gtn_dropin_vs_reference_golden


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _golden_model(g):
    model = layers.GTN_Model(4, 2, 12, 8, 3, 2, True)
    sd = {k: torch.from_numpy(g["param." + k]) for k in model.state_dict().keys()}
    model.load_state_dict(sd, strict=True)
    return model.to(DEV)


def test_golden_logits_and_gradients():
    g = load_golden("gtn_small.npz")
    model = _golden_model(g)
    stack = RelationStack.from_dense(cuda(g["A"]))
    before = _lib.launch_count()
    y, Ws = model(stack, cuda(g["X"]), cuda(g["target"]))
    assert _lib.launch_count() > before
    assert rel_err(y.detach().cpu().numpy(), g["y"]) < TOL32 and len(Ws) == 2 and len(Ws[0]) == 2
    torch.nn.functional.cross_entropy(y, cuda(g["labels"])).backward()
    for name, p in model.named_parameters():
        if f"grad.{name}" not in g:  # `bias` is declared but never used by the reference forward
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, name
            continue
        assert p.grad is not None, name
        assert rel_err(p.grad.cpu().numpy(), g[f"grad.{name}"]) < TOL_GRAD, name


def _random_dense(seed, n, K):
    """Power-law relations plus a cycle in each, so that no column of an off-diagonal H is empty: the dense model's
    `norm` turns an empty column into a NaN gradient (pow(-1) at 0 in its backward), the sparse one has no entry there."""
    rng = np.random.default_rng(seed)
    A = np.zeros((n, n, K), np.float32)
    for k in range(K - 1):
        deg = np.minimum((rng.pareto(2.0, n) * 1.5).astype(int), 200)
        rows = np.repeat(np.arange(n), deg)
        A[rows, rng.integers(0, n, len(rows)), k] = rng.uniform(0.2, 1.0, len(rows)).astype(np.float32)
        perm = rng.permutation(n)
        A[perm, np.roll(perm, 1), k] = rng.uniform(0.2, 1.0, n).astype(np.float32)  # a cycle: no empty column
    A[:, :, K - 1] = np.eye(n, dtype=np.float32)
    return A


def _pair(seed, n, K, C, L):
    torch.manual_seed(seed)
    dense = layers.GTN_Model(K, C, 16, 8, 4, L, True).to(DEV)
    for m in dense.modules():
        if isinstance(m, layers.GTConv):
            torch.nn.init.normal_(m.weight, std=0.5)
    sparse = layers.GTN_Model(K, C, 16, 8, 4, L, True).to(DEV)
    sparse.load_state_dict(dense.state_dict())
    return dense, sparse


@pytest.mark.parametrize("L", [1, 2, 3])
def test_random_stack_matches_dense_dropin(L):
    n, K, C = 2000, 5, 2
    A = cuda(_random_dense(L, n, K))
    X = torch.randn(n, 16, generator=torch.Generator().manual_seed(L)).to(DEV)
    target = torch.arange(0, n, 7, device=DEV)
    labels = torch.randint(0, 4, (target.numel(),), generator=torch.Generator().manual_seed(9)).to(DEV)
    dense, sparse = _pair(L, n, K, C, L)
    stack = RelationStack.from_dense(A)
    yd, _ = dense(A, X, target)
    ys, _ = sparse(stack, X, target)
    assert rel_err(ys.detach().cpu().numpy(), yd.detach().cpu().numpy()) < TOL32
    torch.nn.functional.cross_entropy(yd, labels).backward()
    torch.nn.functional.cross_entropy(ys, labels).backward()
    for (name, pd), (_, ps) in zip(dense.named_parameters(), sparse.named_parameters()):
        if pd.grad is None:
            assert ps.grad is None or float(ps.grad.abs().max()) == 0.0, name
            continue
        assert rel_err(ps.grad.cpu().numpy(), pd.grad.cpu().numpy()) < TOL_GRAD, name


def test_adam_steps_agree():
    g = load_golden("gtn_small.npz")
    dense, sparse = _golden_model(g), _golden_model(g)
    A, X, target, labels = cuda(g["A"]), cuda(g["X"]), cuda(g["target"]), cuda(g["labels"])
    stack = RelationStack.from_dense(A)
    for model, adj in ((dense, A), (sparse, stack)):
        opt = torch.optim.Adam(model.parameters(), lr=0.005, weight_decay=0.001)
        for _ in range(5):
            opt.zero_grad()
            y, _ = model(adj, X, target)
            torch.nn.functional.cross_entropy(y, labels).backward()
            opt.step()
    for (name, pd), (_, ps) in zip(dense.named_parameters(), sparse.named_parameters()):
        assert float((pd - ps).abs().max()) <= 1e-4, name


def test_stack_construction_and_refusals():
    A = _random_dense(4, 300, 4)
    s1 = RelationStack.from_dense(cuda(A))
    graphs = []
    for k in range(4):
        rows, cols = np.nonzero(A[:, :, k])
        g = CSRGraph.from_coo(cuda(rows), cuda(cols), cuda(A[rows, cols, k]), 300, 300)
        graphs.append(g)
    s2 = RelationStack.from_relations(graphs)
    assert torch.equal(s1.U.rowptr, s2.U.rowptr) and torch.equal(s1.U.col, s2.U.col)
    assert torch.equal(s1.V, s2.V) and s1.num_edge == s2.num_edge == 4
    P = s1.patterns(2)[0]
    small = RelationStack.from_dense(cuda(A), max_nnz=P[1].nnz - 1)
    small.patterns(1)
    with pytest.raises(_lib.GnnError, match="max_nnz"):
        small.patterns(2)
    model = layers.GTN_Model(5, 2, 16, 8, 4, 1, True).to(DEV)
    with pytest.raises(ValueError, match="edge types"):
        model(s1, torch.zeros(300, 16, device=DEV), torch.arange(3, device=DEV))
    with pytest.raises(ValueError):
        RelationStack.from_relations([graphs[0], CSRGraph(graphs[1].rowptr, graphs[1].col, None, 300, 301)])
    bad = CSRGraph(graphs[0].rowptr, graphs[0].col.clone(), None, 300, 300)
    bad.col[0] = 300
    with pytest.raises(IndexError):
        RelationStack.from_relations([bad, graphs[1]])
    with pytest.raises(ValueError):
        RelationStack.from_dense(cuda(A[:, :10]))


def test_step_reads_nothing_back_once_cached():
    g = load_golden("gtn_small.npz")
    model = _golden_model(g)
    stack = RelationStack.from_dense(cuda(g["A"]))
    X, target, labels = cuda(g["X"]), cuda(g["target"]), cuda(g["labels"])
    stack.patterns(2)
    stack.gcn_pattern(2)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        y, _ = model(stack, X, target)
        torch.nn.functional.cross_entropy(y, labels).backward()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
