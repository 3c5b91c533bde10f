"""Value-carrying sparse products on the device (`functional.spgemm_values`, gnn_spgemm_values_f32 / _bwd_f32): the
forward and both gradients against float64 scipy element by element, on random and power-law operands at C = 1,
2 and 8, with every routing path forced through the tuning keys; the same bits on a repeat and on every path; the
refusals."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from graphneuralnetwork_b200 import _lib, functional as Fn
from graphneuralnetwork_b200.graph import CSRGraph
from oracle.gtn_sparse import values_on

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
KEYS = ("spgemm.warp_slots", "spgemm.warp_list")
ROUTES = {"default": None, "warp": (1 << 30, 1 << 30), "cta": (-1, -1)}


@pytest.fixture(autouse=True)
def _restore_keys(lib):
    saved = {k: _lib.get_tuning(k) for k in KEYS}
    yield
    for k, v in saved.items():
        _lib.set_tuning(k, v)


def _route(name):
    if ROUTES[name] is not None:
        for k, v in zip(KEYS, ROUTES[name]):
            _lib.set_tuning(k, v)


def _to_dev(M):
    M = sp.csr_matrix(M)
    M.sort_indices()
    return CSRGraph(torch.from_numpy(M.indptr.astype(np.int64)).to(DEV),
                    torch.from_numpy(M.indices.astype(np.int32)).to(DEV), None, *M.shape)


def _operands(seed, n_a, k, n_b, power_law):
    """Patterns of A [n_a, k] and B [k, n_b]: empty rows, A entries whose B row is empty, one hub row in each."""
    rng = np.random.default_rng(seed)

    def rand(n_r, n_c, mean, hub):
        deg = (rng.pareto(1.5, n_r) * mean).astype(np.int64) + 1 if power_law else rng.poisson(mean, n_r)
        deg = np.minimum(deg, n_c)
        deg[::9] = 0
        if hub < n_r:
            deg[hub] = min(n_c, 3000)
        rows = np.repeat(np.arange(n_r), deg)
        cols = np.concatenate([rng.choice(n_c, d, replace=False) for d in deg]) if deg.sum() else np.zeros(0, int)
        return sp.csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(n_r, n_c))

    A = rand(n_a, k, 4, 1)
    B = rand(k, n_b, 5, 2)
    B = sp.csr_matrix(B.multiply(np.arange(k)[:, None] % 7 != 3))  # rows of B without entries, still in A
    B.eliminate_zeros()
    return A, B


def _values(M, C, seed):
    return np.random.default_rng(seed).uniform(-1, 1, (M.nnz, C)).astype(np.float32)


def _check_bound(got, want, terms, absum):
    """|c - c64| <= n·2^-23·Σ|a·b| for an entry of n terms (any summation order)."""
    err = np.abs(got.astype(np.float64) - want)
    assert np.all(err <= terms * 2.0 ** -23 * absum), float((err - terms * 2.0 ** -23 * absum).max())


def _scipy(P, val):
    P = sp.csr_matrix(P)
    P.sort_indices()
    return sp.csr_matrix((val.astype(np.float64), P.indices, P.indptr), shape=P.shape)


CASES = [(0, 300, 200, 250, False), (1, 500, 400, 3500, True), (2, 1, 5, 3, False)]


@pytest.mark.parametrize("C", [1, 2, 8])
@pytest.mark.parametrize("case", CASES)
def test_forward_and_gradients_match_float64_on_every_path(case, C):
    seed, n_a, k, n_b, pl = case
    A, B = _operands(seed, n_a, k, n_b, pl)
    Ad, Bd = _to_dev(A), _to_dev(B)
    Cp = CSRGraph.pattern_product(Ad, Bd)
    a, b = _values(A, C, seed + 10), _values(B, C, seed + 20)
    Cpat = sp.csr_matrix((np.ones(Cp.nnz), Cp.col.cpu().numpy(), Cp.rowptr.cpu().numpy()), shape=(n_a, n_b))
    dc = _values(Cpat, C, seed + 30)
    At, Bt = sp.csr_matrix(A), sp.csr_matrix(B)
    ptrs = dict(c=(Cp.rowptr.cpu().numpy(), Cp.col.cpu().numpy()), a=(At.indptr, At.indices), b=(Bt.indptr, Bt.indices))
    want_c, want_da, want_db = [], [], []
    for ch in range(C):
        Ac, Bc, dCc = _scipy(A, a[:, ch]), _scipy(B, b[:, ch]), _scipy(Cpat, dc[:, ch])
        want_c.append((values_on(Ac @ Bc, *ptrs["c"]), values_on(abs(Ac) @ abs(Bc), *ptrs["c"])))
        want_da.append((values_on(dCc @ Bc.T, *ptrs["a"]), values_on(abs(dCc) @ abs(Bc).T, *ptrs["a"])))
        want_db.append((values_on(Ac.T @ dCc, *ptrs["b"]), values_on(abs(Ac).T @ abs(dCc), *ptrs["b"])))
    ones = lambda M: sp.csr_matrix((np.ones(M.nnz), M.indices, M.indptr), shape=M.shape)
    terms_c = values_on(ones(A) @ ones(B), *ptrs["c"])
    terms_a = values_on(ones(Cpat) @ ones(B).T, *ptrs["a"])
    terms_b = values_on(ones(A).T @ ones(Cpat), *ptrs["b"])
    av, bv, dcv = (torch.from_numpy(x).to(DEV) for x in (a, b, dc))
    results = {}
    for route in ROUTES:
        _route(route)
        pr, prb = (torch.zeros(n, dtype=torch.int64, device=DEV) for n in (2, 4))
        c = Fn.spgemm_values_raw(Ad, av, Bd, bv, Cp, path_rows=pr)
        da, db = Fn.spgemm_values_bwd_raw(Ad, av, Bd, bv, Cp, dcv, path_rows=prb)
        c2 = Fn.spgemm_values_raw(Ad, av, Bd, bv, Cp)
        da2, db2 = Fn.spgemm_values_bwd_raw(Ad, av, Bd, bv, Cp, dcv)
        assert torch.equal(c, c2) and torch.equal(da, da2) and torch.equal(db, db2)  # same bits on a repeat
        pr, prb = pr.cpu().tolist(), prb.cpu().tolist()
        assert sum(pr) == n_a and prb[0] + prb[1] == n_a and prb[2] + prb[3] == k
        if route == "warp":
            assert pr[1] == prb[1] == prb[3] == 0
        elif route == "cta":
            assert pr[0] == prb[0] == prb[2] == 0
        elif n_b > 1024:
            assert pr[0] > 0 and pr[1] > 0, pr  # the hub row of A takes a CTA, the short rows warps
        for ch in range(C):
            _check_bound(c[:, ch].cpu().numpy(), want_c[ch][0], terms_c, want_c[ch][1])
            _check_bound(da[:, ch].cpu().numpy(), want_da[ch][0], terms_a, want_da[ch][1])
            _check_bound(db[:, ch].cpu().numpy(), want_db[ch][0], terms_b, want_db[ch][1])
        results[route] = (c, da, db)
    # one thread sums each entry in ascending order of the inner index on both paths: the same bits
    for route in ROUTES:
        assert all(torch.equal(x, y) for x, y in zip(results[route], results["default"])), route


def test_autograd_reaches_both_value_tensors():
    A, B = _operands(3, 120, 90, 100, True)
    Ad, Bd = _to_dev(A), _to_dev(B)
    Cp = CSRGraph.pattern_product(Ad, Bd)
    av = torch.from_numpy(_values(A, 2, 1)).to(DEV).requires_grad_(True)
    bv = torch.from_numpy(_values(B, 2, 2)).to(DEV).requires_grad_(True)
    c = Fn.spgemm_values(Ad, av, Bd, bv, Cp)
    g = torch.randn_like(c)
    (c * g).sum().backward()
    da, db = Fn.spgemm_values_bwd_raw(Ad, av.detach(), Bd, bv.detach(), Cp, g)
    assert torch.equal(av.grad, da) and torch.equal(bv.grad, db)
    # the pattern is the pattern product's: every entry a product reaches, ascending
    M = (sp.csr_matrix(A) @ sp.csr_matrix(B)).tocsr()
    M.sort_indices()
    assert torch.equal(Cp.col.cpu(), torch.from_numpy(M.indices.astype(np.int32)))


def test_refusals(lib):
    A, B = _operands(4, 50, 40, 30, False)
    Ad, Bd = _to_dev(A), _to_dev(B)
    Cp = CSRGraph.pattern_product(Ad, Bd)
    a9, b9 = (torch.ones((g.nnz, 9), device=DEV) for g in (Ad, Bd))
    with pytest.raises(_lib.GnnError, match="unsupported shape"):
        Fn.spgemm_values(Ad, a9, Bd, b9, Cp)
    a2, b2 = (torch.ones((g.nnz, 2), device=DEV) for g in (Ad, Bd))
    with pytest.raises(_lib.GnnError, match="values"):
        Fn.spgemm_values(Ad, a2, Bd, b2[1:], Cp)
    with pytest.raises(_lib.GnnError, match="fp32"):
        Fn.spgemm_values(Ad, a2.double(), Bd, b2, Cp)
    with pytest.raises(_lib.GnnError, match="does not give"):
        Fn.spgemm_values(Ad, a2, Bd, b2, CSRGraph(Cp.rowptr, Cp.col, None, 50, 31))
    with pytest.raises(_lib.GnnError, match="not on a CUDA device"):
        Fn.spgemm_values(Ad, a2.cpu(), Bd, b2, Cp)
    # column ids of the output pattern outside the product's columns are skipped: those entries are 0
    bad = CSRGraph(Cp.rowptr, Cp.col.clone(), None, 50, 30)
    bad.col[0], bad.col[-1] = 30, -5
    out = Fn.spgemm_values_raw(Ad, a2, Bd, b2, bad)
    ref = Fn.spgemm_values_raw(Ad, a2, Bd, b2, Cp)
    assert float(out[0].abs().max()) == 0.0 and float(out[-1].abs().max()) == 0.0
    assert torch.equal(out[1:-1], ref[1:-1])
    # a short workspace
    Bt = Bd.transpose()
    ws = torch.empty(16, dtype=torch.uint8, device=DEV)
    c = torch.empty((Cp.nnz, 2), device=DEV)
    rc = lib.gnn_spgemm_values_f32(Ad.rowptr.data_ptr(), Ad.col.data_ptr(), a2.data_ptr(), 50, 40, Ad.nnz,
                                   Bt.rowptr.data_ptr(), Bt.col.data_ptr(), Bd.perm_t.data_ptr(), b2.data_ptr(), 30,
                                   Bd.nnz, Cp.rowptr.data_ptr(), Cp.col.data_ptr(), c.data_ptr(), 2, None,
                                   ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    assert rc == 5
    torch.cuda.synchronize()
