"""HAN's metapath composition on the device: `CSRGraph.pattern_product` / `metapath` against the scipy restatement
(oracle/metapath.py, HAN/utils/data_utils.py:85-89) bit for bit, every kernel path forced through the tuning keys,
repeats, the refusals, and `PartitionedMetapaths.from_relations` against `from_global` on one and two ranks."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import ROOT
from graphneuralnetwork_b200 import _lib
from graphneuralnetwork_b200.graph import CSRGraph
from oracle import metapath as O

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
KEYS = ("metapath.small_max", "metapath.medium_max", "metapath.tile_cols")
# (small_max, medium_max, tile_cols): the defaults, then every row forced onto one path; the bitmap runs with a
# 64-column tile, so every n_b below is several tiles wide, and with the widest tile
ROUTES = {"default": None, "small": (256, 8192, 0), "medium": (-1, 8192, 0), "large": (-1, -1, 64),
          "large_wide": (-1, -1, 0)}


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


def _csr(rows, cols, shape, shuffle_seed=None, repeat=False):
    """Pattern CSR with the ids of every row as given (unsorted, repeated), on the device."""
    rows, cols = np.asarray(rows, np.int64), np.asarray(cols, np.int64)
    order = np.argsort(rows, kind="stable")
    rows, cols = rows[order], cols[order]
    indptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=shape[0]))]).astype(np.int64)
    if shuffle_seed is not None:
        rng = np.random.default_rng(shuffle_seed)
        for i in range(shape[0]):
            rng.shuffle(cols[indptr[i]:indptr[i + 1]])
    g = CSRGraph(torch.from_numpy(indptr).to(DEV), torch.from_numpy(cols.astype(np.int32)).to(DEV), None, *shape)
    return g, indptr, cols


def _inputs(seed, n_a, k, n_b, hub_deg):
    """A with ragged rows, empty rows, repeated and unsorted ids; B with rows of degree 0 and hub rows."""
    rng = np.random.default_rng(seed)
    ar, ac = [], []
    for i in range(n_a):
        if i % 7 == 3:
            continue  # empty row of A
        d = int(rng.integers(1, 6)) if i % 11 else int(rng.integers(20, 60))
        ids = rng.integers(0, k, d)
        if i % 5 == 0:
            ids = np.concatenate([ids, ids[:2]])  # repeats
        if i % 13 == 0:
            ids = np.append(ids, rng.integers(0, 2))  # hub rows of B
        ar += [i] * len(ids)
        ac += list(ids)
    br, bc = [], []
    for x in range(k):
        if x % 6 == 5:
            continue  # degree 0
        d = hub_deg if x < 2 else int(rng.integers(1, 9))
        ids = rng.integers(0, n_b, d)
        br += [x] * len(ids)
        bc += list(ids)
    return _csr(ar, ac, (n_a, k), shuffle_seed=seed), _csr(br, bc, (k, n_b), shuffle_seed=seed + 1)


def _expect(A, B, rng_, loops):
    (_, ai, ac), (_, bi, bc) = A, B
    return O.pattern_product(ai, ac, bi, bc, A[0].n_rows, A[0].n_cols, B[0].n_cols, rng_, loops)


CASES = [(0, 300, 90, 300, 400), (1, 257, 40, 5000, 3000), (2, 64, 500, 64, 50), (3, 1, 3, 1, 2)]


@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("case", CASES)
def test_pattern_product_matches_scipy_every_path(route, case):
    seed, n_a, k, n_b, hub = case
    A, B = _inputs(seed, n_a, k, n_b, hub)
    _route(route)
    ranges = [None, (n_a // 3, n_a - n_a // 4), (n_a // 2, n_a // 2), (n_a - 1, n_a)]
    seen = torch.zeros(3, dtype=torch.int64)
    for loops in ([False, True] if n_a == n_b else [False]):
        for rr in ranges:
            path_rows = torch.zeros(3, dtype=torch.int64, device=DEV)
            g = CSRGraph.pattern_product(A[0], B[0], row_range=rr, self_loops=loops, path_rows=path_rows)
            ip, ix = _expect(A, B, rr, loops)
            assert torch.equal(g.rowptr.cpu(), torch.from_numpy(ip)), (route, rr, loops)
            assert torch.equal(g.col.cpu(), torch.from_numpy(ix)), (route, rr, loops)
            lo, hi = (0, n_a) if rr is None else rr
            assert g.n_rows == hi - lo and g.n_cols == n_b and g.val is None
            assert int(path_rows.sum()) == hi - lo
            seen += path_rows.cpu()
            again = CSRGraph.pattern_product(A[0], B[0], row_range=rr, self_loops=loops)
            assert torch.equal(again.rowptr, g.rowptr) and torch.equal(again.col, g.col)
    if route == "small":
        assert seen[0] > 0
    elif route == "medium":  # the warp sort is off: rows up to 8192 products take the CTA sort
        assert seen[0] == 0 and seen[1] > 0
    elif route.startswith("large"):
        assert seen[2] == seen.sum()


def test_default_routing_takes_every_path():
    # hub rows of B with 3000 and 12000 products: rows through the warp sort, the CTA sort and the bitmap; the
    # bitmap's B is 2 M columns wide, more than one tile of the default (widest) width
    A, B = _inputs(5, 400, 60, 20000, 3000)
    n_hub = 2_000_000
    hub = _csr(np.zeros(12000, np.int64), np.random.default_rng(1).integers(0, n_hub, 12000), (1, n_hub))
    one = _csr(np.arange(400), np.zeros(400, np.int64), (400, 1))
    path_rows = torch.zeros(3, dtype=torch.int64, device=DEV)
    for a, b in ((A, B), (one, hub)):
        pr = torch.zeros(3, dtype=torch.int64, device=DEV)
        g = CSRGraph.pattern_product(a[0], b[0], path_rows=pr)
        ip, ix = O.pattern_product(a[1], a[2], b[1], b[2], 400, b[0].n_rows, b[0].n_cols)
        assert torch.equal(g.rowptr.cpu(), torch.from_numpy(ip)) and torch.equal(g.col.cpu(), torch.from_numpy(ix))
        path_rows += pr
    assert all(int(v) > 0 for v in path_rows.cpu()), path_rows


def test_acm_relations_compose_to_the_scipy_metapaths():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from han_dist_train import acm_like_metapaths
    from metapath_build import acm_like_relations
    want = acm_like_metapaths(DEV)
    for R, g in zip(acm_like_relations(DEV), want):
        got = CSRGraph.metapath(R, self_loops=True)
        assert torch.equal(got.rowptr, g.rowptr) and torch.equal(got.col, g.col)
        assert (got.n_rows, got.n_cols) == (g.n_rows, g.n_cols)
        again = CSRGraph.metapath(R, self_loops=True)
        assert torch.equal(again.col, got.col)


def test_metapath_matches_dense_reference_form():
    rng = np.random.default_rng(3)
    P = (rng.random((120, 30)) < 0.05).astype(np.float64)
    R = sp.csr_matrix(P)
    g = CSRGraph.metapath(_csr(*np.nonzero(P), (120, 30))[0])
    dense = torch.from_numpy((P @ P.T > 0).astype(np.float64)).to(DEV)
    want = CSRGraph.from_dense_mask(dense)  # the reference's float64 mask, through the existing device builder
    assert torch.equal(g.rowptr, want.rowptr) and torch.equal(g.col, want.col)
    ip, ix = O.metapath(R.indptr, R.indices, 120, 30)
    assert torch.equal(g.col.cpu(), torch.from_numpy(ix))


def test_refusals():
    A, B = _inputs(0, 50, 20, 60, 30)
    g = CSRGraph.pattern_product(A[0], B[0])
    with pytest.raises(_lib.GnnError, match=f"{g.nnz} entries.*max_nnz = {g.nnz - 1}.*bytes"):
        CSRGraph.pattern_product(A[0], B[0], max_nnz=g.nnz - 1)
    assert CSRGraph.pattern_product(A[0], B[0], max_nnz=g.nnz).nnz == g.nnz
    bad_a = CSRGraph(A[0].rowptr, A[0].col.clone(), None, 50, 20)
    bad_a.col[3] = 20
    with pytest.raises(IndexError):
        CSRGraph.pattern_product(bad_a, B[0])
    with pytest.raises(IndexError):  # checked before the transpose sorts by the bad id
        CSRGraph.metapath(bad_a)
    bad_b = CSRGraph(B[0].rowptr, B[0].col.clone(), None, 20, 60)
    bad_b.col[-1] = -1
    with pytest.raises(IndexError):
        CSRGraph.pattern_product(A[0], bad_b)
    # unvalidated, the kernels skip the ids outside the columns and read nothing out of bounds
    skipped = CSRGraph.pattern_product(A[0], bad_b, validate=False)
    assert skipped.nnz <= g.nnz
    with pytest.raises(_lib.GnnError, match="not square"):
        CSRGraph.pattern_product(A[0], B[0], self_loops=True)
    with pytest.raises(IndexError):
        CSRGraph.pattern_product(A[0], B[0], row_range=(10, 51))
    with pytest.raises(_lib.GnnError, match="not on a CUDA device"):
        CSRGraph.pattern_product(A[0], _cpu(B[0]))


def _cpu(g):
    c = CSRGraph.__new__(CSRGraph)
    c.__dict__.update(vars(g))
    c.rowptr = g.rowptr.cpu()
    return c


def test_raw_abi_bad_arguments_return_status(lib):
    A, B = _inputs(0, 10, 5, 10, 4)
    ws = torch.empty(lib.gnn_pattern_product_count_workspace_size(10), dtype=torch.uint8, device=DEV)
    rp = torch.empty(11, dtype=torch.int64, device=DEV)
    args = [A[0].rowptr.data_ptr(), A[0].col.data_ptr(), 10, 5, B[0].rowptr.data_ptr(), B[0].col.data_ptr(), 10]
    s = torch.cuda.current_stream().cuda_stream
    assert lib.gnn_pattern_product_count(*args, 0, 11, 0, rp.data_ptr(), None, ws.data_ptr(), ws.numel(), s) == 1
    assert lib.gnn_pattern_product_count(*args, 0, 10, 0, None, None, ws.data_ptr(), ws.numel(), s) == 1
    assert lib.gnn_pattern_product_count(*args, 0, 10, 0, rp.data_ptr(), None, ws.data_ptr(), 16, s) == 5
    args[-1] = 11
    assert lib.gnn_pattern_product_count(*args, 0, 10, 1, rp.data_ptr(), None, ws.data_ptr(), ws.numel(), s) == 1
    args[-1] = 10
    assert lib.gnn_pattern_product_count(*args, 0, 10, 1, rp.data_ptr(), None, ws.data_ptr(), ws.numel(), s) == 0
    torch.cuda.synchronize()


def test_one_rank_from_relations_equals_from_global_and_han_logits():
    from graphneuralnetwork_b200.layers.han import HANModel
    from graphneuralnetwork_b200.partition import PartitionedMetapaths
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from metapath_build import acm_like_relations, same_partition
    rels = acm_like_relations(DEV, n=600)
    graphs = [CSRGraph.metapath(R, self_loops=True) for R in rels]
    M, H, Fp, F_in = len(rels), 4, 8, 32
    width = M * H * Fp
    a = PartitionedMetapaths.from_relations(rels, 0, 1, widths=[width])
    b = PartitionedMetapaths.from_global(graphs, 0, 1, widths=[width])
    assert same_partition(a, b)
    X = torch.randn(600, F_in, generator=torch.Generator().manual_seed(2)).to(DEV)
    torch.manual_seed(0)
    model = HANModel(M, F_in, Fp, 3, [H], 0.0).to(DEV).eval()
    with torch.no_grad():
        assert torch.equal(model(a, X), model(b, X))
    a.close()
    b.close()
    with pytest.raises(_lib.GnnError, match="max_nnz_per_rank"):
        PartitionedMetapaths.from_relations(rels, 0, 1, widths=[width], max_nnz_per_rank=sum(g.nnz for g in graphs) - 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one node")
def test_two_rank_metapath_build_check():
    """Two real ranks: device composition of the ACM-shaped relations against scipy's graphs, from_relations against
    from_global on the composed graphs, and a repeat, bit for bit on every rank."""
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tools", "metapath_build.py"), "--check"]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert sorted(d["rank"] for d in lines) == [0, 1], out.stdout[-2000:]
    for d in lines:
        assert d["pass"], d
