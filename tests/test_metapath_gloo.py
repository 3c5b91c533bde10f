"""Host logic of building HAN's metapath graphs one row block per rank (`partition.metapath_row_plan`, the collective
part of `PartitionedMetapaths.from_relations`), world_size 2 and 3 over gloo on CPU, with a scipy count standing in
for the device kernel: the even split and the exchange of per-row counts, the bounds (those `from_global` chooses for
the composed graphs), each rank's block rowptrs, and the collective `max_nnz_per_rank` refusal.  Also the C ABI's
argument checks of the pattern product, which return a status before any CUDA call."""
import os
import socket

import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from graphneuralnetwork_b200 import _lib
from graphneuralnetwork_b200.partition import balanced_bounds, metapath_row_plan, shard_bounds
from oracle import metapath as O


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _relations(n, seed):
    """Two relations over n nodes: ~3 of 2n authors per paper (a few hub authors) and one of 7 subjects; some
    papers have no author."""
    rng = np.random.default_rng(seed)
    rows, cols = [], []
    for i in range(n):
        k = int(rng.integers(0, 4))
        a = rng.integers(0, 2 * n, k)
        if rng.random() < 0.1:
            a = np.append(a, rng.integers(0, 3))  # hub authors 0..2
        rows += [i] * len(a)
        cols += list(a)
    pa = sp.csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(n, 2 * n))
    ps = sp.csr_matrix((np.ones(n), (np.arange(n), rng.integers(0, 7, n))), shape=(n, 7))
    return [pa, ps]


def _counter(rels, self_loops, calls):
    def count(m, lo, hi):
        R = rels[m]
        Rt = R.T.tocsr()
        calls.append((m, lo, hi))
        ip, _ = O.pattern_product(R.indptr, R.indices, Rt.indptr, Rt.indices, R.shape[0], R.shape[1], R.shape[0],
                                  (lo, hi), self_loops)
        return torch.from_numpy(ip)
    return count


def _check(rank, world, n, seed, self_loops):
    rels = _relations(n, seed)
    whole = [O.metapath(R.indptr, R.indices, n, R.shape[1], self_loops) for R in rels]
    calls = []
    bounds, rps = metapath_row_plan(_counter(rels, self_loops, calls), n, len(rels), rank, world)
    even = shard_bounds(n, world)
    assert calls == [(m, even[rank], even[rank + 1]) for m in range(len(rels))]  # only the rank's even rows
    assert bounds == balanced_bounds(torch.from_numpy(sum(ip for ip, _ in whole)), world)
    lo, hi = bounds[rank], bounds[rank + 1]
    for (ip, _), rp in zip(whole, rps):
        assert torch.equal(rp, torch.from_numpy(ip[lo:hi + 1] - ip[lo]))
    block_nnz = [sum(int(ip[bounds[p + 1]] - ip[bounds[p]]) for ip, _ in whole) for p in range(world)]
    # a limit every block meets passes; one below the largest block raises on every rank, naming that rank
    metapath_row_plan(_counter(rels, self_loops, []), n, len(rels), rank, world, max_nnz_per_rank=max(block_nnz))
    worst = int(np.argmax(block_nnz))
    with pytest.raises(_lib.GnnError, match=f"rank {worst}: {block_nnz[worst]}"):
        metapath_row_plan(_counter(rels, self_loops, []), n, len(rels), rank, world,
                          max_nnz_per_rank=max(block_nnz) - 1)
    return block_nnz


def _worker(rank, world, port, out_q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = [_check(rank, world, 301, 3, True), _check(rank, world, 97, 8, False), _check(rank, world, 2, 1, True)]
        dist.barrier()
        out_q.put((rank, "ok", res))
    except Exception:  # reported to the parent, which fails the test with it
        import traceback
        out_q.put((rank, traceback.format_exc(), None))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_metapath_row_plan_split_exchange_bounds_and_refusal(world):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for rank, status, _ in results:
        assert status == "ok", f"rank {rank}:\n{status}"
    for p in procs:
        assert p.exitcode == 0
    assert len({str(res) for _, _, res in results}) == 1  # every rank saw the same block sizes


def test_world_one_plan_is_the_whole_graph():
    rels = _relations(50, 4)
    bounds, rps = metapath_row_plan(_counter(rels, True, []), 50, 2, 0, 1)
    assert bounds == [0, 50]
    for R, rp in zip(rels, rps):
        ip, _ = O.metapath(R.indptr, R.indices, 50, R.shape[1], True)
        assert torch.equal(rp, torch.from_numpy(ip))


def test_oracle_matches_dense_reference_composition():
    """The restatement against the reference's dense float64 form (P·Pᵀ, binarised; + I for the training graphs)."""
    for R in _relations(40, 6):
        P = R.toarray()
        for loops in (False, True):
            dense = (P @ P.T + (np.eye(40) if loops else 0)) > 0
            ip, ix = O.metapath(R.indptr, R.indices, 40, R.shape[1], loops)
            rows, cols = np.nonzero(dense)
            assert np.array_equal(ip, np.concatenate([[0], np.cumsum(dense.sum(1))]))
            assert np.array_equal(ix, cols.astype(np.int32)) and len(rows) == ip[-1]


def test_pattern_product_bad_arguments_return_status(lib):
    # argument validation happens before any CUDA call, so this is safe without a GPU
    ws, dummy = 1 << 20, 1  # non-null stand-ins: none of these calls reaches a pointer
    count, fill = lib.gnn_pattern_product_count, lib.gnn_pattern_product_fill
    good = dict(a=dummy, n_a=4, k=3, n_b=4, lo=0, hi=4, loops=0)

    def call(fn, **over):
        a = {**good, **over}
        return fn(a["a"], a["a"], a["n_a"], a["k"], a["a"], a["a"], a["n_b"], a["lo"], a["hi"], a["loops"], dummy,
                  dummy, dummy, ws, None)

    for fn in (count, fill):
        assert call(fn, a=None) == 1 and b"null pointer" in lib.gnn_last_error_string()
        assert call(fn, k=-1) == 1 and b"negative size" in lib.gnn_last_error_string()
        assert call(fn, hi=5) == 1 and b"row range" in lib.gnn_last_error_string()
        assert call(fn, lo=3, hi=2) == 1 and b"row range" in lib.gnn_last_error_string()
        assert call(fn, n_b=1 << 31) == 1 and b"int32" in lib.gnn_last_error_string()
        assert call(fn, loops=1, n_b=5) == 1 and b"not square" in lib.gnn_last_error_string()
    assert count(dummy, dummy, 4, 3, dummy, dummy, 4, 0, 4, 0, None, None, dummy, ws, None) == 1
    assert fill(dummy, dummy, 4, 3, dummy, dummy, 4, 0, 4, 0, dummy, None, dummy, ws, None) == 1
