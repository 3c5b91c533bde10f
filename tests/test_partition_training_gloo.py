"""Host logic of partitioned GCN training, world_size 2 and 3 over gloo on CPU: where the fused bias/ReLU epilogue
lands in the schedule of the partitioned SpMM, its float64 replay against the global product, and the training
rules (loss over the global row count, gradient all-reduce, parameter broadcast)."""
import os
import socket

import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from graphneuralnetwork_b200.partition import (allreduce_gradients, balanced_bounds, broadcast_parameters,
                                               build_halo_plan, global_count, partitioned_cross_entropy,
                                               reference_step_cpu)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _global_graph(n, seed, F):
    rng = np.random.default_rng(seed)
    deg = rng.poisson(6, size=n)
    deg[::11] = 0
    deg[5] = 300  # a hub row
    rowptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64)
    col = np.minimum((n * rng.random(rowptr[-1]) ** 3).astype(np.int64), n - 1)
    val = rng.standard_normal(rowptr[-1]).astype(np.float32)
    X = rng.standard_normal((n, F)).astype(np.float32)
    return rowptr, col, val, X


def _check_schedule(rank, world, n, seed, waves, c0):
    F = 7
    rowptr, col, val, X = _global_graph(n, seed, F)
    bounds = balanced_bounds(torch.from_numpy(rowptr), world)
    lo, hi = bounds[rank], bounds[rank + 1]
    rp = torch.from_numpy(rowptr[lo:hi + 1] - rowptr[lo])
    plan = build_halo_plan(rp, torch.from_numpy(col[rowptr[lo]:rowptr[hi]]), torch.from_numpy(val[rowptr[lo]:rowptr[hi]]),
                           bounds, rank, world, waves=waves, two_pass_chunks=c0, F=F)
    n_loc = hi - lo
    rows_of = lambda c: np.arange(n_loc) if c.row_map is None else c.row_map.numpy()  # noqa: E731
    # P1's skip prefix is exactly its two-pass mixed rows (local columns now, remote columns in a later pass)
    mixed = np.diff(plan.rowptr_rem.numpy()) > 0
    two_pass = np.nonzero(mixed & (np.arange(n_loc) < plan.chunk_bounds[plan.two_pass_chunks]))[0]
    p1 = plan.p1
    assert p1 is not None
    assert np.array_equal(np.sort(rows_of(p1)[:p1.epilogue_skip]), two_pass)
    assert not np.any(mixed[rows_of(p1)[p1.epilogue_skip:]])  # the rest of P1 are interior rows
    # every local row gets the epilogue exactly once, from the consumer that adds its last contribution
    epi, last = np.zeros(n_loc, int), np.full(n_loc, -1)
    epi_by = np.full(n_loc, -1)
    for i, c in enumerate([p1] + list(plan.p2)):
        if c is None:
            continue
        r = rows_of(c)
        last[r] = i
        r_epi = r[c.epilogue_skip:] if c.mode == "local" else r
        epi[r_epi] += 1
        epi_by[r_epi] = i
        if c.mode != "local":
            assert c.epilogue_skip == 0
    assert np.all(epi == 1) and np.array_equal(epi_by, last)
    # the float64 replay with the epilogue == relu(Â·X + b) of the global graph, own rows
    b = np.random.default_rng(seed + 2).standard_normal(F).astype(np.float32)
    halo = torch.from_numpy(X[plan.halo_ids.numpy()])
    A = sp.csr_matrix((val.astype(np.float64), col, rowptr), shape=(n, n))
    full = A @ X.astype(np.float64)
    for bias, relu in [(b, True), (b, False), (None, True)]:
        Y = reference_step_cpu(plan, torch.from_numpy(X[lo:hi]), halo, None if bias is None else torch.from_numpy(bias),
                               relu).numpy()
        ref = full[lo:hi] + (0.0 if bias is None else bias.astype(np.float64))
        if relu:
            ref = np.maximum(ref, 0.0)
        assert float(np.abs(Y - ref).max()) <= 1e-9
    return plan.two_pass_chunks, plan.waves


def _check_training_rules(rank, world):
    # loss rule: Σ over the ranks of (Σ own-row losses / global count) == the mean over all training rows
    n, C = 97, 5
    g = torch.Generator().manual_seed(3)
    logits = torch.randn(n, C, generator=g, dtype=torch.float64)
    labels = torch.randint(0, C, (n,), generator=g)
    idx_train = torch.randperm(n, generator=g)[:41].sort().values
    bounds = [n * p // world for p in range(world + 1)]
    lo, hi = bounds[rank], bounds[rank + 1]
    mine = idx_train[(idx_train >= lo) & (idx_train < hi)]
    n_train = global_count(mine.numel(), "cpu")
    assert n_train == idx_train.numel()
    loss = partitioned_cross_entropy(logits[mine], labels[mine], n_train)
    total = loss.detach().clone()
    dist.all_reduce(total)
    want = torch.nn.functional.cross_entropy(logits[idx_train], labels[idx_train])
    assert abs(float(total) - float(want)) <= 1e-12
    # replicated toy model: different initial weights per rank, rank 0's broadcast, per-rank loss on own rows,
    # summed gradients == the gradient of the global loss
    torch.manual_seed(100 + rank)
    model = torch.nn.Sequential(torch.nn.Linear(C, 4), torch.nn.ReLU(), torch.nn.Linear(4, C)).double()
    broadcast_parameters(model)
    torch.manual_seed(100)
    ref = torch.nn.Sequential(torch.nn.Linear(C, 4), torch.nn.ReLU(), torch.nn.Linear(4, C)).double()
    for p, q in zip(model.parameters(), ref.parameters()):
        assert torch.equal(p, q)
    partitioned_cross_entropy(model(logits[mine]), labels[mine], n_train).backward()
    allreduce_gradients(model)
    torch.nn.functional.cross_entropy(ref(logits[idx_train]), labels[idx_train]).backward()
    for p, q in zip(model.parameters(), ref.parameters()):
        assert torch.allclose(p.grad, q.grad, rtol=1e-10, atol=1e-13)


def _worker(rank, world, port, cases, out_q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = [_check_schedule(rank, world, 400, 7, waves, c0) for waves, c0 in cases]
        _check_training_rules(rank, world)
        out_q.put((rank, "ok", res))
    except Exception as e:  # reported to the parent, which fails the test with it
        import traceback
        out_q.put((rank, traceback.format_exc(), None))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_epilogue_schedule_replay_and_training_rules(world):
    cases = [(1, None), (1, 0), (1, 1), (4, 2), (3, 0), (4, 4), (None, None)]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, cases, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for rank, status, _ in results:
        assert status == "ok", f"rank {rank}:\n{status}"
    for p in procs:
        assert p.exitcode == 0
    for rank, _, res in results:  # the fixed schedules ran as requested
        for (waves, c0), (chosen, k) in zip(cases, res):
            assert c0 is None or chosen == c0
            assert waves is None or k == waves
