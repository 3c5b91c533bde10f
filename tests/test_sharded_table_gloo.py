"""Host logic of the sharded feature table, world_size 2 and 3 over gloo on CPU: the default row bounds, a numpy replay
of the sharded gather's addressing (shard lookup, row within the shard) against the gather over the concatenated
table, and the collective refusal when the ranks disagree on F, ld, dtype or the bounds (every rank raises)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from graphneuralnetwork_b200 import _lib
from graphneuralnetwork_b200.partition import agree_layout, locate_rows, shard_bounds


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_shard_bounds():
    assert shard_bounds(10, 3) == [0, 3, 6, 10]
    assert shard_bounds(2, 3) == [0, 0, 1, 2]  # N < world: empty shards
    assert shard_bounds(0, 2) == [0, 0, 0]
    for n in (1, 7, 232_965, 111_059_956):
        for w in range(1, 9):
            b = shard_bounds(n, w)
            sizes = np.diff(b)
            assert b[0] == 0 and b[-1] == n and sizes.min() >= 0 and sizes.max() - sizes.min() <= 1
    with pytest.raises(ValueError):
        shard_bounds(5, 0)


def _replay(shards, bounds, ids, fanout, reduce):
    """The sharded gather in numpy: each id read from its shard at its row within the shard; skipped ids (shard -1)
    contribute nothing, mean still divides by the fanout."""
    s, r = locate_rows(torch.from_numpy(ids), bounds)
    s, r = s.numpy(), r.numpy()
    F = shards[0].shape[1]
    rows = np.zeros((ids.size, F))
    valid = s >= 0
    for k in np.nonzero(valid)[0]:
        rows[k] = shards[s[k]][r[k]]
    return _reduce(rows, valid, fanout, reduce)


def _reduce(rows, valid, fanout, reduce):
    rows = rows.reshape(-1, fanout, rows.shape[1])
    valid = valid.reshape(-1, fanout)[:, :, None]
    if reduce == "max":
        return np.where(valid, rows, -np.inf).max(axis=1)
    total = np.where(valid, rows, 0.0).sum(axis=1)
    return total / fanout if reduce == "mean" else total


@pytest.mark.parametrize("bounds", [[0, 997], [0, 400, 997], [0, 1, 600, 997], [0, 100, 100, 250, 251, 600, 700, 900, 997],
                                    [0, 0, 0, 997]])
def test_shard_addressing_replay(bounds):
    rng = np.random.default_rng(len(bounds))
    N, F, fanout = bounds[-1], 5, 4
    X = rng.standard_normal((N, F))
    shards = [X[bounds[s]:bounds[s + 1]] for s in range(len(bounds) - 1)]
    edges = sorted({b for b in bounds[:-1]} | {b - 1 for b in bounds[1:] if b > 0})
    ids = np.concatenate([edges, [-1, N, N + 3, -7], rng.integers(0, N, 400)]).astype(np.int64)
    ids = ids[:ids.size // fanout * fanout]
    s, r = locate_rows(torch.from_numpy(ids), bounds)
    for i, (sh, row) in enumerate(zip(s.tolist(), r.tolist())):
        if 0 <= ids[i] < N:  # the last shard whose first row is <= id, and the row lies inside that shard
            assert bounds[sh] <= ids[i] < bounds[sh + 1] and row == ids[i] - bounds[sh]
            assert all(bounds[q] > ids[i] for q in range(sh + 1, len(bounds) - 1))
        else:
            assert sh == -1 and row == -1
    valid = (ids >= 0) & (ids < N)
    whole = np.where(valid[:, None], X[np.clip(ids, 0, N - 1)], 0.0)
    for reduce in ("mean", "sum", "max"):
        want = _reduce(whole, valid, fanout, reduce)
        assert np.array_equal(_replay(shards, bounds, ids, fanout, reduce), want)


def _worker(rank, world, port, out_q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = []
        bounds = shard_bounds(1000, world)
        agree_layout(602, 604, torch.float32, bounds, None, rank, world)  # agreement: no error
        other = list(bounds)
        other[1] += 1 if rank == world - 1 else 0
        cases = {
            "F": (602 if rank else 601, 604, torch.float32, bounds, None),
            "ld": (602, 604 if rank else 608, torch.float32, bounds, None),
            "dtype": (602, 604, torch.bfloat16 if rank == world - 1 else torch.float32, bounds, None),
            "bounds": (602, 604, torch.float32, other, None),
            "refusal": (602, 604, torch.float32, bounds, "the table requires grad" if rank == 1 else None),
        }
        for name, (F, ld, dt, b, err) in cases.items():
            try:
                agree_layout(F, ld, dt, b, err, rank, world)
                res.append((name, None))
            except _lib.GnnError as e:
                res.append((name, str(e)))
        out_q.put((rank, "ok", res))
    except Exception:
        import traceback
        out_q.put((rank, traceback.format_exc(), None))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_layout_disagreement_is_refused_on_every_rank(world):
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
    msgs = {}
    for rank, _, res in results:
        for name, msg in res:
            assert msg is not None, (rank, name)  # every rank raised
            msgs.setdefault(name, set()).add(msg)
    for name, m in msgs.items():
        assert len(m) == 1, name  # the same message everywhere
    assert "disagree" in msgs["F"].pop() and "disagree" in msgs["ld"].pop() and "disagree" in msgs["dtype"].pop()
    assert "disagree on the bounds" in msgs["bounds"].pop()
    assert "rank 1: the table requires grad" in msgs["refusal"].pop()
