"""Host logic of partitioned GAT training, world_size 2 and 3 over gloo on CPU: the attention view of every rank's row
block (combined column space, edge-slot base), a float64 replay of the partitioned attention layer — halo exchange,
its backward with the ordered gradient return, and the parameter gradients summed over the ranks — against
whole-graph autograd, and the collective refusal of graphs with rows without edges."""
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from graphneuralnetwork_b200 import _lib
from graphneuralnetwork_b200.functional import AttentionDropout, attention_keep_mask_from_seed
from graphneuralnetwork_b200.partition import balanced_bounds, build_attention_view, build_halo_plan

H, FP, F_IN, ALPHA = 4, 3, 5, 0.2


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _global_graph(n, seed, empty_row=None):
    """Power-law-ish CSR with a self-loop in every row (first edge), a hub row and unsorted duplicate-free columns."""
    rng = np.random.default_rng(seed)
    deg = rng.poisson(5, size=n)
    deg[7] = 120  # a hub row
    cols = []
    for i in range(n):
        c = np.unique(np.minimum((n * rng.random(deg[i]) ** 2).astype(np.int64), n - 1))
        c = c[c != i]
        rng.shuffle(c)
        cols.append(np.concatenate([[i], c]) if i != empty_row else np.zeros(0, np.int64))
    rowptr = np.concatenate([[0], np.cumsum([len(c) for c in cols])]).astype(np.int64)
    return rowptr, np.concatenate(cols).astype(np.int64)


def _block(rowptr, col, bounds, rank):
    lo, hi = bounds[rank], bounds[rank + 1]
    return torch.from_numpy(rowptr[lo:hi + 1] - rowptr[lo]), torch.from_numpy(col[rowptr[lo]:rowptr[hi]])


def gat_layer64(rowptr, col, Wh_tab, s_rows, t_tab):
    """ELU of the multi-head attention aggregation (GAT/models/layers.py:22-37, sparse form) in float64:
    rows of `rowptr`, columns indexing the table rows of Wh_tab / t_tab."""
    n = rowptr.numel() - 1
    rows = torch.repeat_interleave(torch.arange(n), rowptr[1:] - rowptr[:-1])
    col = col.long()
    e = torch.nn.functional.leaky_relu(s_rows[rows] + t_tab[col], ALPHA)  # [nnz, H]
    m = torch.full((n, H), -torch.inf, dtype=e.dtype).scatter_reduce(0, rows[:, None].expand(-1, H), e.detach(),
                                                                      "amax", include_self=True)
    p = torch.exp(e - m[rows])
    den = torch.zeros((n, H), dtype=e.dtype).index_add(0, rows, p)
    att = p / den[rows]
    msg = att[:, :, None] * Wh_tab[col].view(-1, H, FP)
    out = torch.zeros((n, H, FP), dtype=e.dtype).index_add(0, rows, msg)
    return torch.nn.functional.elu(out.reshape(n, H * FP))


class _HaloReplay(torch.autograd.Function):
    """Test-side replay of functional.halo_exchange over gloo: forward [X ; halo] by all_to_all of the send list;
    backward dX = dX_comb[:n_local] + the returned halo gradients added in (peer, slot) order — the order of the
    pattern-only CSR `R` of PartitionedSpmm (positions of the send list, ascending)."""

    @staticmethod
    def forward(ctx, X, plan):
        ctx.plan = plan
        send = X[plan.send_rows.long()].contiguous()
        halo = torch.empty((plan.n_halo, X.shape[1]), dtype=X.dtype)
        dist.all_to_all_single(halo, send, output_split_sizes=plan.recv_counts, input_split_sizes=plan.send_counts)
        return torch.cat([X, halo], 0)

    @staticmethod
    def backward(ctx, dX_comb):
        plan = ctx.plan
        n_loc = plan.n_local
        back = torch.empty((int(plan.send_rows.numel()), dX_comb.shape[1]), dtype=dX_comb.dtype)
        dist.all_to_all_single(back, dX_comb[n_loc:].contiguous(), output_split_sizes=plan.send_counts,
                               input_split_sizes=plan.recv_counts)
        dX = dX_comb[:n_loc].clone()
        for k, r in enumerate(plan.send_rows.tolist()):  # (peer, slot) order
            dX[r] += back[k]
        return dX, None


def _params(seed):
    g = torch.Generator().manual_seed(seed)
    W = torch.randn(F_IN, H * FP, generator=g, dtype=torch.float64) * 0.5
    a_src = torch.randn(H, FP, generator=g, dtype=torch.float64)
    a_dst = torch.randn(H, FP, generator=g, dtype=torch.float64)
    return [t.requires_grad_() for t in (W, a_src, a_dst)]


def _check(rank, world, n, seed):
    rowptr, col = _global_graph(n, seed)
    bounds = balanced_bounds(torch.from_numpy(rowptr), world)
    lo, hi = bounds[rank], bounds[rank + 1]
    rp, cc = _block(rowptr, col, bounds, rank)
    plan = build_halo_plan(rp, cc, None, bounds, rank, world, waves=2)
    view = build_attention_view(plan, rp, cc)
    view.require_edges()
    assert view.n_rows == hi - lo and view.n_cols == hi - lo + plan.n_halo
    assert view.edge_slot_base == int(rowptr[lo]) and not view.any_empty_row
    # the views mapped back through halo_ids reproduce the global CSR exactly
    table_ids = torch.cat([torch.arange(lo, hi), plan.halo_ids])
    mine = (view.rowptr.numpy(), table_ids[view.col.long()].numpy())
    every = [None] * world
    dist.all_gather_object(every, mine)
    rp_all = np.concatenate([every[0][0]] + [r[1:] + sum(len(e[1]) for e in every[:q]) for q, (r, _) in
                                             enumerate(every) if q > 0])
    assert np.array_equal(rp_all, rowptr) and np.array_equal(np.concatenate([c for _, c in every]), col)
    # the seeded attention-dropout mask of the block with its slot base == the global mask's block of slots
    cpu = lambda m: types.SimpleNamespace(nnz=m, device="cpu")  # noqa: E731
    drop = AttentionDropout(0.6, 12345)
    full = attention_keep_mask_from_seed(cpu(int(rowptr[-1])), H, drop)
    part = attention_keep_mask_from_seed(cpu(view.col.numel()), H, AttentionDropout(0.6, 12345, None, view.edge_slot_base))
    assert torch.equal(part, full[rowptr[lo]:rowptr[hi]])
    # float64 replay of the partitioned layer against whole-graph autograd
    X = torch.from_numpy(np.random.default_rng(seed + 1).standard_normal((n, F_IN)))
    G = torch.from_numpy(np.random.default_rng(seed + 2).standard_normal((n, H * FP)))
    W, a_src, a_dst = _params(seed + 3)
    Xg = X.clone().requires_grad_()
    Wh = Xg @ W
    Wh3 = Wh.view(n, H, FP)
    out = gat_layer64(torch.from_numpy(rowptr), torch.from_numpy(col), Wh, (Wh3 * a_src).sum(-1), (Wh3 * a_dst).sum(-1))
    (out * G).sum().backward()
    ref = {"X": Xg.grad[lo:hi].clone(), "W": W.grad.clone(), "a_src": a_src.grad.clone(), "a_dst": a_dst.grad.clone()}
    out_ref = out.detach()[lo:hi]
    for p in (W, a_src, a_dst):
        p.grad = None
    Xl = X[lo:hi].clone().requires_grad_()
    Wh_comb = _HaloReplay.apply(Xl @ W, plan)
    Wc3 = Wh_comb.view(-1, H, FP)
    y = gat_layer64(view.rowptr, view.col, Wh_comb, (Wc3[:hi - lo] * a_src).sum(-1), (Wc3 * a_dst).sum(-1))
    (y * G[lo:hi]).sum().backward()
    got = {"X": Xl.grad, "W": W.grad.clone(), "a_src": a_src.grad.clone(), "a_dst": a_dst.grad.clone()}
    for k in ("W", "a_src", "a_dst"):  # partition.allreduce_gradients
        dist.all_reduce(got[k])

    def rel(a, b):
        return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-300)

    assert rel(y.detach(), out_ref) <= 1e-12
    for k in ref:
        assert rel(got[k], ref[k]) <= 1e-12, k
    return plan.n_halo


def _check_empty_row_refused(rank, world, n, seed):
    # the only row without edges lives in the LAST rank's block: every rank must raise
    rowptr, col = _global_graph(n, seed, empty_row=n - 3)
    bounds = balanced_bounds(torch.from_numpy(rowptr), world)
    rp, cc = _block(rowptr, col, bounds, rank)
    plan = build_halo_plan(rp, cc, None, bounds, rank, world)
    view = build_attention_view(plan, rp, cc)
    with pytest.raises(_lib.GnnError, match="rows without edges"):
        view.require_edges()


def _worker(rank, world, port, out_q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = [_check(rank, world, 300, 5), _check(rank, world, 157, 9)]
        _check_empty_row_refused(rank, world, 200, 4)
        out_q.put((rank, "ok", res))
    except Exception:  # reported to the parent, which fails the test with it
        import traceback
        out_q.put((rank, traceback.format_exc(), None))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_attention_view_replay_and_empty_row_refusal(world):
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
    assert all(h > 0 for _, _, res in results for h in res)  # every block read remote rows


def test_world_one_view_is_the_whole_graph():
    rowptr, col = _global_graph(90, 2)
    rp, cc = torch.from_numpy(rowptr), torch.from_numpy(col)
    plan = build_halo_plan(rp, cc, None, [0, 90], 0, 1)
    view = build_attention_view(plan, rp, cc)
    assert view.n_cols == 90 and view.edge_slot_base == 0
    assert torch.equal(view.col.long(), cc) and torch.equal(view.rowptr, rp)


def test_rectangular_backward_is_in_the_abi_table():
    assert "gnn_gat_fused_bwd_ex_f32" in _lib.SIGNATURES
    assert [f for f, _ in _lib.GatDropout._fields_][-1] == "edge_slot_base"
