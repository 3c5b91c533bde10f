"""Host logic of partitioned HAN training, world_size 2 and 3 over gloo on CPU: the union halo plan of M metapath row
blocks and the renaming of each block into its combined column space, the per-graph dropout slot shifts against the
global block-diagonal numbering, a float64 replay of the partitioned HAN layer (one halo exchange of the stacked Wh,
the batched attention over the renamed blocks, semantic attention with rank-ordered node sums) against a whole-graph
float64 HAN layer, and the collective refusal of a metapath row without edges."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from graphneuralnetwork_b200 import _lib
from graphneuralnetwork_b200.partition import balanced_bounds, build_halo_plan, build_metapath_view, union_block

M, H, FP, F_IN, K, ALPHA = 3, 2, 3, 5, 4, 0.2


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _metapaths(n, seed, empty=None):
    """M CSRs over n nodes with a self-loop first in every row and mean degrees 3, 8, 20 (unsorted columns);
    `empty` = (graph, row) left without edges."""
    rng = np.random.default_rng(seed)
    out = []
    for m, deg in enumerate((3, 8, 20)):
        cols = []
        for i in range(n):
            c = np.unique(rng.integers(0, n, rng.poisson(deg)))
            c = c[c != i]
            rng.shuffle(c)
            cols.append(np.zeros(0, np.int64) if empty == (m, i) else np.concatenate([[i], c]).astype(np.int64))
        rowptr = np.concatenate([[0], np.cumsum([len(c) for c in cols])]).astype(np.int64)
        out.append((rowptr, np.concatenate(cols)))
    return out


def _blocks(gs, bounds, rank):
    lo, hi = bounds[rank], bounds[rank + 1]
    return ([torch.from_numpy(rp[lo:hi + 1] - rp[lo]) for rp, _ in gs],
            [torch.from_numpy(c[rp[lo]:rp[hi]]) for rp, c in gs])


def _bounds(gs, world):
    return balanced_bounds(torch.from_numpy(sum(rp for rp, _ in gs)), world)


def attention64(rowptr, col, Wh_tab, s_rows, t_tab):
    """ELU(ELU(multi-head attention aggregation)) in float64 (NodeAttention.py:25-35, 62): rows of `rowptr`, columns
    indexing the table rows of Wh_tab [*, H*FP] / t_tab [*, H]."""
    n = rowptr.numel() - 1
    rows = torch.repeat_interleave(torch.arange(n), rowptr[1:] - rowptr[:-1])
    col = col.long()
    e = torch.nn.functional.leaky_relu(s_rows[rows] + t_tab[col], ALPHA)
    mx = torch.full((n, H), -torch.inf, dtype=e.dtype).scatter_reduce(0, rows[:, None].expand(-1, H), e.detach(),
                                                                        "amax", include_self=True)
    p = torch.exp(e - mx[rows])
    att = p / torch.zeros((n, H), dtype=e.dtype).index_add(0, rows, p)[rows]
    out = torch.zeros((n, H, FP), dtype=e.dtype).index_add(0, rows, att[:, :, None] * Wh_tab[col].view(-1, H, FP))
    return torch.nn.functional.elu(torch.nn.functional.elu(out.reshape(n, H * FP)))


class _HaloReplay(torch.autograd.Function):
    """[X ; halo] by all_to_all of the send list; backward: the halo gradients return to their owners and are added
    in (peer, slot) order (functional.halo_exchange)."""

    @staticmethod
    def forward(ctx, X, plan):
        ctx.plan = plan
        halo = torch.empty((plan.n_halo, X.shape[1]), dtype=X.dtype)
        dist.all_to_all_single(halo, X[plan.send_rows.long()].contiguous(), output_split_sizes=plan.recv_counts,
                               input_split_sizes=plan.send_counts)
        return torch.cat([X, halo], 0)

    @staticmethod
    def backward(ctx, dX_comb):
        plan = ctx.plan
        back = torch.empty((int(plan.send_rows.numel()), dX_comb.shape[1]), dtype=dX_comb.dtype)
        dist.all_to_all_single(back, dX_comb[plan.n_local:].contiguous(), output_split_sizes=plan.send_counts,
                               input_split_sizes=plan.recv_counts)
        dX = dX_comb[:plan.n_local].clone()
        for k, r in enumerate(plan.send_rows.tolist()):
            dX[r] += back[k]
        return dX, None


class _RankSum(torch.autograd.Function):
    """Σ over the ranks in rank order (functional._rank_ordered_sum); its backward is the sum over the ranks of the
    gradients every rank's result received."""

    @staticmethod
    def forward(ctx, x):
        parts = [torch.empty_like(x) for _ in range(dist.get_world_size())]
        dist.all_gather(parts, x.contiguous())
        acc = parts[0]
        for p in parts[1:]:
            acc = acc + p
        return acc

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous().clone()
        dist.all_reduce(g)
        return g


def _params(seed):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)  # noqa: E731
    ps = {"W": r(M, F_IN, H * FP) * 0.5, "a_src": r(M, H, FP), "a_dst": r(M, H, FP), "W1": r(K, H * FP) * 0.3,
          "b1": r(K) * 0.3, "q": r(K)}
    return {k: v.requires_grad_() for k, v in ps.items()}


def semantic64(z, P, n_total, rank_sum=None):
    """β = softmax_M(Σ_n q·tanh(W1 z + b1) / n_total), out = Σ_m β_m z_m; the node sum through `rank_sum`."""
    w = (torch.tanh(z @ P["W1"].t() + P["b1"]) @ P["q"]).sum(0)
    if rank_sum is not None:
        w = rank_sum(w)
    beta = torch.softmax(w / n_total, 0)
    return torch.einsum("m,nmd->nd", beta, z)


def _check(rank, world, n, seed):
    gs = _metapaths(n, seed)
    bounds = _bounds(gs, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    rps, cols = _blocks(gs, bounds, rank)
    rp_u, col_u = union_block(rps, cols, n)
    plan = build_halo_plan(rp_u, col_u, None, bounds, rank, world, waves=2)
    view = build_metapath_view(plan, rps, cols)
    view.require_edges()
    n_loc = hi - lo
    assert view.n_local == n_loc and view.n_comb == n_loc + plan.n_halo and view.n_graphs == M
    # the union block's rows are the per-row unions of the metapaths' columns
    for i in range(0, n_loc, 7):
        want = sorted(set().union(*[set(c[rp[i]:rp[i + 1]].tolist()) for rp, c in zip(rps, cols)]))
        assert col_u[rp_u[i]:rp_u[i + 1]].tolist() == want
    # every metapath's renamed block maps back through the table ids to its global rows, in edge order
    table_ids = torch.cat([torch.arange(lo, hi), plan.halo_ids])
    rows_local = view.rowptr.numel() - 1
    assert rows_local == M * n_loc and int(view.col.max()) < M * view.n_comb
    for m, (rp, c) in enumerate(zip(rps, cols)):
        r = view.rowptr[m * n_loc:(m + 1) * n_loc + 1]
        got = view.col[int(r[0]):int(r[-1])].long() - m * view.n_comb
        assert torch.equal(r - r[0], rp)
        assert bool(((got >= 0) & (got < view.n_comb)).all())
        assert torch.equal(table_ids[got], c)
    # slot shifts: local batched slot e of graph m + shift[m] == its slot in the global block diagonal
    nnz_g = [int(rp[-1]) for rp, _ in gs]
    for m, (rpg, _) in enumerate(gs):
        r = view.rowptr[m * n_loc:(m + 1) * n_loc + 1]
        local = torch.arange(int(r[0]), int(r[-1]))
        glob = sum(nnz_g[:m]) + int(rpg[lo]) + torch.arange(int(r[-1]) - int(r[0]))
        assert torch.equal(local + view.slot_shift[m], glob)
    # the halo of the union against the per-metapath halos
    assert max(view.halo_rows_per_graph) <= plan.n_halo <= sum(view.halo_rows_per_graph)
    # float64 replay of the partitioned HAN layer against the whole-graph layer: forward and every gradient
    X = torch.from_numpy(np.random.default_rng(seed + 1).standard_normal((n, F_IN)))
    G = torch.from_numpy(np.random.default_rng(seed + 2).standard_normal((n, H * FP)))
    P = _params(seed + 3)
    Xg = X.clone().requires_grad_()
    z = []
    for m, (rp, c) in enumerate(gs):
        Wh = Xg @ P["W"][m]
        Wh3 = Wh.view(n, H, FP)
        z.append(attention64(torch.from_numpy(rp), torch.from_numpy(c), Wh, (Wh3 * P["a_src"][m]).sum(-1),
                             (Wh3 * P["a_dst"][m]).sum(-1)))
    out = semantic64(torch.stack(z, 1), P, n)
    (out * G).sum().backward()
    ref = {"X": Xg.grad[lo:hi].clone(), **{k: v.grad.clone() for k, v in P.items()}}
    out_ref = out.detach()[lo:hi]
    for v in P.values():
        v.grad = None
    Xl = X[lo:hi].clone().requires_grad_()
    Wh_loc = torch.cat([Xl @ P["W"][m] for m in range(M)], 1)         # [n_local, M*H*FP]
    Wh_comb = _HaloReplay.apply(Wh_loc, plan)                         # one exchange for all metapaths
    nc = Wh_comb.shape[0]
    Wh4 = Wh_comb.view(nc, M, H, FP)
    s = (Wh4[:n_loc] * P["a_src"][None]).sum(-1).permute(1, 0, 2).reshape(M * n_loc, H)
    t = (Wh4 * P["a_dst"][None]).sum(-1).permute(1, 0, 2).reshape(M * nc, H)
    Wh_rows = Wh4.reshape(nc, M, H * FP).permute(1, 0, 2).reshape(M * nc, H * FP)   # batched table rows
    y = attention64(view.rowptr, view.col, Wh_rows, s, t)             # [M*n_local, H*FP], one batched "launch"
    zb = y.view(M, n_loc, H * FP).permute(1, 0, 2)
    outp = semantic64(zb, P, n, _RankSum.apply)
    (outp * G[lo:hi]).sum().backward()
    got = {"X": Xl.grad, **{k: v.grad.clone() for k, v in P.items()}}
    for k in P:  # partition.allreduce_gradients
        dist.all_reduce(got[k])

    def rel(a, b):
        return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-300)

    assert rel(outp.detach(), out_ref) <= 1e-12
    for k in ref:
        assert rel(got[k], ref[k]) <= 1e-12, k
    return plan.n_halo, sum(view.halo_rows_per_graph)


def _check_empty_row_refused(rank, world, n, seed):
    # the only row without edges is in metapath 1, in the LAST rank's block: every rank must raise
    gs = _metapaths(n, seed, empty=(1, n - 3))
    bounds = _bounds(gs, world)
    rps, cols = _blocks(gs, bounds, rank)
    rp_u, col_u = union_block(rps, cols, n)
    plan = build_halo_plan(rp_u, col_u, None, bounds, rank, world)
    view = build_metapath_view(plan, rps, cols)
    with pytest.raises(_lib.GnnError, match="rows without edges"):
        view.require_edges()


def _worker(rank, world, port, out_q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res = [_check(rank, world, 240, 5), _check(rank, world, 131, 9)]
        _check_empty_row_refused(rank, world, 150, 4)
        out_q.put((rank, "ok", res))
    except Exception:  # reported to the parent, which fails the test with it
        import traceback
        out_q.put((rank, traceback.format_exc(), None))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_metapath_view_replay_and_empty_row_refusal(world):
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
    assert all(h > 0 for _, _, res in results for h, _ in res)  # every block read remote rows


def test_world_one_view_is_the_block_diagonal():
    gs = _metapaths(70, 2)
    rps = [torch.from_numpy(rp) for rp, _ in gs]
    cols = [torch.from_numpy(c) for _, c in gs]
    rp_u, col_u = union_block(rps, cols, 70)
    plan = build_halo_plan(rp_u, col_u, None, [0, 70], 0, 1)
    view = build_metapath_view(plan, rps, cols)
    assert view.n_comb == 70 and view.slot_shift == [0] * M and plan.n_halo == 0
    assert torch.equal(view.col.long(), torch.cat([c + 70 * m for m, c in enumerate(cols)]))


def test_batched_rectangular_entries_are_in_the_abi_table():
    for f in ("gnn_gat_fused_fwd_batch_f32", "gnn_gat_fused_bwd_batch_f32", "gnn_semantic_scores_partial_f32",
              "gnn_semantic_scores_finalize_f32", "gnn_semantic_combine_bwd_partial_f32",
              "gnn_semantic_combine_bwd_finalize_f32"):
        assert f in _lib.SIGNATURES
    assert [f for f, _ in _lib.GatBatch._fields_] == ["struct_size", "n_graphs", "rows_per_graph", "cols_per_graph",
                                                      "slot_shift"]
