"""GTN over a row partition without a GPU, world_size 2 and 3 over gloo on CPU: a float64 replay of what
`PartitionedRelationStack` and `GTN_Model.forward(ps, X_local, target_local)` compute — row blocks of every H_l, the
diagonal of a block at (r, lo + r), rank-ordered all-reduces of the column sums and of the gcn_conv degrees, the
reduce-scatter of the gcn_conv output with its ReLU and the all-gather that is its adjoint — against oracle/gtn_sparse.py
on the whole graph (logits) and the autograd of oracle/gtn.py's dense float64 model (every parameter gradient).  Also
the bounds of the layer chain (`metapath_row_plan` with one "metapath" per layer), the collective `max_nnz_per_rank`
refusal, and the C ABI of the ordered row reduction refusing bad arguments before any CUDA call."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from graphneuralnetwork_b200 import _lib
from graphneuralnetwork_b200.partition import balanced_bounds, metapath_row_plan
from oracle import gtn as ogtn
from oracle import gtn_sparse as S
from oracle.metapath import pattern_product

N, K, CH, W_IN, W_OUT, CLASSES = 36, 4, 2, 5, 3, 3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _stack(seed):
    """K relations over N nodes, the last the identity; a cycle in each relation keeps every off-diagonal column of
    every H non-empty (the dense model's `norm` has no gradient at an empty column)."""
    rng = np.random.default_rng(seed)
    A = np.zeros((N, N, K))
    for k in range(K - 1):
        A[:, :, k] = (rng.random((N, N)) < 0.03) * rng.uniform(0.2, 1.0, (N, N))
        perm = rng.permutation(N)
        A[perm, np.roll(perm, 1), k] = rng.uniform(0.2, 1.0, N)
    A[:, :, K - 1] = np.eye(N)
    return A


def _params(seed, L):
    g = torch.Generator().manual_seed(seed)
    p = {f"layers.{l}.conv{j}.weight": torch.randn(CH, K, 1, 1, generator=g, dtype=torch.float64)
         for l in range(L) for j in ((1, 2) if l == 0 else (1,))}
    p["weight"] = torch.randn(W_IN, W_OUT, generator=g, dtype=torch.float64) * 0.5
    p["linear1.weight"] = torch.randn(W_OUT, CH * W_OUT, generator=g, dtype=torch.float64) * 0.5
    p["linear1.bias"] = torch.randn(W_OUT, generator=g, dtype=torch.float64) * 0.1
    p["linear2.weight"] = torch.randn(CLASSES, W_OUT, generator=g, dtype=torch.float64) * 0.5
    p["linear2.bias"] = torch.randn(CLASSES, generator=g, dtype=torch.float64) * 0.1
    return p


def _drop_diag(indptr, indices, lo):
    rows = np.repeat(np.arange(len(indptr) - 1), np.diff(indptr)) + lo
    keep = rows != indices
    cum = np.concatenate([[0], np.cumsum(keep)])
    return cum[indptr].astype(np.int64), indices[keep]


def _chain(U, lo, hi, L):
    """[(indptr, indices) of the block of P_l] and [of D_l], rows [lo, hi): P_1 = U[lo:hi]·U, P_{l+1} = D_l·U."""
    ip, ix = U
    P, D = [], []
    a_ip, a_ix, rr, n_a = ip, ix, (lo, hi), N
    for _ in range(L):
        p = pattern_product(a_ip, a_ix, ip, ix, n_a, N, N, rr)
        d = _drop_diag(*p, lo)
        P.append(p)
        D.append(d)
        a_ip, a_ix, rr, n_a = d[0], d[1], None, hi - lo
    return P, D


def _mask(ptr, idx, rows):
    m = torch.zeros(rows, N, dtype=torch.float64)
    r = np.repeat(np.arange(rows), np.diff(ptr))
    m[torch.from_numpy(r), torch.from_numpy(idx.astype(np.int64))] = 1.0
    return m


class _AllSum(torch.autograd.Function):
    """Σ over the ranks in rank order (one all_gather); backward: the same sum of the gradients."""

    @staticmethod
    def forward(ctx, x):
        return _ordered_sum(x)

    @staticmethod
    def backward(ctx, dy):
        return _ordered_sum(dy)


def _ordered_sum(x):
    parts = [torch.empty_like(x) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, x.contiguous())
    acc = parts[0]
    for p in parts[1:]:
        acc = acc + p
    return acc


class _ReduceScatterRelu(torch.autograd.Function):
    """relu(Σ_q x_q)[lo:hi]; backward: the all-gather of every rank's dy ⊙ [y > 0] in rank order."""

    @staticmethod
    def forward(ctx, x, bounds, rank):
        y = _ordered_sum(x)[bounds[rank]:bounds[rank + 1]].clamp_min(0.0)
        ctx.save_for_backward(y)
        ctx.bounds = bounds
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        dz = dy * (y > 0).to(dy.dtype)
        b = ctx.bounds
        width = max(b[p + 1] - b[p] for p in range(len(b) - 1))
        pad = torch.zeros(width, dz.shape[1], dtype=dz.dtype)
        pad[:dz.shape[0]] = dz
        parts = [torch.empty_like(pad) for _ in range(len(b) - 1)]
        dist.all_gather(parts, pad)
        return torch.cat([p[:b[q + 1] - b[q]] for q, p in enumerate(parts)]), None, None


def _safe_inv(s):
    nz = s != 0
    return torch.where(nz, 1.0 / torch.where(nz, s, torch.ones_like(s)), torch.zeros_like(s))


def _replay(A, X, target, G, params, L, bounds, rank):
    """This rank's logits and its share of the loss Σ_t y[t]·G[t] of the partitioned model, float64."""
    sm = lambda name: torch.softmax(params[name][:, :, 0, 0], dim=1)  # [C, K]
    ip, ix, V = S.union(A)
    V = torch.from_numpy(V)
    lo, hi = bounds[rank], bounds[rank + 1]
    n_loc = hi - lo
    _, D = _chain((ip, ix), lo, hi, L)
    rows = torch.from_numpy(np.repeat(np.arange(N), np.diff(ip)))
    cols = torch.from_numpy(ix.astype(np.int64))

    def dense(vals):  # [nnz_U, C] on U -> [C, N, N]
        M = torch.zeros(CH, N, N, dtype=torch.float64)
        return M.index_put((torch.arange(CH)[:, None], rows[None, :], cols[None, :]), vals.t())

    a = dense(V @ sm("layers.0.conv1.weight").t())
    H = a[:, lo:hi] @ dense(V @ sm("layers.0.conv2.weight").t())  # [C, n_loc, N], the block of P_1
    for l in range(1, L):
        Hd = H * _mask(*D[l - 1], n_loc)                          # the block of D_l: diagonal at (r, lo + r)
        sums = _AllSum.apply(Hd.sum(dim=1))                        # column sums over every rank's rows
        H = (Hd * _safe_inv(sums)[:, None, :]) @ dense(V @ sm(f"layers.{l}.conv1.weight").t())
    eye = torch.zeros(n_loc, N, dtype=torch.float64)
    eye[torch.arange(n_loc), torch.arange(lo, hi)] = 1.0
    Hp = H * _mask(*D[-1], n_loc) + eye                           # (D_L + I), this rank's rows
    deg = _AllSum.apply(Hp.sum(dim=1))                             # [C, N] degrees of gcn_conv
    XW = torch.from_numpy(X[lo:hi]) @ params["weight"]
    Y = torch.cat([(Hp[c] * _safe_inv(deg[c])[None, :]).t() @ XW for c in range(CH)], dim=1)  # partial [N, C*w]
    X_ = _ReduceScatterRelu.apply(Y, bounds, rank)
    X_ = torch.relu(X_ @ params["linear1.weight"].t() + params["linear1.bias"])
    mine = (target >= lo) & (target < hi)
    y = X_[torch.from_numpy(target[mine] - lo)] @ params["linear2.weight"].t() + params["linear2.bias"]
    return y, (y * torch.from_numpy(G[mine])).sum(), mine


def _chain_counter(U, L):
    """count(m, lo, hi) of the layer chain, as PartitionedRelationStack builds it (scipy in place of the kernels)."""
    state = {}

    def count(m, lo, hi):
        ip, ix = U
        a_ip, a_ix, rr, n_a = (ip, ix, (lo, hi), N) if m == 0 else (*state["D"], None, hi - lo)
        p = pattern_product(a_ip, a_ix, ip, ix, n_a, N, N, rr)
        state["D"] = _drop_diag(*p, lo)
        return torch.from_numpy(p[0])
    return count


def _check_plan(rank, world, A, L):
    ip, ix, _ = S.union(A)
    P_whole, _ = S.patterns(ip, ix, N, L)
    bounds, rps = metapath_row_plan(_chain_counter((ip, ix), L), N, L, rank, world, what="PartitionedRelationStack",
                                    items="layers")
    assert bounds == balanced_bounds(torch.from_numpy(sum(p[0] for p in P_whole)), world)
    lo, hi = bounds[rank], bounds[rank + 1]
    for (p_ip, _), rp in zip(P_whole, rps):
        assert torch.equal(rp, torch.from_numpy(p_ip[lo:hi + 1] - p_ip[lo]))
    block = [sum(int(p[0][bounds[q + 1]] - p[0][bounds[q]]) for p in P_whole) for q in range(world)]
    worst = int(np.argmax(block))
    with pytest.raises(_lib.GnnError, match=f"PartitionedRelationStack: .* over the {L} layers .*rank {worst}: "
                                            f"{block[worst]}"):
        metapath_row_plan(_chain_counter((ip, ix), L), N, L, rank, world, max(block) - 1, what="PartitionedRelationStack",
                          items="layers")
    return bounds


def _check_replay(rank, world, A, L, bounds, seed):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, W_IN))
    target = np.arange(0, N, 2)
    G = rng.standard_normal((len(target), CLASSES))
    params = {k: v.clone().requires_grad_(True) for k, v in _params(seed, L).items()}
    y, loss, mine = _replay(A, X, target, G, params, L, bounds, rank)
    loss.backward()
    grads = {k: _ordered_sum(p.grad) for k, p in params.items()}  # what allreduce_gradients adds up
    y64 = S.gtn_forward(A, X, target, {k: v.detach().numpy() for k, v in params.items()}, CH, L)
    ref = torch.from_numpy(y64[mine])
    scale = max(float(np.abs(y64).max()), 1e-30)
    err = float((y.detach() - ref).abs().max()) if y.numel() else 0.0
    assert err <= 1e-12 * scale, (err, bounds)
    dense = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    yd = ogtn.gtn_forward(torch.from_numpy(A), torch.from_numpy(X), torch.from_numpy(target), dense, CH, L)
    assert float((yd.detach() - torch.from_numpy(y64)).abs().max()) <= 1e-12 * scale
    (yd * torch.from_numpy(G)).sum().backward()
    for k, g in grads.items():
        ref_g = dense[k].grad
        err = float((g - ref_g).abs().max()) / max(float(ref_g.abs().max()), 1e-30)
        assert err <= 1e-12, (k, err, bounds)


def _worker(rank, world, port, out_q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        seen = []
        for L in (1, 2, 3):
            A = _stack(10 + L)
            bounds = _check_plan(rank, world, A, L)
            seen.append(bounds)
            uneven = [0, 0, N] if world == 2 else [0, 5, 5, N]  # a rank with an empty block
            for b in (bounds, uneven):
                _check_replay(rank, world, A, L, b, 20 + L)
        dist.barrier()
        out_q.put((rank, "ok", seen))
    except Exception:  # reported to the parent, which fails the test with it
        import traceback
        out_q.put((rank, traceback.format_exc(), None))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_partitioned_gtn_replay_bounds_and_refusal(world):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for rank, status, _ in results:
        assert status == "ok", f"rank {rank}:\n{status}"
    for p in procs:
        assert p.exitcode == 0
    assert len({str(seen) for _, _, seen in results}) == 1  # every rank chose the same bounds


def test_reduce_rows_abi_bad_arguments_return_status(lib):
    # every check runs before any CUDA call: no device needed
    fake = 256  # a non-null address that is never dereferenced
    fn = lib.gnn_peer_reduce_rows_f32
    two = (C.c_void_p * 2)(fake, fake)
    assert fn(two, 2, 4, 4, 0, 0, fake, 4, 0, None) == 0  # an empty row range launches nothing
    assert fn(None, 2, 4, 4, 0, 4, fake, 4, 0, None) == 1 and b"null pointer" in lib.gnn_last_error_string()
    assert fn(two, 2, 4, 4, 0, 4, None, 4, 0, None) == 1
    assert fn((C.c_void_p * 2)(fake, None), 2, 4, 4, 0, 4, fake, 4, 0, None) == 1
    assert b"source 1" in lib.gnn_last_error_string()
    assert fn(two, 0, 4, 4, 0, 4, fake, 4, 0, None) == 1
    assert fn((C.c_void_p * 17)(*([fake] * 17)), 17, 4, 4, 0, 4, fake, 4, 0, None) == 1
    assert fn(two, 2, 4, 0, 0, 4, fake, 4, 0, None) == 1
    assert fn(two, 2, 3, 4, 0, 4, fake, 4, 0, None) == 1  # ld_src < F
    assert fn(two, 2, 4, 4, 0, 4, fake, 3, 0, None) == 1  # ld_out < F
    assert fn(two, 2, 4, 4, 5, 4, fake, 4, 0, None) == 1 and b"row range" in lib.gnn_last_error_string()
    assert fn(two, 2, 4, 4, -1, 4, fake, 4, 0, None) == 1
