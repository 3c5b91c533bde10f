"""Partitioned HAN on the GPU: the batched-rectangular attention kernels against the square batched kernels (same
bits when the two strides are equal; a rank's block of an M-graph set with a union halo and per-graph dropout slot
shifts against the whole set), the semantic attention split at the cross-rank sums, HANModel on a one-rank
PartitionedMetapaths against the 1-GPU HANModel bit for bit, the refusals, and two real ranks through
tools/han_dist_train.py."""
import ctypes as C

import numpy as np
import pytest
import torch

from graphneuralnetwork_b200 import _lib, functional as Fn
from graphneuralnetwork_b200.graph import CSRGraph
from graphneuralnetwork_b200.layers.han import HANLayer, HANModel
from graphneuralnetwork_b200.partition import PartitionedMetapaths

pytestmark = pytest.mark.gpu
DEV = "cuda"
N, LONG_ROW, HUB_COL = 3000, 1200, 2990


def _graph(seed, hub=True):
    """Square pattern with a self-loop first in every row, mean degree ~8, one row of 1500 edges (the long-row path)
    and (hub=True) a column read by 1030 rows (above gat.long_row), 50 of them inside both test blocks."""
    rng = np.random.default_rng(seed)
    cols = []
    for i in range(N):
        d = 1500 if i == LONG_ROW else int(rng.integers(2, 14))
        c = np.unique(rng.integers(0, N, d))
        c = c[(c != i) & (c != HUB_COL)]
        rng.shuffle(c)
        extra = [HUB_COL] if hub and (1050 <= i < 1100 or 2000 <= i < 2980) else []
        cols.append(np.concatenate([[i], c, extra]).astype(np.int64))
    rowptr = np.concatenate([[0], np.cumsum([len(c) for c in cols])]).astype(np.int64)
    return rowptr, np.concatenate(cols)


def _csr(rowptr, col, n_rows, n_cols):
    return CSRGraph(torch.from_numpy(rowptr).to(DEV), torch.from_numpy(col.astype(np.int32)).to(DEV), None, n_rows,
                    n_cols)


def _set(M, seed):
    gs = [_graph(seed + m, hub=(m == M - 1)) for m in range(M)]
    return gs, CSRGraph.block_diagonal([_csr(rp, c, N, N) for rp, c in gs])


def _block_set(gs, lo, hi):
    """Rows [lo, hi) of every graph in ONE combined column space (the union halo): local c -> c - lo, remote ->
    n_local + slot in the sorted union; the M renamed blocks stacked as a block diagonal.  Also the per-graph slot
    shifts (global batched slot - local batched slot) and the table's global ids."""
    n_loc = hi - lo
    blocks = [(rp[lo:hi + 1] - rp[lo], c[rp[lo]:rp[hi]]) for rp, c in gs]
    halo = np.unique(np.concatenate([c[(c < lo) | (c >= hi)] for _, c in blocks]))
    nc = n_loc + len(halo)
    rps, cols, off, shift, nnz_g, nnz_l = [], [], 0, [], 0, 0
    for m, ((rp, c), (rpg, _)) in enumerate(zip(blocks, gs)):
        is_loc = (c >= lo) & (c < hi)
        comb = np.where(is_loc, c - lo, n_loc + np.searchsorted(halo, c))
        rps.append(rp[:-1] + off)
        cols.append(comb + m * nc)
        shift.append(nnz_g - nnz_l + int(rpg[lo]))
        off += len(c)
        nnz_g += int(rpg[-1])
        nnz_l += len(c)
    g = _csr(np.concatenate(rps + [[off]]).astype(np.int64), np.concatenate(cols), len(gs) * n_loc, len(gs) * nc)
    return g, torch.from_numpy(np.concatenate([np.arange(lo, hi), halo])).to(DEV), torch.tensor(shift, device=DEV)


def _rel(a, b):
    return float((a.double() - b.double()).abs().max()) / max(float(b.double().abs().max()), 1e-30)


def _p(x):
    return Fn._p(x)


def _fwd_square(g, M, Wh, s, t, H, Fp, d):
    lib = _lib.load()
    lr, thr = g.gat_long_rows()
    n = g.n_rows // M
    pre, act = torch.empty(n, M * H * Fp, device=DEV), torch.empty(n, M * H * Fp, device=DEV)
    rm, rs = torch.empty(g.n_rows, H, device=DEV), torch.empty(g.n_rows, H, device=DEV)
    _lib.check(lib.gnn_gat_fused_fwd_train_f32(_p(g.rowptr), _p(g.col), _p(Wh), M * H * Fp, _p(s), _p(t), g.n_rows,
                                               g.nnz, H, Fp, 0.2, _lib.GAT_SOFTMAX, 2, None, None,
                                               C.byref(d) if d is not None else None, _p(pre), _p(act), M * H * Fp,
                                               _p(rm), _p(rs), _p(lr), lr.numel(), thr, n, Fn._stream_ptr()), "square")
    return pre, act, rm, rs


def _batch(M, rows, cols, shift=None):
    b = _lib.GatBatch()
    b.struct_size, b.n_graphs, b.rows_per_graph, b.cols_per_graph = C.sizeof(_lib.GatBatch), M, rows, cols
    b.slot_shift = _p(shift)
    return b


def _fwd_batch(g, M, Wh, s, t, H, Fp, d, b):
    lib = _lib.load()
    lr, thr = g.gat_long_rows()
    n = g.n_rows // M
    pre, act = torch.empty(n, M * H * Fp, device=DEV), torch.empty(n, M * H * Fp, device=DEV)
    rm, rs = torch.empty(g.n_rows, H, device=DEV), torch.empty(g.n_rows, H, device=DEV)
    _lib.check(lib.gnn_gat_fused_fwd_batch_f32(_p(g.rowptr), _p(g.col), _p(Wh), M * H * Fp, _p(s), _p(t), g.nnz, H, Fp,
                                               0.2, _lib.GAT_SOFTMAX, 2, None, C.byref(d) if d is not None else None,
                                               _p(pre), _p(act), M * H * Fp, _p(rm), _p(rs), _p(lr), lr.numel(), thr,
                                               C.byref(b), Fn._stream_ptr()), "batch")
    return pre, act, rm, rs


def _bwd(g, M, Wh, s, t, H, Fp, d, fwd, d_act, b=None):
    lib = _lib.load()
    pre, _, rm, rs = fwd
    gt = g.transpose()
    (lr, thr), (lrt, _) = g.gat_long_rows(), gt.gat_long_rows()
    dWh, ds, dt = torch.empty_like(Wh), torch.empty_like(s), torch.empty_like(t)
    scratch = torch.empty(g.n_rows, 4, H, device=DEV)
    d_pre = torch.empty_like(pre)
    common = (_p(g.rowptr), _p(g.col), _p(gt.rowptr), _p(gt.col), _p(g.perm_t), _p(Wh), M * H * Fp, _p(s), _p(t),
              _p(rm), _p(rs), _p(pre), _p(d_act), M * H * Fp)
    tail = (None, _p(dWh), M * H * Fp, _p(ds), _p(dt), _p(scratch), g.nnz, _p(lr), lr.numel(), _p(lrt), lrt.numel(),
            thr, 2, _p(d_pre), C.byref(d) if d is not None else None)
    if b is None:
        rc = lib.gnn_gat_fused_bwd_f32(*common, g.n_rows, H, Fp, 0.2, _lib.GAT_SOFTMAX, *tail, g.n_rows // M,
                                       Fn._stream_ptr())
    else:
        rc = lib.gnn_gat_fused_bwd_batch_f32(*common, H, Fp, 0.2, _lib.GAT_SOFTMAX, *tail, C.byref(b), Fn._stream_ptr())
    _lib.check(rc, "bwd")
    return dWh, ds, dt


def _inputs(M, n_rows, H, Fp, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(n_rows, M * H * Fp, device=DEV, generator=gen), torch.randn(M * n_rows, H, device=DEV,
            generator=gen), torch.randn(M * n_rows, H, device=DEV, generator=gen), gen)


@pytest.mark.parametrize("p", [0.0, 0.6])
@pytest.mark.parametrize("H,Fp", [(8, 8), (1, 16)])
@pytest.mark.parametrize("M", [2, 3])
def test_equal_strides_match_square_batched_kernels(M, H, Fp, p):
    _, g = _set(M, 10)
    Wh, s, t, gen = _inputs(M, N, H, Fp, 1)
    d = Fn.AttentionDropout(p, 4242).c_struct() if p else None
    b = _batch(M, N, N)
    sq = _fwd_square(g, M, Wh, s, t, H, Fp, d)
    rb = _fwd_batch(g, M, Wh, s, t, H, Fp, d, b)
    for x, y in zip(rb, sq):
        assert torch.equal(x, y)
    d_act = torch.randn(N, M * H * Fp, device=DEV, generator=gen)
    for x, y in zip(_bwd(g, M, Wh, s, t, H, Fp, d, rb, d_act, b), _bwd(g, M, Wh, s, t, H, Fp, d, sq, d_act)):
        assert torch.equal(x, y)


def _batched_rows(x, M, n):
    """[n, M*W] (graph m's columns at m*W) -> [M*n, W] batched-row major."""
    return x.view(n, M, -1).permute(1, 0, 2).reshape(M * n, -1)


def _gat64(g, Wh_rows, s, t, H, Fp, keep, d_out_rows):
    """float64 gradients (Wh rows, s, t) of sum(d_out * ELU(ELU(Σ_j softmax_j(LeakyReLU(s_i + t_j)) keep Wh_j)))
    over a block-diagonal CSR whose table rows are Wh_rows [n_cols, H*Fp]."""
    Wh, s, t = (x.double().clone().requires_grad_() for x in (Wh_rows, s, t))
    rows = g.edge_rows().long()
    col = g.col.long()
    e = torch.nn.functional.leaky_relu(s[rows] + t[col], 0.2)
    mx = torch.full((g.n_rows, H), -torch.inf, dtype=torch.float64, device=DEV).scatter_reduce(
        0, rows[:, None].expand(-1, H), e.detach(), "amax", include_self=True)
    pr = torch.exp(e - mx[rows])
    att = pr / torch.zeros((g.n_rows, H), dtype=torch.float64, device=DEV).index_add(0, rows, pr)[rows]
    if keep is not None:
        att = att * keep.double()
    out = torch.zeros((g.n_rows, H, Fp), dtype=torch.float64, device=DEV).index_add(
        0, rows, att[:, :, None] * Wh[col].view(-1, H, Fp))
    y = torch.nn.functional.elu(torch.nn.functional.elu(out.view(g.n_rows, H * Fp)))
    return torch.autograd.grad(y, [Wh, s, t], d_out_rows.double())


@pytest.mark.parametrize("where", ["first", "middle"])
@pytest.mark.parametrize("p", [0.0, 0.6])
@pytest.mark.parametrize("H,Fp", [(8, 8), (1, 16)])
def test_rank_block_with_union_halo_matches_square_batched_kernels(H, Fp, p, where):
    M = 3
    gs, g = _set(M, 20)
    lo, hi = (0, N // 2) if where == "first" else (N // 3, 2 * N // 3)
    assert lo <= LONG_ROW < hi and not lo <= HUB_COL < hi
    gb, table, shift = _block_set(gs, lo, hi)
    n_loc, nc = hi - lo, table.numel()
    assert nc > n_loc
    Wh, s, t, gen = _inputs(M, N, H, Fp, 5)
    d = Fn.AttentionDropout(p, 777).c_struct() if p else None
    # block inputs: Wh's table rows, s of the own rows and t of the table rows, per graph
    Wh_b = Wh[table]
    s_b = s.view(M, N, H)[:, lo:hi].reshape(M * n_loc, H)
    t_b = t.view(M, N, H)[:, table].reshape(M * nc, H)
    sq = _fwd_square(g, M, Wh, s, t, H, Fp, d)
    rb = _fwd_batch(gb, M, Wh_b, s_b, t_b, H, Fp, d, _batch(M, n_loc, nc, shift))
    # forward rows, activations and row statistics: bit-identical (with p = 0.6 the shifts draw the whole set's mask)
    assert torch.equal(rb[0], sq[0][lo:hi]) and torch.equal(rb[1], sq[1][lo:hi])
    for x, y in zip(rb[2:], sq[2:]):
        assert torch.equal(x, y.view(M, N, H)[:, lo:hi].reshape(M * n_loc, H))
    # backward with d_out zero outside the block
    d_blk = torch.randn(n_loc, M * H * Fp, device=DEV, generator=gen)
    d_act = torch.zeros(N, M * H * Fp, device=DEV)
    d_act[lo:hi] = d_blk
    dWh_sq, ds_sq, dt_sq = _bwd(g, M, Wh, s, t, H, Fp, d, sq, d_act)
    dWh_b, ds_b, dt_b = _bwd(gb, M, Wh_b, s_b, t_b, H, Fp, d, rb, d_blk, _batch(M, n_loc, nc, shift))
    assert torch.equal(ds_b, ds_sq.view(M, N, H)[:, lo:hi].reshape(M * n_loc, H))
    # d_Wh / d_t per (graph, table row): bit-identical where both runs take the warp path
    thr = _lib.get_tuning("gat.long_row")
    deg_sq = torch.bincount(g.col.long(), minlength=M * N).view(M, N)[:, table]
    deg_b = torch.bincount(gb.col.long(), minlength=M * nc).view(M, nc)
    warp_both = (deg_sq <= thr) & (deg_b <= thr)                 # [M, nc]
    assert warp_both.sum() > 0 and (~warp_both).sum() >= 1       # the hub column of the last graph
    dWh_sq_t = dWh_sq[table].view(nc, M, H * Fp).permute(1, 0, 2)  # [M, nc, H*Fp]
    dWh_b_t = dWh_b.view(nc, M, H * Fp).permute(1, 0, 2)
    dt_sq_t, dt_b_t = dt_sq.view(M, N, H)[:, table], dt_b.view(M, nc, H)
    assert torch.equal(dWh_b_t[warp_both], dWh_sq_t[warp_both])
    keep = None
    if p:
        keep = Fn.attention_keep_mask_from_seed(g, H, Fn.AttentionDropout(p, 777))
    r_dWh, _, r_dt = _gat64(g, _batched_rows(Wh, M, N), s, t, H, Fp, keep, _batched_rows(d_act, M, N))
    r_dWh = r_dWh.view(M, N, H * Fp)[:, table]
    r_dt = r_dt.view(M, N, H)[:, table]
    if where == "first":
        assert torch.equal(dt_b_t[warp_both], dt_sq_t[warp_both])
    else:
        assert _rel(dt_b_t[warp_both], r_dt[warp_both]) <= 1e-6
    other = ~warp_both
    assert _rel(dWh_b_t[other], r_dWh[other]) <= 1e-6 and _rel(dt_b_t[other], r_dt[other]) <= 1e-6
    assert _rel(dWh_b_t, r_dWh) <= 1e-5 and _rel(dt_b_t, r_dt) <= 1e-5


def _semantic_parts(z, W1, b1, q, bounds, d_out):
    """The split semantic attention over the row ranges `bounds` in one process: partial per part, rank-ordered sums,
    finalize; returns (out, dz, dq, db, dW1)."""
    lib = _lib.load()
    n, M, D = z.shape
    K = W1.shape[0]
    ws = Fn._semantic_workspace(K, z.device)
    st = Fn._stream_ptr()
    parts = [(a, b) for a, b in zip(bounds[:-1], bounds[1:])]
    Ps = [torch.mm(z[a:b].reshape((b - a) * M, D), W1.t()) for a, b in parts]
    sums = []
    for (a, b), P in zip(parts, Ps):
        sm = torch.empty(M, device=DEV)
        _lib.check(lib.gnn_semantic_scores_partial_f32(_p(P), K, _p(b1), _p(q), b - a, M, K, _p(sm), _p(ws), ws.numel(),
                                                       st), "partial")
        sums.append(sm)
    tot = sums[0]
    for x in sums[1:]:
        tot = tot + x
    scores, beta = torch.empty(M, device=DEV), torch.empty(M, device=DEV)
    _lib.check(lib.gnn_semantic_scores_finalize_f32(_p(tot), n, M, _p(scores), _p(beta), st), "finalize")
    out = torch.empty(n, D, device=DEV)
    for a, b in parts:
        _lib.check(lib.gnn_semantic_combine_f32(_p(beta), _p(z[a:b].contiguous()), b - a, M, D,
                                                _p(out[a:b]), st), "combine")
    dz, dbs = torch.empty_like(z), []
    for a, b in parts:
        dzp, db_ = torch.empty(b - a, M, D, device=DEV), torch.empty(M, device=DEV)
        _lib.check(lib.gnn_semantic_combine_bwd_partial_f32(_p(d_out[a:b].contiguous()), _p(z[a:b].contiguous()),
                                                            _p(beta), b - a, M, D, _p(dzp), _p(db_), _p(ws),
                                                            ws.numel(), st), "bwd partial")
        dz[a:b] = dzp
        dbs.append(db_)
    dbeta = dbs[0]
    for x in dbs[1:]:
        dbeta = dbeta + x
    dsn = torch.empty(M, device=DEV)
    _lib.check(lib.gnn_semantic_combine_bwd_finalize_f32(_p(dbeta), _p(beta), n, M, _p(dsn), st), "bwd finalize")
    dq, db, dW1 = torch.zeros(K, device=DEV), torch.zeros(K, device=DEV), torch.zeros_like(W1)
    for (a, b), P in zip(parts, Ps):
        dP, dqp, dbp = torch.empty_like(P), torch.empty(K, device=DEV), torch.empty(K, device=DEV)
        _lib.check(lib.gnn_semantic_scores_bwd_f32(_p(P), K, _p(b1), _p(q), _p(dsn), b - a, M, K, _p(dP), K, _p(dqp),
                                                   _p(dbp), _p(ws), ws.numel(), st), "scores bwd")
        dq, db = dq + dqp, db + dbp
        zp = z[a:b].reshape((b - a) * M, D)
        dW1 = dW1 + dP.t() @ zp
        dz[a:b] += (dP @ W1).view(b - a, M, D)
    return out, dz, dq, db, dW1


def test_semantic_split_matches_fused_and_float64():
    n, M, D, K = 3025, 3, 64, 128
    gen = torch.Generator(device=DEV).manual_seed(3)
    z = torch.randn(n, M, D, device=DEV, generator=gen)
    W1 = torch.randn(K, D, device=DEV, generator=gen) * 0.1
    b1 = torch.randn(K, device=DEV, generator=gen) * 0.1
    q = torch.randn(K, device=DEV, generator=gen) * 0.1
    d_out = torch.randn(n, D, device=DEV, generator=gen)
    # one part: partial + finalize inside autograd == the fused entries, bit for bit
    grads = []
    for fn in (lambda *a: Fn.semantic_attention(*a), lambda *a: Fn.semantic_attention_partitioned(*a, n, 1)):
        xs = [x.clone().requires_grad_() for x in (z, W1, b1, q)]
        y = fn(*xs)
        grads.append([y.detach()] + list(torch.autograd.grad(y, xs, d_out)))
    for a, b in zip(*grads):
        assert torch.equal(a, b)
    # float64 reference
    xs = [x.double().clone().requires_grad_() for x in (z, W1, b1, q)]
    w = (torch.tanh(xs[0] @ xs[1].t() + xs[2]) @ xs[3]).mean(0)
    y = torch.einsum("m,nmd->nd", torch.softmax(w, 0), xs[0])
    ref = [y.detach()] + list(torch.autograd.grad(y, xs, d_out.double()))
    # dq / db are column sums of terms whose weights d_scores_over_n add up to zero over the metapaths: the fused
    # entries' own fp32 error bounds them (measured 7e-6 of float64 for this input)
    fused_err = [_rel(grads[0][i], ref[i]) for i in range(5)]
    for bounds in ([0, n], [0, 1000, n], [0, 17, 2000, n]):
        out, dz, dq, db, dW1 = _semantic_parts(z, W1, b1, q, bounds, d_out)
        for i, got in enumerate((out, dz, dW1, db, dq)):
            tol = 1e-6 if i < 3 else max(1e-6, 2 * fused_err[i])
            assert _rel(got, ref[i]) <= tol, (i, _rel(got, ref[i]), fused_err[i])


def _metapath_adjs(n, M, seed):
    """Dense 0/1 float64 metapath adjacencies with self-loops (HANModel takes the reference's dense masks)."""
    rng = np.random.default_rng(seed)
    out = []
    for m in range(M):
        A = rng.random((n, n)) < (0.004 * (1 + 6 * m))
        A = A | A.T | np.eye(n, dtype=bool)
        out.append(torch.from_numpy(A.astype(np.float64)).to(DEV))
    return out


@pytest.mark.parametrize("layers", [1, 2])
def test_world_one_partitioned_han_is_bit_identical(layers):
    n, f_in, hidden, classes, heads, M = 600, 40, 8, 3, 8, 3
    adjs = _metapath_adjs(n, M, 1)
    gen = torch.Generator(device=DEV).manual_seed(2)
    x = torch.randn(n, f_in, device=DEV, generator=gen)
    G = torch.randn(n, classes, device=DEV, generator=gen)
    torch.manual_seed(0)
    model = HANModel(M, f_in, hidden, classes, [heads] * layers, 0.6).to(DEV).train()

    def run(g):
        torch.manual_seed(123)
        Fn._drop_counters.clear()
        model.zero_grad(set_to_none=True)
        out = model(g, x)
        (out * G).sum().backward()
        return out.detach().clone(), {k: p.grad.clone() for k, p in model.named_parameters()}

    o1, g1 = run(adjs)
    from graphneuralnetwork_b200.graph import adj_cache
    pm = PartitionedMetapaths.from_global([adj_cache.get(a) for a in adjs], 0, 1, widths=[M * heads * hidden])
    assert len(pm) == M and pm.slot_shift == [0] * M and pm.halo_rows == 0
    o2, g2 = run(pm)
    assert torch.equal(o1, o2)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k
    pm.close()


def test_partitioned_han_refusals():
    n, M = 300, 2
    from graphneuralnetwork_b200.graph import adj_cache
    gs = [adj_cache.get(a) for a in _metapath_adjs(n, M, 3)]
    pm = PartitionedMetapaths.from_global(gs, 0, 1, widths=[M * 64, M * 320])
    x = torch.randn(n, 20, device=DEV)
    with pytest.raises(_lib.GnnError, match="fp32"):
        HANLayer(M, 20, 8, 8, 0.0).to(DEV).to(torch.bfloat16)(pm, x.bfloat16())
    with pytest.raises(_lib.GnnError, match="256"):
        HANLayer(M, 20, 40, 8, 0.0).to(DEV)(pm, x)  # 8 heads x 40 = 320 columns
    pm.close()
    # a metapath row without edges: the whole-set mean is not defined on a row block
    g0 = gs[0]
    empty = CSRGraph(torch.cat([g0.rowptr[:6], g0.rowptr[5:]]), g0.col, None, n + 1, n + 1)
    g1 = CSRGraph(torch.cat([gs[1].rowptr, gs[1].rowptr[-1:]]), gs[1].col, None, n + 1, n + 1)
    pe = PartitionedMetapaths.from_global([empty, g1], 0, 1, widths=[M * 64])
    with pytest.raises(_lib.GnnError, match="rows without edges"):
        HANLayer(M, 20, 8, 8, 0.0).to(DEV)(pe, torch.randn(n + 1, 20, device=DEV))
    pe.close()
    # the C entries refuse a bad description with a status, before any launch
    lib = _lib.load()
    b = _batch(33, 4, 4)
    assert lib.gnn_gat_fused_fwd_batch_f32(None, None, None, 8, None, None, 0, 1, 8, 0.2, 0, 0, None, None, None, None,
                                           8, None, None, None, 0, 0, C.byref(b), None) == 3
    b = _batch(2, 8, 4)
    assert lib.gnn_gat_fused_fwd_batch_f32(None, None, None, 8, None, None, 0, 1, 8, 0.2, 0, 0, None, None, None, None,
                                           8, None, None, None, 0, 0, C.byref(b), None) != 0
    b = _batch(2, 4, 4)
    b.struct_size = 8
    assert lib.gnn_gat_fused_fwd_batch_f32(None, None, None, 8, None, None, 0, 1, 8, 0.2, 0, 0, None, None, None, None,
                                           8, None, None, None, 0, 0, C.byref(b), None) != 0


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one node")
def test_two_rank_han_training_all_transports_check():
    """Two real ranks train HAN on PartitionedMetapaths (ACM-shaped metapaths, self-loops, 8 heads x 8, attention
    dropout 0.6) over p2p, ce and nccl; every rank compares its rows of the logits, the step-1 gradients and the
    weights after 3 Adam steps with the same model trained on one GPU, and repeats the run bit for bit."""
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
           "127.0.0.1", "--master-port", str(port), os.path.join(root, "tools", "han_dist_train.py"), "--check",
           "--transports", "p2p", "ce", "nccl"]
    out = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 2 * 3, out.stdout[-2000:]  # ranks x transports
    for d in lines:
        tag = (d["transport"], d["rank"])
        assert d["logits_rel_err"] <= 1e-5 and d["grad_rel_err"] <= 2e-5, (tag, d)
        assert d["weights_rel_err"] <= 1e-4 and d["bitwise_repeat"], (tag, d)
