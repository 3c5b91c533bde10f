"""Partitioned GAT on the GPU: the fused attention kernels over a row block in the combined column space against the
square kernels over the whole graph (forward, rectangular backward, seeded dropout with an edge-slot base), the
versioned gnn_gat_dropout, GAT / SpGAT on a one-rank PartitionedGraph against the 1-GPU models bit for bit, the
limits the partitioned layer refuses, and two real ranks through tools/gat_dist_train.py."""
import ctypes as C

import numpy as np
import pytest
import torch

from graphneuralnetwork_b200 import _lib, functional as Fn
from graphneuralnetwork_b200 import synthetic as S
from graphneuralnetwork_b200.graph import CSRGraph, adj_cache
from graphneuralnetwork_b200.layers import GAT, SpGAT
from graphneuralnetwork_b200.layers.han import HANLayer
from graphneuralnetwork_b200.partition import PartitionedGraph

pytestmark = pytest.mark.gpu
DEV = "cuda"
N, LONG_ROW, HUB_COL = 4000, 1500, 3900


def _square(seed):
    """Square pattern with a self-loop in every row, mean degree ~9 (below gat.coop_min_avg_deg: the block and the
    whole graph get the same warp-per-row schedule), one row of 1500 edges (the long-row path) and a column that 1100
    rows read, 50 of them inside both test blocks (a transposed row that is long over the whole graph, short over a
    block: few enough terms that its fp32 sum stays within 1e-6 of float64)."""
    rng = np.random.default_rng(seed)
    cols = []
    for i in range(N):
        d = 1500 if i == LONG_ROW else int(rng.integers(2, 14))
        c = np.unique(rng.integers(0, N, d))
        c = c[(c != i) & (c != HUB_COL)]
        extra = [HUB_COL] if (1400 <= i < 1450 or 2700 <= i < 3750) else []
        cols.append(np.concatenate([[i], c, extra]).astype(np.int64))
    rowptr = np.concatenate([[0], np.cumsum([len(c) for c in cols])]).astype(np.int64)
    return rowptr, np.concatenate(cols)


def _block(rowptr, col, lo, hi):
    """The rows [lo, hi) in the combined column space: local c -> c - lo, remote -> hi - lo + halo slot."""
    rp = rowptr[lo:hi + 1] - rowptr[lo]
    cb = col[rowptr[lo]:rowptr[hi]]
    is_loc = (cb >= lo) & (cb < hi)
    halo = np.unique(cb[~is_loc])
    comb = np.where(is_loc, cb - lo, hi - lo + np.searchsorted(halo, cb))
    g = CSRGraph(torch.from_numpy(rp).to(DEV), torch.from_numpy(comb.astype(np.int32)).to(DEV), None, hi - lo,
                 hi - lo + len(halo))
    return g, torch.from_numpy(np.concatenate([np.arange(lo, hi), halo])).to(DEV)


def _gat64(g, Wh, s, t, H, Fp, keep, d_out):
    """float64 restatement: gradients (Wh, s, t) of sum(d_out * ELU(Σ_j softmax_j(LeakyReLU(s_i + t_j)) keep Wh_j))."""
    Wh, s, t = (x.double().clone().requires_grad_() for x in (Wh, s, t))
    rows = g.edge_rows().long()
    col = g.col.long()
    e = torch.nn.functional.leaky_relu(s[rows] + t[col], 0.2)
    m = torch.full((g.n_rows, H), -torch.inf, dtype=torch.float64, device=DEV).scatter_reduce(
        0, rows[:, None].expand(-1, H), e.detach(), "amax", include_self=True)
    p = torch.exp(e - m[rows])
    att = p / torch.zeros((g.n_rows, H), dtype=torch.float64, device=DEV).index_add(0, rows, p)[rows]
    if keep is not None:
        att = att * keep.double()
    out = torch.zeros((g.n_rows, H, Fp), dtype=torch.float64, device=DEV).index_add(
        0, rows, att[:, :, None] * Wh[col].view(-1, H, Fp))
    y = torch.nn.functional.elu(out.view(g.n_rows, H * Fp))
    return torch.autograd.grad(y, [Wh, s, t], d_out.double())


def _grads(g, Wh, s, t, H, Fp, drop, d_out):
    Wh, s, t = (x.clone().requires_grad_() for x in (Wh, s, t))
    y = Fn.gat_aggregate(g, Wh, s, t, H, Fp, 0.2, elu=1, dropout=drop)
    return torch.autograd.grad(y, [Wh, s, t], d_out)


def _rel(a, b):
    return float((a.double() - b.double()).abs().max()) / max(float(b.double().abs().max()), 1e-30)


@pytest.mark.parametrize("where", ["first", "middle"])
@pytest.mark.parametrize("p", [0.0, 0.6])
@pytest.mark.parametrize("H,Fp", [(8, 8), (1, 16)])
def test_rectangular_block_matches_square_kernels(H, Fp, p, where):
    rowptr, col = _square(3)
    lo, hi = (0, N // 2) if where == "first" else (N // 3, 2 * N // 3)
    assert lo <= LONG_ROW < hi and not lo <= HUB_COL < hi
    g = CSRGraph(torch.from_numpy(rowptr).to(DEV), torch.from_numpy(col.astype(np.int32)).to(DEV), None, N, N)
    gb, table = _block(rowptr, col, lo, hi)
    assert gb.n_cols > gb.n_rows
    gen = torch.Generator(device=DEV).manual_seed(5)
    Wh = torch.randn(N, H * Fp, device=DEV, generator=gen)
    s = torch.randn(N, H, device=DEV, generator=gen)
    t = torch.randn(N, H, device=DEV, generator=gen)
    drop = Fn.AttentionDropout(p, 777) if p else None
    drop_b = Fn.AttentionDropout(p, 777, None, int(rowptr[lo])) if p else None
    # forward: output, activation and row statistics are bit-identical to the square kernel's rows [lo, hi)
    res = []
    for gg, W_, s_, t_, d_ in ((g, Wh, s, t, drop), (gb, Wh[table], s[lo:hi], t[table], drop_b)):
        pre = torch.empty((gg.n_rows, H * Fp), device=DEV)
        act = torch.empty_like(pre)
        _, rm, rs = Fn.gat_fwd_raw(gg, W_, s_, t_, H, Fp, 0.2, elu=1, save_stats=True, out=pre, dropout=d_, out_act=act)
        res.append((pre, act, rm, rs))
    for a, b in zip(res[1], res[0]):
        assert torch.equal(a, b[lo:hi])
    # backward with d_out zero outside the block: every term the block does not contribute is an exact zero
    d_blk = torch.randn(hi - lo, H * Fp, device=DEV, generator=gen)
    d_out = torch.zeros(N, H * Fp, device=DEV)
    d_out[lo:hi] = d_blk
    dWh_sq, ds_sq, dt_sq = _grads(g, Wh, s, t, H, Fp, drop, d_out)
    dWh_b, ds_b, dt_b = _grads(gb, Wh[table], s[lo:hi], t[table], H, Fp, drop_b, d_blk)
    assert torch.equal(ds_b, ds_sq[lo:hi])
    outside = torch.ones(N, dtype=torch.bool, device=DEV)
    outside[table] = False
    assert not dWh_sq[outside].any() and not dt_sq[outside].any()
    thr = _lib.get_tuning("gat.long_row")
    deg_sq = torch.bincount(g.col.long(), minlength=N)[table]
    deg_b = torch.bincount(gb.col.long(), minlength=gb.n_cols)
    warp_both = (deg_sq <= thr) & (deg_b <= thr)
    one_only = (deg_sq > thr) != (deg_b > thr)
    assert warp_both.sum() > 0 and one_only.sum() == 1  # the hub column
    # d_Wh: each lane's sum runs over the column's edges in source order, so the exact zeros leave it unchanged
    assert torch.equal(dWh_b[warp_both], dWh_sq[table][warp_both])
    keep = Fn.attention_keep_mask_from_seed(g, H, drop) if p else None
    r_dWh, _, r_dt = _gat64(g, Wh, s, t, H, Fp, keep, d_out)
    r_dWh, r_dt = r_dWh[table], r_dt[table]
    if where == "first":
        # the block's sources come first in every transposed row: the per-head correction sums see the same
        # edges in the same lanes, so d_t is bit-identical too
        assert torch.equal(dt_b[warp_both], dt_sq[table][warp_both])
    else:
        # the zero terms of the rows before the block shift the block's edges to other lanes of the correction sum
        assert _rel(dt_b[warp_both], r_dt[warp_both]) <= 1e-6
    # a transposed row on the long-row path in only one run splits its edges over the warps differently
    assert _rel(dWh_b[one_only], r_dWh[one_only]) <= 1e-6 and _rel(dt_b[one_only], r_dt[one_only]) <= 1e-6
    assert _rel(dWh_b, r_dWh) <= 1e-5 and _rel(dt_b, r_dt) <= 1e-5


def _fwd_train(g, Wh, s, t, H, Fp, d, pre, act):
    lib = _lib.load()
    lr, thr = g.gat_long_rows()
    return lib.gnn_gat_fused_fwd_train_f32(Fn._p(g.rowptr), Fn._p(g.col), Fn._p(Wh), H * Fp, Fn._p(s), Fn._p(t),
                                           g.n_rows, g.nnz, H, Fp, 0.2, _lib.GAT_SOFTMAX, 1, None, None, C.byref(d),
                                           Fn._p(pre), Fn._p(act), H * Fp, None, None, Fn._p(lr), lr.numel(), thr, 0,
                                           Fn._stream_ptr())


def test_dropout_struct_versions():
    rowptr, col = _square(4)
    g = CSRGraph(torch.from_numpy(rowptr).to(DEV), torch.from_numpy(col.astype(np.int32)).to(DEV), None, N, N)
    H, Fp = 8, 8
    Wh, s, t = torch.randn(N, H * Fp, device=DEV), torch.randn(N, H, device=DEV), torch.randn(N, H, device=DEV)
    outs = []
    for size in (C.sizeof(_lib.GatDropout), _lib.GatDropout.edge_slot_base.offset):
        d = Fn.AttentionDropout(0.5, 99).c_struct()
        d.struct_size = size
        pre, act = torch.empty(N, H * Fp, device=DEV), torch.empty(N, H * Fp, device=DEV)
        _lib.check(_fwd_train(g, Wh, s, t, H, Fp, d, pre, act), "versioned dropout")
        outs.append(act)
    assert torch.equal(outs[0], outs[1])  # the previous layout reads as edge_slot_base = 0
    pre, act = torch.empty(N, H * Fp, device=DEV), torch.empty(N, H * Fp, device=DEV)
    d = Fn.AttentionDropout(0.5, 99).c_struct()
    d.struct_size = C.sizeof(_lib.GatDropout) - 4
    assert _fwd_train(g, Wh, s, t, H, Fp, d, pre, act) != _lib.GNN_OK
    # a slot base needs the whole seed on the host
    d = Fn.AttentionDropout(0.5, 99, torch.ones(1, dtype=torch.int64, device=DEV), 10).c_struct()
    assert _fwd_train(g, Wh, s, t, H, Fp, d, pre, act) != _lib.GNN_OK
    # with_slot_base mixes the device half into the host seed: the same stream
    dd = Fn.AttentionDropout(0.5, 99, torch.full((1,), 7, dtype=torch.int64, device=DEV))
    assert torch.equal(Fn.attention_keep_mask_from_seed(g, H, dd),
                       Fn.attention_keep_mask_from_seed(g, H, dd.with_slot_base(0)))


def _dense_adj(n, seed):
    return torch.from_numpy(S.symmetric_mask(n, 12 * n, seed=seed)).float().to(DEV)


@pytest.mark.parametrize("cls", [GAT, SpGAT])
def test_world_one_partitioned_model_is_bit_identical(cls):
    n, f_in, nhid, nclass, heads = 700, 50, 8, 7, 8
    adj = _dense_adj(n, 1)
    gen = torch.Generator(device=DEV).manual_seed(2)
    x = torch.randn(n, f_in, device=DEV, generator=gen)
    G = torch.randn(n, nclass, device=DEV, generator=gen)
    torch.manual_seed(0)
    model = cls(f_in, nhid, nclass, 0.6, 0.2, heads).to(DEV).train()

    def run(a):
        torch.manual_seed(123)
        Fn._drop_counters.clear()
        model.zero_grad(set_to_none=True)
        out = model(x, a)
        (out * G).sum().backward()
        return out.detach().clone(), {k: p.grad.clone() for k, p in model.named_parameters()}

    o1, g1 = run(adj)
    pg = PartitionedGraph.from_global(adj_cache.get(adj), 0, 1, widths=[heads * nhid, nclass])
    o2, g2 = run(pg)
    assert torch.equal(o1, o2)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k
    pg.close()


def test_partitioned_limits_are_refused():
    n = 300
    g = adj_cache.get(_dense_adj(n, 3))
    pg = PartitionedGraph.from_global(g, 0, 1, widths=[320, 64, 7])
    x = torch.randn(n, 20, device=DEV)
    with pytest.raises(_lib.GnnError, match="256"):
        GAT(20, 40, 7, 0.0, 0.2, 8).to(DEV)(x, pg)  # 8 heads x 40 = 320 columns
    with pytest.raises(_lib.GnnError, match="fp32"):
        GAT(20, 8, 7, 0.0, 0.2, 8).to(DEV).to(torch.bfloat16)(x.bfloat16(), pg)
    with pytest.raises(_lib.GnnError, match="PartitionedGraph"):
        HANLayer(2, 20, 8, 8, 0.0).to(DEV)([pg, pg], x)
    # rows without edges: the whole-graph mean is not defined on a row block
    empty = CSRGraph(torch.cat([g.rowptr[:6], g.rowptr[5:]]), g.col, None, n + 1, n + 1)
    pe = PartitionedGraph.from_global(empty, 0, 1, widths=[64, 7])
    with pytest.raises(_lib.GnnError, match="rows without edges"):
        GAT(20, 8, 7, 0.0, 0.2, 8).to(DEV)(torch.randn(n + 1, 20, device=DEV), pe)
    pg.close()
    pe.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one node")
def test_two_rank_gat_training_all_transports_check():
    """Two real ranks train GAT and SpGAT on a PartitionedGraph (Cora-like graph and a 200 k-row power-law graph,
    self-loops, 8 heads x 8, 41 classes, attention dropout 0.6) over p2p, ce and nccl; every rank compares its rows of
    the logits, the step-1 gradients and the weights after 3 Adam steps with the same model trained on one GPU, and
    repeats the run bit for bit."""
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
           "127.0.0.1", "--master-port", str(port), os.path.join(root, "tools", "gat_dist_train.py"), "--check",
           "--transports", "p2p", "ce", "nccl"]
    out = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 2 * 2 * 2 * 3, out.stdout[-2000:]  # ranks x graphs x models x transports
    for d in lines:
        tag = (d["model"], d["graph"], d["transport"], d["rank"])
        assert d["logits_rel_err"] <= 1e-5 and d["grad_rel_err"] <= 2e-5, (tag, d)
        assert d["weights_rel_err"] <= 1e-4 and d["bitwise_repeat"], (tag, d)
