"""bf16 features on partitioned graphs, on the GPU: the bf16 rectangular and batched-rectangular attention entries
against the square bf16 kernels (forward and d_s bit for bit, d_Wh / d_t bit for bit where both runs take the same
schedule and against float64 elsewhere), their ABI refusals, GCN / GAT / SpGAT on a one-rank bf16 PartitionedGraph
against the 1-GPU bf16 models bit for bit in train mode, HAN on a one-rank bf16 PartitionedMetapaths against the 1-GPU
bf16 HAN, the dtype refusals, and two real ranks through the three training tools with --dtype bf16."""
import ctypes as C

import numpy as np
import pytest
import torch

from graphneuralnetwork_b200 import _lib, functional as Fn
from graphneuralnetwork_b200 import synthetic as S
from graphneuralnetwork_b200.graph import CSRGraph, adj_cache
from graphneuralnetwork_b200.layers import GAT, GCN_Model, SpGAT
from graphneuralnetwork_b200.layers.han import HANLayer, HANModel
from graphneuralnetwork_b200.partition import PartitionedGraph, PartitionedMetapaths

from test_gpu_partition_gat import HUB_COL, LONG_ROW, N, _block, _gat64, _square
import test_gpu_partition_han as han_t

pytestmark = pytest.mark.gpu
DEV = "cuda"
BF = torch.bfloat16
# bf16 bounds against float64 / against the 1-GPU model: the tolerances of the bf16 parity tests
TOL_OUT, TOL_GRAD = 1e-2, 3e-2


def _rel(a, b):
    return float((a.double() - b.double()).abs().max()) / max(float(b.double().abs().max()), 1e-30)


def _grads(g, Wh, s, t, H, Fp, drop, d_out):
    Wh, s, t = (x.clone().requires_grad_() for x in (Wh, s, t))
    y = Fn.gat_aggregate(g, Wh, s, t, H, Fp, 0.2, elu=1, dropout=drop)
    return torch.autograd.grad(y, [Wh, s, t], d_out)


@pytest.mark.parametrize("where", ["first", "middle"])
@pytest.mark.parametrize("p", [0.0, 0.6])
@pytest.mark.parametrize("H,Fp", [(8, 8), (1, 7), (4, 16)])
def test_bf16_rectangular_block_matches_square_kernels(H, Fp, p, where):
    """(8, 8) and (4, 16) take the packed column-pair path, (1, 7) the unpacked one."""
    rowptr, col = _square(3)
    lo, hi = (0, N // 2) if where == "first" else (N // 3, 2 * N // 3)
    assert lo <= LONG_ROW < hi and not lo <= HUB_COL < hi
    g = CSRGraph(torch.from_numpy(rowptr).to(DEV), torch.from_numpy(col.astype(np.int32)).to(DEV), None, N, N)
    gb, table = _block(rowptr, col, lo, hi)
    assert gb.n_cols > gb.n_rows
    gen = torch.Generator(device=DEV).manual_seed(5)
    Wh = torch.randn(N, H * Fp, device=DEV, generator=gen).to(BF)
    s = torch.randn(N, H, device=DEV, generator=gen)
    t = torch.randn(N, H, device=DEV, generator=gen)
    drop = Fn.AttentionDropout(p, 777) if p else None
    drop_b = Fn.AttentionDropout(p, 777, None, int(rowptr[lo])) if p else None
    res = []
    for gg, W_, s_, t_, d_ in ((g, Wh, s, t, drop), (gb, Wh[table], s[lo:hi], t[table], drop_b)):
        pre = torch.empty((gg.n_rows, H * Fp), device=DEV, dtype=BF)
        act = torch.empty_like(pre)
        _, rm, rs = Fn.gat_fwd_raw(gg, W_, s_, t_, H, Fp, 0.2, elu=1, save_stats=True, out=pre, dropout=d_, out_act=act)
        res.append((pre, act, rm, rs))
    for a, b in zip(res[1], res[0]):
        assert torch.equal(a, b[lo:hi])
    d_blk = torch.randn(hi - lo, H * Fp, device=DEV, generator=gen).to(BF)
    d_out = torch.zeros(N, H * Fp, device=DEV, dtype=BF)
    d_out[lo:hi] = d_blk
    dWh_sq, ds_sq, dt_sq = _grads(g, Wh, s, t, H, Fp, drop, d_out)
    dWh_b, ds_b, dt_b = _grads(gb, Wh[table], s[lo:hi], t[table], H, Fp, drop_b, d_blk)
    assert dWh_b.dtype == BF and dWh_b.shape == (gb.n_cols, H * Fp)
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
    # the same fp32 sum in the same order, rounded once to bf16
    assert torch.equal(dWh_b[warp_both], dWh_sq[table][warp_both])
    if where == "first":
        assert torch.equal(dt_b[warp_both], dt_sq[table][warp_both])
    keep = Fn.attention_keep_mask_from_seed(g, H, drop) if p else None
    r_dWh, _, r_dt = _gat64(g, Wh, s, t, H, Fp, keep, d_out)
    r_dWh, r_dt = r_dWh[table], r_dt[table]
    # bf16 rounding points: out_pre, the pre-activation gradient and d_Wh itself
    for got, ref in ((dWh_b, r_dWh), (dt_b, r_dt), (dWh_b[one_only], r_dWh[one_only]),
                     (dt_b[one_only], r_dt[one_only])):
        assert _rel(got, ref) <= TOL_GRAD, _rel(got, ref)


# ---- batched rectangular (HAN's metapaths on a row block) -------------------------------------------------------

def _fwd(g, M, Wh, s, t, H, Fp, d, b=None):
    """bf16 training forward: the square batched entry (b None, batch_nodes) or the batched-rectangular one."""
    lib = _lib.load()
    lr, thr = g.gat_long_rows()
    n = g.n_rows // M
    pre = torch.empty(n, M * H * Fp, device=DEV, dtype=BF)
    act = torch.empty_like(pre)
    rm, rs = torch.empty(g.n_rows, H, device=DEV), torch.empty(g.n_rows, H, device=DEV)
    dd = C.byref(d) if d is not None else None
    p = Fn._p
    if b is None:
        rc = lib.gnn_gat_fused_fwd_train_bf16(p(g.rowptr), p(g.col), p(Wh), M * H * Fp, p(s), p(t), g.n_rows, g.nnz, H,
                                              Fp, 0.2, _lib.GAT_SOFTMAX, 2, None, None, dd, p(pre), p(act), M * H * Fp,
                                              p(rm), p(rs), p(lr), lr.numel(), thr, n, Fn._stream_ptr())
    else:
        rc = lib.gnn_gat_fused_fwd_batch_bf16(p(g.rowptr), p(g.col), p(Wh), M * H * Fp, p(s), p(t), g.nnz, H, Fp, 0.2,
                                              _lib.GAT_SOFTMAX, 2, None, dd, p(pre), p(act), M * H * Fp, p(rm), p(rs),
                                              p(lr), lr.numel(), thr, C.byref(b), Fn._stream_ptr())
    _lib.check(rc, "bf16 batched forward")
    return pre, act, rm, rs


def _bwd(g, M, Wh, s, t, H, Fp, d, fwd, d_act, b=None):
    lib = _lib.load()
    pre, _, rm, rs = fwd
    gt = g.transpose()
    (lr, thr), (lrt, _) = g.gat_long_rows(), gt.gat_long_rows()
    dWh, ds, dt = torch.empty_like(Wh), torch.empty_like(s), torch.empty_like(t)
    scratch = torch.empty(g.n_rows, 4, H, device=DEV)
    d_pre = torch.empty_like(pre)
    p = Fn._p
    common = (p(g.rowptr), p(g.col), p(gt.rowptr), p(gt.col), p(g.perm_t), p(Wh), M * H * Fp, p(s), p(t), p(rm), p(rs),
              p(pre), p(d_act), M * H * Fp)
    tail = (None, p(dWh), M * H * Fp, p(ds), p(dt), p(scratch), g.nnz, p(lr), lr.numel(), p(lrt), lrt.numel(), thr, 2,
            p(d_pre), C.byref(d) if d is not None else None)
    if b is None:
        rc = lib.gnn_gat_fused_bwd_bf16(*common, g.n_rows, H, Fp, 0.2, _lib.GAT_SOFTMAX, *tail, g.n_rows // M,
                                        Fn._stream_ptr())
    else:
        rc = lib.gnn_gat_fused_bwd_batch_bf16(*common, H, Fp, 0.2, _lib.GAT_SOFTMAX, *tail, C.byref(b),
                                              Fn._stream_ptr())
    _lib.check(rc, "bf16 batched backward")
    return dWh, ds, dt


def _inputs(M, n_rows, H, Fp, seed):
    Wh, s, t, gen = han_t._inputs(M, n_rows, H, Fp, seed)
    return Wh.to(BF), s, t, gen


@pytest.mark.parametrize("p", [0.0, 0.6])
@pytest.mark.parametrize("H,Fp", [(8, 8), (1, 16), (1, 7)])
@pytest.mark.parametrize("M", [2, 3])
def test_bf16_equal_strides_match_square_batched_kernels(M, H, Fp, p):
    _, g = han_t._set(M, 10)
    Wh, s, t, gen = _inputs(M, han_t.N, H, Fp, 1)
    d = Fn.AttentionDropout(p, 4242).c_struct() if p else None
    b = han_t._batch(M, han_t.N, han_t.N)
    sq = _fwd(g, M, Wh, s, t, H, Fp, d)
    rb = _fwd(g, M, Wh, s, t, H, Fp, d, b)
    for x, y in zip(rb, sq):
        assert torch.equal(x, y)
    d_act = torch.randn(han_t.N, M * H * Fp, device=DEV, generator=gen).to(BF)
    for x, y in zip(_bwd(g, M, Wh, s, t, H, Fp, d, rb, d_act, b), _bwd(g, M, Wh, s, t, H, Fp, d, sq, d_act)):
        assert torch.equal(x, y)


@pytest.mark.parametrize("where", ["first", "middle"])
@pytest.mark.parametrize("p", [0.0, 0.6])
@pytest.mark.parametrize("H,Fp", [(8, 8), (1, 16)])
def test_bf16_rank_block_with_union_halo_matches_whole_set(H, Fp, p, where):
    M, NN = 3, han_t.N
    gs, g = han_t._set(M, 20)
    lo, hi = (0, NN // 2) if where == "first" else (NN // 3, 2 * NN // 3)
    gb, table, shift = han_t._block_set(gs, lo, hi)
    n_loc, nc = hi - lo, table.numel()
    assert nc > n_loc
    Wh, s, t, gen = _inputs(M, NN, H, Fp, 5)
    d = Fn.AttentionDropout(p, 777).c_struct() if p else None
    Wh_b = Wh[table]
    s_b = s.view(M, NN, H)[:, lo:hi].reshape(M * n_loc, H)
    t_b = t.view(M, NN, H)[:, table].reshape(M * nc, H)
    sq = _fwd(g, M, Wh, s, t, H, Fp, d)
    rb = _fwd(gb, M, Wh_b, s_b, t_b, H, Fp, d, han_t._batch(M, n_loc, nc, shift))
    assert torch.equal(rb[0], sq[0][lo:hi]) and torch.equal(rb[1], sq[1][lo:hi])
    for x, y in zip(rb[2:], sq[2:]):
        assert torch.equal(x, y.view(M, NN, H)[:, lo:hi].reshape(M * n_loc, H))
    d_blk = torch.randn(n_loc, M * H * Fp, device=DEV, generator=gen).to(BF)
    d_act = torch.zeros(NN, M * H * Fp, device=DEV, dtype=BF)
    d_act[lo:hi] = d_blk
    dWh_sq, ds_sq, dt_sq = _bwd(g, M, Wh, s, t, H, Fp, d, sq, d_act)
    dWh_b, ds_b, dt_b = _bwd(gb, M, Wh_b, s_b, t_b, H, Fp, d, rb, d_blk, han_t._batch(M, n_loc, nc, shift))
    assert torch.equal(ds_b, ds_sq.view(M, NN, H)[:, lo:hi].reshape(M * n_loc, H))
    thr = _lib.get_tuning("gat.long_row")
    deg_sq = torch.bincount(g.col.long(), minlength=M * NN).view(M, NN)[:, table]
    deg_b = torch.bincount(gb.col.long(), minlength=M * nc).view(M, nc)
    warp_both = (deg_sq <= thr) & (deg_b <= thr)
    assert warp_both.sum() > 0
    dWh_sq_t = dWh_sq[table].view(nc, M, H * Fp).permute(1, 0, 2)
    dWh_b_t = dWh_b.view(nc, M, H * Fp).permute(1, 0, 2)
    dt_sq_t, dt_b_t = dt_sq.view(M, NN, H)[:, table], dt_b.view(M, nc, H)
    assert torch.equal(dWh_b_t[warp_both], dWh_sq_t[warp_both])
    if where == "first":
        assert torch.equal(dt_b_t[warp_both], dt_sq_t[warp_both])
    keep = Fn.attention_keep_mask_from_seed(g, H, Fn.AttentionDropout(p, 777)) if p else None
    r_dWh, _, r_dt = han_t._gat64(g, han_t._batched_rows(Wh, M, NN), s, t, H, Fp, keep,
                                  han_t._batched_rows(d_act, M, NN))
    r_dWh = r_dWh.view(M, NN, H * Fp)[:, table]
    r_dt = r_dt.view(M, NN, H)[:, table]
    assert _rel(dWh_b_t, r_dWh) <= TOL_GRAD and _rel(dt_b_t, r_dt) <= TOL_GRAD


def test_bf16_entries_refuse_bad_descriptions_before_launch():
    lib = _lib.load()
    args = (None, None, None, 8, None, None, 0, 1, 8, 0.2, 0, 0, None, None, None, None, 8, None, None, None, 0, 0)
    assert lib.gnn_gat_fused_fwd_batch_bf16(*args, C.byref(han_t._batch(33, 4, 4)), None) == 3  # n_graphs
    assert lib.gnn_gat_fused_fwd_batch_bf16(*args, C.byref(han_t._batch(2, 8, 4)), None) != 0  # rows > cols
    b = han_t._batch(2, 4, 4)
    b.struct_size = 8
    assert lib.gnn_gat_fused_fwd_batch_bf16(*args, C.byref(b), None) != 0
    assert lib.gnn_gat_fused_fwd_batch_bf16(*args, None, None) != 0
    bargs = (None,) * 6 + (8,) + (None,) * 6 + (8, 1, 8, 0.2, 0, None, None, 8, None, None, None, 0, None, 0, None, 0,
                                                 0, 0, None, None)
    for bad in (han_t._batch(33, 4, 4), han_t._batch(2, 8, 4)):
        assert lib.gnn_gat_fused_bwd_batch_bf16(*bargs, C.byref(bad), None) != 0
    b = han_t._batch(2, 4, 4)
    b.struct_size = 8
    assert lib.gnn_gat_fused_bwd_batch_bf16(*bargs, C.byref(b), None) != 0
    # the rectangular backward: fewer table rows than forward rows
    ex = (None,) * 6 + (8,) + (None,) * 6 + (8, 10, 5, 1, 8, 0.2, 0, None, None, 8, None, None, None, 0, None, 0, None,
                                             0, 0, 0, None, None, None)
    assert lib.gnn_gat_fused_bwd_ex_bf16(*ex) != 0


# ---- models on a one-rank bf16 partition --------------------------------------------------------------------------

def _run(model, x, adj, G, seed=123):
    torch.manual_seed(seed)
    Fn._drop_counters.clear()
    model.zero_grad(set_to_none=True)
    out = model(x, adj) if not isinstance(model, HANModel) else model(adj, x)
    (out.float() * G).sum().backward()
    return out.detach().clone(), {k: p.grad.clone() for k, p in model.named_parameters()}


def test_world_one_bf16_gcn_is_bit_identical():
    n, f_in = 5000, 37
    g = S.powerlaw_csr(n, 11.0, seed=31, device=DEV)
    gen = torch.Generator(device=DEV).manual_seed(2)
    x = torch.randn(n, f_in, device=DEV, generator=gen).to(BF)
    G = torch.randn(n, 41, device=DEV, generator=gen)
    torch.manual_seed(7)
    model = GCN_Model(f_in, 16, 41, 2, 0.5).to(DEV).to(BF).train()
    o1, g1 = _run(model, x, g, G)
    pg = PartitionedGraph.from_global(g, 0, 1, widths=[16, 41], dtype=BF)
    assert pg.dtype == BF
    o2, g2 = _run(model, x, pg, G)
    assert o2.dtype == BF and torch.equal(o1, o2)
    for k in g1:
        assert g2[k].dtype == BF and torch.equal(g1[k], g2[k]), k
    pg.close()


@pytest.mark.parametrize("cls", [GAT, SpGAT])
def test_world_one_bf16_gat_is_bit_identical(cls):
    n, f_in, nhid, nclass, heads = 700, 50, 8, 7, 8
    adj = torch.from_numpy(S.symmetric_mask(n, 12 * n, seed=1)).float().to(DEV)
    gen = torch.Generator(device=DEV).manual_seed(2)
    x = torch.randn(n, f_in, device=DEV, generator=gen).to(BF)
    G = torch.randn(n, nclass, device=DEV, generator=gen)
    torch.manual_seed(0)
    model = cls(f_in, nhid, nclass, 0.6, 0.2, heads).to(DEV).to(BF).train()
    o1, g1 = _run(model, x, adj, G)
    pg = PartitionedGraph.from_global(adj_cache.get(adj), 0, 1, widths=[heads * nhid, nclass], dtype=BF)
    o2, g2 = _run(model, x, pg, G)
    assert o2.dtype == BF and torch.equal(o1, o2)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k
    pg.close()


def _han_case(layers):
    n, f_in, hidden, classes, heads, M = 600, 40, 8, 3, 8, 3
    adjs = han_t._metapath_adjs(n, M, 1)
    gen = torch.Generator(device=DEV).manual_seed(2)
    x = torch.randn(n, f_in, device=DEV, generator=gen).to(BF)
    G = torch.randn(n, classes, device=DEV, generator=gen)
    torch.manual_seed(0)
    model = HANModel(M, f_in, hidden, classes, [heads] * layers, 0.6).to(DEV)
    pm = PartitionedMetapaths.from_global([adj_cache.get(a) for a in adjs], 0, 1, widths=[M * heads * hidden],
                                          dtype=BF)
    assert pm.dtype == BF
    return model, x, adjs, pm, G


def test_world_one_bf16_han_matches_one_gpu():
    """One layer in train mode (dropout 0.6): the node-level attention runs the same bf16 kernels and draws the same
    masks; the semantic attention differs (fp32 split kernels on the partition, the torch formula in bf16 on one GPU),
    so the bound is bf16's."""
    model, x, adjs, pm, G = _han_case(1)
    model = model.to(BF).train()
    o1, g1 = _run(model, x, adjs, G)
    o2, g2 = _run(model, x, pm, G)
    assert o2.dtype == BF
    errs = {k: _rel(g2[k], g1[k]) for k in g1}
    assert _rel(o2, o1) <= TOL_OUT, (_rel(o2, o1), errs)
    assert max(errs.values()) <= TOL_GRAD, errs
    pm.close()


def test_two_layer_bf16_han_partition_tracks_fp32():
    """Two layers: the two bf16 semantic formulations drift apart (a second layer starts from inputs that already
    differ by the first layer's rounding, and the semantic-score gradients are small differences of larger terms), so
    both bf16 runs are held against the same model in fp32 instead (eval mode: the same computation in every run).
    The partition's logits stay within 2 x 1e-2 of fp32, and its worst gradient (max-normalised error against fp32,
    over all parameters) is no worse than the 1-GPU bf16 model's worst.  Per parameter neither bf16 model is closer
    to fp32: the second layer's attention-vector gradients are sums over nodes that cancel to a fraction of their
    terms, and bf16 rounding moves them by up to 7 % on the partition and 23 % on one GPU (different parameters)."""
    import copy
    model, x, adjs, pm, G = _han_case(2)
    model.eval()
    m16 = copy.deepcopy(model).to(BF).eval()
    o_ref, g_ref = _run(model, x.float(), adjs, G)
    o1, g1 = _run(m16, x, adjs, G)
    o2, g2 = _run(m16, x, pm, G)
    assert _rel(o2, o_ref) <= 2 * TOL_OUT, (_rel(o2, o_ref), _rel(o1, o_ref))
    part = {k: _rel(g2[k], g_ref[k]) for k in g_ref}
    one = {k: _rel(g1[k], g_ref[k]) for k in g_ref}
    worst = max(part, key=part.get)
    assert part[worst] <= max(TOL_GRAD, max(one.values())), (worst, part[worst], max(one.values()))
    pm.close()


def test_dtype_mismatch_is_refused():
    n = 300
    g = adj_cache.get(torch.from_numpy(S.symmetric_mask(n, 12 * n, seed=3)).float().to(DEV))
    x = torch.randn(n, 20, device=DEV)
    p32 = PartitionedGraph.from_global(g, 0, 1, widths=[64, 16, 7])
    p16 = PartitionedGraph.from_global(g, 0, 1, widths=[64, 16, 7], dtype=BF)
    # a bf16 model on an fp32 partition: the message names the partition's fp32
    with pytest.raises(_lib.GnnError, match="fp32"):
        GAT(20, 8, 7, 0.0, 0.2, 8).to(DEV).to(BF)(x.to(BF), p32)
    with pytest.raises(_lib.GnnError, match="fp32"):
        GCN_Model(20, 16, 7, 2, 0.0).to(DEV).to(BF)(x.to(BF), p32)
    # an fp32 model on a bf16 partition
    with pytest.raises(_lib.GnnError, match="bf16"):
        GAT(20, 8, 7, 0.0, 0.2, 8).to(DEV)(x, p16)
    with pytest.raises(_lib.GnnError, match="bf16"):
        SpGAT(20, 8, 7, 0.0, 0.2, 8).to(DEV)(x, p16)
    with pytest.raises(_lib.GnnError, match="bf16"):
        GCN_Model(20, 16, 7, 2, 0.0).to(DEV)(x, p16)
    with pytest.raises(_lib.GnnError, match="bf16"):
        Fn.halo_exchange(p16, torch.randn(n, 64, device=DEV))
    p32.close()
    p16.close()
    gs = [adj_cache.get(a) for a in han_t._metapath_adjs(n, 2, 3)]
    pm = PartitionedMetapaths.from_global(gs, 0, 1, widths=[2 * 64], dtype=BF)
    with pytest.raises(_lib.GnnError, match="bf16"):
        HANLayer(2, 20, 8, 8, 0.0).to(DEV)(pm, x)
    pm.close()


# ---- two real ranks ----------------------------------------------------------------------------------------------

@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one node")
@pytest.mark.parametrize("tool,per_rank", [("gcn_dist_train.py", 2 * 3 * 3), ("gat_dist_train.py", 2 * 2 * 3),
                                           ("han_dist_train.py", 3)])
def test_two_rank_bf16_training_all_transports_check(tool, per_rank):
    """Two ranks train the bf16 model over p2p, ce and nccl and compare with the same bf16 model on one GPU: logits
    within 1e-2, step-1 gradients within 3e-2, the weights after 3 Adam steps within the tool's stated bound, and a
    bit-for-bit repeat."""
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
           "127.0.0.1", "--master-port", str(port), os.path.join(root, "tools", tool), "--check", "--dtype", "bf16",
           "--transports", "p2p", "ce", "nccl"]
    out = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 2 * per_rank, out.stdout[-2000:]
    for d in lines:
        assert d["dtype"] == "bf16"
        assert d["logits_rel_err"] <= TOL_OUT and d["grad_rel_err"] <= TOL_GRAD, d
        assert d["weights_norm_rel_err"] <= d["weights_bound"] and d["bitwise_repeat"], d
        assert d["ok"], d
