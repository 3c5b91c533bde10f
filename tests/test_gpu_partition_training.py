"""Partitioned GCN training on the GPU: the bias/ReLU epilogue in every consumer form of the extended SpMM entry
point (gnn_spmm_csr_ex_*), the consumers of a two-rank step built in one process with the epilogue on, the
drop-in GCN_Model on a one-rank PartitionedGraph against the same model on the CSRGraph, and two real ranks
training through tools/gcn_dist_train.py --check."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import rel_err
from graphneuralnetwork_b200 import _lib, functional as Fn
from graphneuralnetwork_b200.graph import CSRGraph
from graphneuralnetwork_b200.layers import GCN_Model
from graphneuralnetwork_b200.partition import Consumer, PartitionedGraph, PartitionedSpmm, select_rows
from test_gpu_partition import _graph, _push, _two_rank_plans

pytestmark = pytest.mark.gpu
DEV = "cuda"


def cuda(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return t.to(DEV) if dtype is None else t.to(DEV, dtype)


def _epilogue(y, b, relu):
    y = y + b.astype(np.float64)
    return np.maximum(y, 0.0) if relu else y


@pytest.mark.parametrize("F", [7, 16, 41, 128, 602])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("skip_frac", [0.25, 0.75])
def test_spmm_ex_epilogue_with_accumulate_two_tables_and_skip_prefix(lib, F, dtype, skip_frac):
    """ONE launch: row map (not ascending), accumulate_prefix, a second table, bias, ReLU and epilogue_skip_prefix.
    Compact rows [0, k) add into Y, the rest overwrite; rows [0, s) get no epilogue, the others relu(. + b) after
    the add — against float64."""
    n_rows, n_loc, n_halo = 3000, 2500, 700
    rowptr, col, val = _graph(n_rows, n_loc + n_halo, 9, seed=F, long_row=(1234, 5000))
    rng = np.random.default_rng(F + 1)
    X = rng.standard_normal((n_loc, F)).astype(np.float32)
    H = rng.standard_normal((n_halo, F)).astype(np.float32)
    Y0 = rng.standard_normal((n_rows, F)).astype(np.float32)
    b = rng.standard_normal(F).astype(np.float32)
    if dtype == torch.bfloat16:
        X, H, Y0 = [torch.from_numpy(a).bfloat16().float().numpy() for a in (X, H, Y0)]
    rows = np.union1d(rng.choice(n_rows, size=1700, replace=False), [1234])
    rows = rng.permutation(rows)  # the partitioned P1 lists its rows in two ascending runs
    k, s = len(rows) // 2, int(len(rows) * skip_frac)
    rp, cc, vv = select_rows(torch.from_numpy(rowptr), torch.from_numpy(col), torch.from_numpy(val),
                             torch.from_numpy(rows))
    g = CSRGraph(rp.to(DEV), cc.to(DEV), vv.to(DEV), len(rows), n_loc + n_halo)
    assert g.long_row_plan() is not None  # the long row takes the chunked path and its finalize
    Xd, Hd = Fn._padded_empty(n_loc, F, dtype, DEV), Fn._padded_empty(n_halo, F, dtype, DEV)
    Xd.copy_(cuda(X, dtype))
    Hd.copy_(cuda(H, dtype))
    A = sp.csr_matrix((val.astype(np.float64), col, rowptr), shape=(n_rows, n_loc + n_halo))
    full = A @ np.vstack([X, H]).astype(np.float64)
    ref = Y0.astype(np.float64).copy()
    ref[rows[:k]] += full[rows[:k]]
    ref[rows[k:]] = full[rows[k:]]
    ref[rows[s:]] = _epilogue(ref[rows[s:]], b, True)
    Y = cuda(Y0, dtype)
    Fn.spmm_ex(g, Xd, Y, row_map=cuda(rows.astype(np.int32)), accumulate_prefix=k, X2=Hd, split=n_loc,
               bias=cuda(b), relu=True, epilogue_skip_prefix=s)
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    got = Y.float().cpu().numpy()
    assert rel_err(got, ref) < tol
    untouched = np.setdiff1d(np.arange(n_rows), rows)
    assert np.array_equal(got[untouched], Y0[untouched])
    # the remote pass: every row accumulates, then relu(y_prev + sum + b)
    Y = cuda(Y0, dtype)
    Fn.spmm_ex(g, Xd, Y, row_map=cuda(rows.astype(np.int32)), accumulate=True,
               X2=Hd, split=n_loc, bias=cuda(b), relu=True)
    ref2 = _epilogue(Y0.astype(np.float64)[rows] + full[rows], b, True)
    assert rel_err(Y.float().cpu().numpy()[rows], ref2) < tol


def test_spmm_ex_previous_struct_size_and_planned_refusal(lib):
    """The layout before epilogue_skip_prefix (struct_size = its offset) is accepted and reads as 0; any other
    size is refused; the planned entry still refuses accumulate together with bias/ReLU."""
    rowptr, col, val = _graph(200, 200, 5, seed=4)
    g = CSRGraph(cuda(rowptr), cuda(col), cuda(val), 200, 200)
    X = torch.randn(200, 16, device=DEV)
    b = torch.randn(16, device=DEV)
    want = torch.relu(Fn.spmm_raw(g, X) + b)
    for size, status in [(_lib.SpmmOpts.epilogue_skip_prefix.offset, 0), (C.sizeof(_lib.SpmmOpts), 0),
                         (_lib.SpmmOpts.epilogue_skip_prefix.offset - 8, 1), (C.sizeof(_lib.SpmmOpts) + 8, 1)]:
        o = _lib.SpmmOpts()
        o.struct_size, o.relu, o.bias = size, 1, b.data_ptr()
        o.epilogue_skip_prefix = 0 if size == C.sizeof(_lib.SpmmOpts) else 150  # must not be read at the old size
        Y = torch.full_like(want, 9.0)
        st = lib.gnn_spmm_csr_ex_f32(g.rowptr.data_ptr(), g.col.data_ptr(), g.val.data_ptr(), X.data_ptr(), Y.data_ptr(),
                                     200, 200, 16, 16, 16, C.byref(o), torch.cuda.current_stream().cuda_stream)
        assert st == status, size
        if status == 0:
            assert torch.allclose(Y, want, rtol=1e-6, atol=1e-6)
    with pytest.raises(_lib.GnnError):
        Fn.spmm_raw(g, X, out=torch.zeros_like(X), accumulate=True, bias=b)
    with pytest.raises(_lib.GnnError):
        Fn.spmm_raw(g, X, out=torch.zeros_like(X), accumulate=True, relu=True)


def _signed_two_rank_case(seed):
    """A graph whose local columns pull rows down and remote columns push them up: many two-pass rows have a
    negative local partial and a positive total (an epilogue on the first pass would zero them)."""
    n, F = 6000, 41
    rowptr, col, val = _graph(n, n, 12, seed=seed, long_row=(10, 4000))
    bounds = [0, 2900, n]
    row_of = np.repeat(np.arange(n), np.diff(rowptr))
    owner_row = (row_of >= bounds[1]).astype(int)
    owner_col = (col >= bounds[1]).astype(int)
    val = np.where(owner_row == owner_col, -np.abs(val), 3.0 * np.abs(val)).astype(np.float32)
    X = np.abs(np.random.default_rng(seed + 1).standard_normal((n, F))).astype(np.float32)
    return n, F, rowptr, col, val, X, bounds


def _exchange(lib, plans, Xs, F):
    halos = [torch.full((max(p.n_halo, 1), F), float("nan"), device=DEV) for p in plans]
    for r, plan in enumerate(plans):
        q = 1 - r
        send = plan.send_rows.to(DEV)
        for w in range(plan.waves):
            bb = sum(plan.send_wave_counts[q][:w])
            seg_begin, seg_rows, dst_row = [0, 0], [0, 0], [0, 0]
            seg_begin[q] = plan.send_off()[q] + bb
            seg_rows[q] = plan.send_wave_counts[q][w]
            dst_row[q] = plan.dst_off[q] + bb
            _lib.check(_push(lib, Xs[r], send, seg_begin, seg_rows, [halos[0], halos[1]], dst_row, F, F, 4, 1), "push")
    torch.cuda.synchronize()
    return halos


def _consumers(plan, p1, X, halo, bias, relu, sentinel=None):
    op = PartitionedSpmm.__new__(PartitionedSpmm)  # consumers only: no process group in this test
    op.plan, op.dev, op._cons = plan, torch.device(DEV), {}
    Y = torch.full((plan.n_local, X.shape[1]), 123.0 if sentinel is None else sentinel, device=DEV)
    written = np.zeros(plan.n_local, bool)
    for c in [p1] + list(plan.p2):
        if c is None:
            continue
        op._run(c, X, halo, Y, 0, bias, relu)
        written[np.arange(plan.n_local) if c.row_map is None else c.row_map.numpy()] = True
        if sentinel is not None:  # rows no consumer has written yet are untouched
            assert torch.all(Y[torch.from_numpy(~written).to(DEV)] == sentinel)
    assert written.all()
    return Y


def _old_p1(plan):
    """P1 as it was built before the two-pass rows were moved to its front: every kept row in ascending order."""
    n_loc = plan.n_local
    mixed = (plan.rowptr_rem[1:] - plan.rowptr_rem[:-1]) > 0
    rows = torch.arange(n_loc)
    keep = (~mixed) | (rows < plan.chunk_bounds[plan.two_pass_chunks])
    if plan.two_pass_chunks == plan.waves:
        return Consumer("local", plan.rowptr_loc, plan.col_loc, plan.val_loc, None, n_loc)
    rows = rows[keep]
    rp, cc, vv = select_rows(plan.rowptr_loc, plan.col_loc, plan.val_loc, rows)
    return Consumer("local", rp, cc, vv, rows.to(torch.int32), n_loc)


@pytest.mark.parametrize("c0", [0, 2, 4])
def test_two_rank_consumers_with_fused_epilogue(lib, c0):
    n, F, rowptr, col, val, X, bounds = _signed_two_rank_case(21)
    blocks = [(torch.from_numpy(rowptr[lo:hi + 1] - rowptr[lo]), torch.from_numpy(col[rowptr[lo]:rowptr[hi]]),
               torch.from_numpy(val[rowptr[lo]:rowptr[hi]])) for lo, hi in zip(bounds[:-1], bounds[1:])]
    plans = _two_rank_plans(blocks, bounds, 4, c0, F)
    Xs = [cuda(X[bounds[r]:bounds[r + 1]]) for r in range(2)]
    halos = _exchange(lib, plans, Xs, F)
    b = np.random.default_rng(5).uniform(0.2, 0.6, F).astype(np.float32)
    bias = cuda(b)
    A = sp.csr_matrix((val.astype(np.float64), col, rowptr), shape=(n, n))
    full = A @ X.astype(np.float64)
    ref = _epilogue(full, b, True)
    hits = 0
    for r, plan in enumerate(plans):
        lo, hi = bounds[r], bounds[r + 1]
        assert plan.waves == 4 and plan.two_pass_chunks == c0
        skip = plan.p1.epilogue_skip
        if c0 > 0:  # two-pass rows whose local partial is negative and total positive
            first = plan.p1.row_map[:skip].long().numpy()
            loc = sp.csr_matrix((plan.val_loc.numpy().astype(np.float64), plan.col_loc.numpy(), plan.rowptr_loc.numpy()),
                                shape=(hi - lo, hi - lo)) @ X[lo:hi].astype(np.float64)
            hits += int(np.sum((loc[first] + b < 0) & (full[lo:hi][first] + b > 0)))
        Y = _consumers(plan, plan.p1, Xs[r], halos[r], bias, True, sentinel=123.0)
        assert rel_err(Y.cpu().numpy(), ref[lo:hi]) < 1e-5
        assert torch.equal(Y, _consumers(plan, plan.p1, Xs[r], halos[r], bias, True))  # deterministic
        # no epilogue: the reordered P1 gives the same bits as the ascending one
        assert torch.equal(_consumers(plan, plan.p1, Xs[r], halos[r], None, False),
                           _consumers(plan, _old_p1(plan), Xs[r], halos[r], None, False))
    if c0 > 0:
        assert hits > 50, hits


def _model_pair(layers, g, F_in, seed):
    torch.manual_seed(seed)
    a = GCN_Model(F_in, 16, 41, layers, 0.0).to(DEV)
    b = GCN_Model(F_in, 16, 41, layers, 0.0).to(DEV)
    b.load_state_dict(a.state_dict())
    return a, b


@pytest.mark.parametrize("layers", [2, 3])
def test_world1_partitioned_graph_matches_csr_graph_bitwise(lib, layers):
    """One rank: GCN_Model on a PartitionedGraph runs the same kernels as on the CSRGraph — outputs and
    gradients bit-identical; the state_dict keys are the reference's."""
    n, F_in = 5000, 37
    rowptr, col, val = _graph(n, n, 11, seed=31, long_row=(17, 4500))
    g = CSRGraph(cuda(rowptr), cuda(col), cuda(val), n, n)
    pg = PartitionedGraph.from_global(g, 0, 1, widths=[16, 41])
    X = torch.randn(n, F_in, device=DEV)
    target = torch.randint(0, 41, (n,), device=DEV)
    idx = torch.arange(0, n, 3, device=DEV)
    m_csr, m_pg = _model_pair(layers, g, F_in, 7)
    assert list(m_pg.state_dict()) == list(m_csr.state_dict())
    assert "gcn_blocks.gcn0.dense.weight" in m_pg.state_dict() and "gcn_blocks.gcn0.bias" in m_pg.state_dict()
    outs = []
    for m, adj in [(m_csr, g), (m_pg, pg)]:
        out = m(X, adj)
        torch.nn.functional.cross_entropy(out[idx], target[idx]).backward()
        outs.append((out.detach(), {k: p.grad for k, p in m.named_parameters()}))
    (o1, g1), (o2, g2) = outs
    assert torch.equal(o1, o2)
    for k in g1:
        assert torch.equal(g1[k], g2[k]), k
    assert torch.equal(pg.local_index(torch.tensor([4999, 3, 0], device=DEV)), torch.tensor([4999, 3, 0], device=DEV))
    with pytest.raises(_lib.GnnError):
        pg.op(99)
    pg.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one node")
def test_two_rank_gcn_training_all_transports_check():
    """Two real ranks train GCN_Model on a PartitionedGraph (Cora-like graph and a 200 k-row power-law graph,
    widths 16 / 41) over p2p, ce and nccl with fixed and automatic schedules; every rank compares its rows of the
    logits, the step-1 gradients and the weights after 3 Adam steps with the same model trained on one GPU, and
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
           "127.0.0.1", "--master-port", str(port), os.path.join(root, "tools", "gcn_dist_train.py"), "--check",
           "--transports", "p2p", "ce", "nccl", "--configs", "1:auto", "4:2", "auto:auto"]
    out = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 2 * 2 * 3 * 3, out.stdout[-2000:]  # ranks x graphs x transports x configs
    for d in lines:
        tag = (d["graph"], d["transport"], d["config"], d["rank"])
        assert d["logits_rel_err"] <= 1e-5 and d["grad_rel_err"] <= 2e-5, (tag, d)
        assert d["weights_rel_err"] <= 1e-4 and d["bitwise_repeat"], (tag, d)
