"""The gather over a feature table sharded into row blocks (gnn_gather_reduce_multi_sharded_*, partition.ShardedTable)
on one GPU: every reduced row bit for bit against the same gather over the concatenated table, the refusals of the C
ABI and of ShardedTable, GraphSage logits and gradients over ShardedTable.local against the tensor table, the captured
runner, and two real ranks through tools/sage_sharded.py."""
import ctypes as C

import pytest
import torch

from graphneuralnetwork_b200 import _lib, functional as Fn
from graphneuralnetwork_b200.graph import CSRGraph
from graphneuralnetwork_b200.layers import CapturedGraphSage, GraphSage
from graphneuralnetwork_b200.partition import ShardedTable

pytestmark = pytest.mark.gpu
DEV = "cuda"

# global row bounds of the shard layouts: uneven, an empty shard, a one-row shard
LAYOUTS = {
    1: [0, 997],
    2: [0, 400, 997],
    3: [0, 1, 600, 997],
    8: [0, 100, 100, 250, 251, 600, 700, 900, 997],
}


def _table(n, F, dtype, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(n, F, device=DEV, generator=g).to(dtype)


def _sharded(X, bounds):
    return ShardedTable.local([X[bounds[s]:bounds[s + 1]] for s in range(len(bounds) - 1)])


def _ids(bounds, n_src, fanout, id_dtype, seed):
    """Uniform ids, plus every shard boundary (first and last row of every shard), -1 and out-of-range ids."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    N = bounds[-1]
    ids = torch.randint(0, N, (n_src * fanout,), device=DEV, generator=g)
    edge = torch.tensor(sorted({b for b in bounds[:-1]} | {b - 1 for b in bounds[1:] if b > 0}), device=DEV)
    ids[:edge.numel()] = edge
    ids[edge.numel()] = -1
    ids[edge.numel() + 1] = N
    ids[edge.numel() + 2] = N + 5
    return ids.to(id_dtype)


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


@pytest.mark.parametrize("n_shards", [1, 2, 3, 8])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("reduce", ["mean", "sum", "max"])
@pytest.mark.parametrize("F", [64, 128, 602])
def test_sharded_gather_is_bit_identical(n_shards, dtype, reduce, F):
    bounds = LAYOUTS[n_shards]
    X = _table(bounds[-1], F, dtype, seed=n_shards)
    ref_table = Fn.pad_table(X)
    st = _sharded(X, bounds)
    if F * X.element_size() < 256:  # 64 bf16 columns: 128-byte rows, below what one bulk copy per row needs
        with pytest.raises(_lib.GnnError, match="TMA path only"):
            Fn.gather_reduce_multi_raw(st, [(None, 4, 2)], reduce)
        return
    for id_dtype in (torch.int32, torch.int64):
        b1 = (_ids(bounds, 70, 25, id_dtype, 1), 70, 25)
        b2 = (_ids(bounds, 300, 10, id_dtype, 2), 300, 10)
        b3 = (None, 40, 7)  # identity block: rows [0, 280)
        b4 = (_ids(bounds, 33, 1, id_dtype, 3), 33, 1)
        blocks = [b1, b2, b3, b4]
        want = Fn.gather_reduce_multi_raw(ref_table, blocks, reduce)
        got = Fn.gather_reduce_multi_raw(st, blocks, reduce)
        for w, g in zip(want, got):
            assert torch.equal(_bits(w.contiguous()), _bits(g.contiguous()))
    st.close()


def test_sharded_split_form_is_bit_identical():
    F, ld = 602, 604
    for n_shards in (1, 3, 8):
        bounds = LAYOUTS[n_shards]
        X = _table(bounds[-1], F, torch.float32, seed=7)
        st, ref = _sharded(X, bounds), Fn.pad_table(X)
        blocks = [(_ids(bounds, 64, 25, torch.int32, 4), 64, 25), (_ids(bounds, 64, 1, torch.int32, 5), 64, 1)]
        outs = []
        for table in (ref, st):
            Z = torch.zeros((128, 4 * ld), dtype=torch.float16, device=DEV)
            Fn.gather_reduce_multi_split_raw(table, blocks, "mean", [Z[:64, :F], Z[64:, :F]], lo_off=2 * ld)
            outs.append(Z)
        assert torch.equal(outs[0].view(torch.int16), outs[1].view(torch.int16))
        st.close()


def _call(lib, desc, ld, F, idx, out, reduce=0, dtype="f32", n_src=4, fanout=2):
    fn = {"f32": lib.gnn_gather_reduce_multi_sharded_f32, "bf16": lib.gnn_gather_reduce_multi_sharded_bf16}[dtype]
    idx_arr = (C.c_void_p * 1)(idx.data_ptr())
    n_arr, f_arr = (C.c_int64 * 1)(n_src), (C.c_int32 * 1)(fanout)
    o_arr, ldo = (C.c_void_p * 1)(out.data_ptr()), (C.c_int64 * 1)(out.stride(0))
    return fn(None if desc is None else C.byref(desc), ld, F, reduce, 1, idx_arr, 32, n_arr, f_arr, o_arr, ldo, None)


def test_sharded_abi_refusals():
    lib = _lib.load()
    F, ld = 128, 128
    shards = [torch.zeros((10, ld), device=DEV) for _ in range(2)]
    idx = torch.zeros(8, dtype=torch.int32, device=DEV)
    out = torch.full((4, F), 7.0, device=DEV)

    def desc(**kw):
        d = _lib.ShardedTableDesc()
        d.struct_size, d.n_shards = C.sizeof(d), 2
        d.base[0], d.base[1] = shards[0].data_ptr(), shards[1].data_ptr()
        d.row_begin[0], d.row_begin[1], d.row_begin[2] = 0, 10, 20
        for k, v in kw.items():
            if k == "base1":
                d.base[1] = v
            elif k == "rb1":
                d.row_begin[1] = v
            elif k == "rb0":
                d.row_begin[0] = v
            else:
                setattr(d, k, v)
        return d

    before = lib.gnn_launch_count()
    cases = [
        (None, ld, F, 1, b"null sharded table"),
        (desc(struct_size=8), ld, F, 1, b"struct_size"),
        (desc(n_shards=0), ld, F, 1, b"n_shards"),
        (desc(n_shards=9), ld, F, 1, b"n_shards"),
        (desc(rb0=1), ld, F, 1, b"row_begin[0]"),
        (desc(rb1=25), ld, F, 1, b"decreases"),
        (desc(base1=None), ld, F, 2, b"non-null"),
        (desc(base1=shards[1].data_ptr() + 4), ld, F, 2, b"16-byte aligned"),
        (desc(), 130, 129, 2, b"multiple of 16"),
        (desc(), 100, F, 1, b"smaller than F"),
        (desc(), ld, 48, 3, b"TMA path only"),  # 192-byte rows
    ]
    for d, ld_, F_, status, msg in cases:
        rc = _call(lib, d, ld_, F_, idx, out)
        assert rc == status, (msg, rc)
        assert msg in lib.gnn_last_error_string(), (msg, lib.gnn_last_error_string())
    rc = _call(lib, desc(), ld, 64, idx, out, dtype="bf16")  # 64 bf16 = 128 bytes
    assert rc == 3 and b"TMA path only" in lib.gnn_last_error_string()
    # an empty shard may have a null base; the call then runs
    torch.cuda.synchronize()
    assert lib.gnn_launch_count() == before
    d = desc(base1=None, rb1=20)
    assert _call(lib, d, ld, F, idx, out) == 0
    torch.cuda.synchronize()
    assert torch.equal(out, torch.zeros_like(out))


def test_sharded_table_refusals():
    X = torch.randn(50, 128, device=DEV)
    with pytest.raises(_lib.GnnError, match="requires grad"):
        ShardedTable.local([X.clone().requires_grad_()])
    with pytest.raises(_lib.GnnError, match="CPU"):
        ShardedTable.local([X.cpu()])
    with pytest.raises(_lib.GnnError, match="differ"):
        ShardedTable.local([X, X.bfloat16()])
    with pytest.raises(_lib.GnnError, match="differ"):
        ShardedTable.local([X, X[:, :64]])
    with pytest.raises(_lib.GnnError, match="at most|1 to 8"):
        ShardedTable.local([X[i:i + 5] for i in range(0, 45, 5)])
    with pytest.raises(_lib.GnnError, match="float32 or bfloat16"):
        ShardedTable.local([X.half()])
    st = ShardedTable.local([X[:20], X[20:]])
    with pytest.raises(_lib.GnnError, match="fp32 table only"):
        Fn.gather_reduce_multi_split_raw(ShardedTable.local([X.bfloat16()]), [], "mean", [], 0)
    assert st.shape == (50, 128) and st.stride(0) == 128 and not st.requires_grad
    assert st.abs_max == float(X.abs().max())
    st.close()


def _model(L, F, seed):
    torch.manual_seed(seed)
    hidden = [64] * (L - 1) + [41]
    fan = [5, 3, 2][:L]
    return GraphSage(F, hidden, fan).to(DEV), fan


def _blocks(N, fan, B, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    out = [torch.randint(0, N, (B,), device=DEV, generator=g, dtype=torch.int32)]
    for f in fan:
        out.append(torch.randint(0, N, (out[-1].numel() * f,), device=DEV, generator=g, dtype=torch.int32))
    return out


@pytest.mark.parametrize("L", [2, 3])
def test_graphsage_eval_logits_bit_identical(L):
    F, N = 602, 3001
    X = _table(N, F, torch.float32, seed=11)
    ref = Fn.pad_table(X)
    st = _sharded(X, [0, 1000, 1001, N])
    model, fan = _model(L, F, 3)
    model.eval()
    blocks = _blocks(N, fan, 64, 5)
    for tc in (True, False):  # fp16-split tensor-core product and the fp32 product (one-launch path at L = 2)
        model.tensor_core_gemm = tc
        with torch.no_grad():
            a = model.forward_sampled(ref, blocks)
            b = model.forward_sampled(st, blocks)
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), tc
    st.close()


@pytest.mark.parametrize("L", [2, 3])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_graphsage_training_loss_and_gradients_bit_identical(L, dtype):
    F, N = 602, 3001
    X = _table(N, F, dtype, seed=12)
    ref = Fn.pad_table(X)
    st = _sharded(X, [0, 1500, 1501, N])
    results = []
    for table in (ref, st):
        model, fan = _model(L, F, 4)
        model = model.to(dtype).train()
        blocks = _blocks(N, fan, 64, 6)
        y = torch.randint(0, 41, (64,), device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
        loss = torch.nn.functional.cross_entropy(model.forward_sampled(table, blocks).float(), y)
        loss.backward()
        results.append((loss.detach(), {k: p.grad.clone() for k, p in model.named_parameters()}))
    (l1, g1), (l2, g2) = results
    assert torch.equal(l1, l2)
    assert g1.keys() == g2.keys()
    for k in g1:
        assert torch.equal(_bits(g1[k]), _bits(g2[k])), k
    st.close()


def test_captured_runner_over_sharded_table():
    F, N = 602, 5000
    X = _table(N, F, torch.float32, seed=13)
    rng = torch.Generator().manual_seed(0)
    deg = torch.randint(1, 30, (N,), generator=rng)
    rowptr = torch.cat([torch.zeros(1, dtype=torch.int64), deg.cumsum(0)])
    col = torch.randint(0, N, (int(rowptr[-1]),), generator=rng, dtype=torch.int32)
    g = CSRGraph(rowptr.to(DEV), col.to(DEV), None, N, N)
    model, _ = _model(2, F, 5)
    model.eval()
    st = _sharded(X, [0, 2000, 3500, N])
    ref = Fn.pad_table(X)
    r_sh = CapturedGraphSage(model, st, batch=128, adjacency=g, seed=9)
    r_ref = CapturedGraphSage(model, ref, batch=128, adjacency=g, seed=9)
    ids = torch.randint(0, N, (128,), dtype=torch.int32, generator=rng).pin_memory()
    for _ in range(3):
        a = r_sh(ids).clone()
        b = r_ref(ids).clone()
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
        assert torch.isfinite(a).all()
    st.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one node")
def test_two_rank_sharded_table_check():
    """Two real ranks over peer mappings: each rank's sharded gather and one training step against a replica of the
    table, identical weights across the ranks after 3 Adam steps, and those weights against one process that runs
    the union of the ranks' minibatches."""
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
           "127.0.0.1", "--master-port", str(port), os.path.join(root, "tools", "sage_sharded.py"), "--check"]
    out = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [json.loads(l) for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 2, out.stdout[-2000:]
    for d in lines:
        assert d["gather_bitwise"] and d["step_bitwise"] and d["weights_equal_across_ranks"], d
        assert d["weights_vs_union_max_abs"] <= 1e-5, d
