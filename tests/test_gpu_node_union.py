"""gnn_node_union (csrc/node_union.cu) bit for bit against np.unique(..., return_inverse=True): random, ragged and
duplicate-heavy inputs, -1 padding, empty sides, int32 and int64 ids (ids past 2^31 too), repeats, and every refusal."""
import ctypes as C

import numpy as np
import pytest
import torch
from hypothesis import HealthCheck, given, settings, strategies as st

from graphneuralnetwork_b200 import _lib, functional as Fn

DEV = "cuda"
SETTINGS = dict(max_examples=60, deadline=None, suppress_health_check=[HealthCheck.function_scoped_fixture])


def _expected(a, b):
    valid = np.concatenate([a[a >= 0], b[b >= 0]])
    uniq = np.unique(valid)
    pos = lambda x: np.where(x >= 0, np.searchsorted(uniq, x), -1).astype(np.int64)  # noqa: E731
    if valid.size:  # the inverse of np.unique is the map over the valid slots
        _, inv = np.unique(valid, return_inverse=True)
        assert np.array_equal(inv, np.concatenate([pos(a)[a >= 0], pos(b)[b >= 0]]))
    return uniq, pos(a), pos(b)


def _check(a, b, dtype):
    out, count, map_a, map_b = Fn.node_union(torch.from_numpy(a.astype(dtype)).to(DEV),
                                             torch.from_numpy(b.astype(dtype)).to(DEV))
    uniq, ea, eb = _expected(a, b)
    n = int(count.item())
    assert n == uniq.size
    out = out.cpu().numpy()
    assert out.dtype == dtype and out.size == a.size + b.size
    assert np.array_equal(out[:n], uniq.astype(dtype)) and (out[n:] == -1).all()
    assert np.array_equal(map_a.cpu().numpy(), ea) and np.array_equal(map_b.cpu().numpy(), eb)
    return out, map_a.cpu().numpy(), map_b.cpu().numpy()


@st.composite
def inputs(draw):
    n_a = draw(st.integers(0, 300))
    n_b = draw(st.integers(0, 900))
    wide = draw(st.booleans())
    hi = draw(st.sampled_from([3, 50, 5000, 2 ** 31 - 1] + ([2 ** 40] if wide else [])))
    seed = draw(st.integers(0, 2 ** 31 - 1))
    rng = np.random.default_rng(seed)
    a = rng.integers(0, hi, n_a)
    b = rng.integers(0, hi, n_b)
    if n_b and draw(st.booleans()):  # -1 padding, from a few ids to every id
        b[rng.random(n_b) < draw(st.floats(0.0, 1.0))] = -1
    if n_a and draw(st.booleans()):  # a padded set as the first side
        a[rng.random(n_a) < 0.2] = -1
    if n_a and n_b and draw(st.booleans()):  # the second side repeats the first (a node's own neighbours)
        b[: min(n_a, n_b)] = a[: min(n_a, n_b)]
    return a, b, (np.int64 if wide else draw(st.sampled_from([np.int32, np.int64])))


@pytest.mark.gpu
@settings(**SETTINGS)
@given(inputs())
def test_node_union_matches_numpy_unique(lib, case):
    a, b, dtype = case
    _check(a, b, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_node_union_edge_cases(lib, dtype):
    rng = np.random.default_rng(3)
    _check(np.full(7, -1), np.full(40, -1), dtype)  # nothing valid: count 0, all -1
    _check(np.zeros(0, np.int64), rng.integers(-1, 20, 100), dtype)  # n_a = 0
    _check(rng.integers(0, 20, 100), np.zeros(0, np.int64), dtype)  # n_b = 0
    _check(np.full(50, 7), np.full(500, 7), dtype)  # one id everywhere
    _check(np.arange(1000)[::-1].copy(), np.arange(1000), dtype)
    _check(rng.integers(0, 2 ** 31 - 1, 70000), rng.integers(0, 300, 200000), dtype)  # many keys, many CTAs
    out, _, _ = _check(np.zeros(0, np.int64), np.zeros(0, np.int64), dtype)
    assert out.size == 0


@pytest.mark.gpu
def test_node_union_int64_ids_past_2_31(lib):
    big = np.array([2 ** 31, 2 ** 33 + 5, 2 ** 62, 2 ** 31 - 1, 0], np.int64)
    out, ma, mb = _check(big, np.concatenate([big[::-1], [-1, 2 ** 31]]), np.int64)
    assert out[:5].tolist() == sorted(big.tolist())


@pytest.mark.gpu
def test_node_union_repeats_bit_for_bit(lib):
    rng = np.random.default_rng(11)
    for dtype in (torch.int32, torch.int64):
        a = torch.from_numpy(rng.integers(0, 5000, 3000)).to(DEV, dtype)
        b = torch.from_numpy(rng.integers(-1, 5000, 30000)).to(DEV, dtype)
        r1, r2 = Fn.node_union(a, b), Fn.node_union(a, b)
        for x, y in zip(r1, r2):
            assert torch.equal(x, y)


def test_node_union_refusals(lib):
    """Bad sizes, id widths and null pointers return GNN_ERR_BAD_ARG before any CUDA call (runs without a GPU)."""
    BAD = 1
    nb = C.c_size_t(0)
    assert lib.gnn_node_union_workspace_size(-1, 4, C.byref(nb)) == BAD
    assert lib.gnn_node_union_workspace_size(2 ** 30, 2 ** 30, C.byref(nb)) == BAD
    assert lib.gnn_node_union_workspace_size(4, 4, None) == BAD
    fake = 256  # never dereferenced: every call below is refused first
    args = dict(ids_a=fake, n_a=4, ids_b=fake, n_b=4, id_bits=64, out=fake, count=fake, map_a=fake, map_b=fake)

    def call(**kw):
        a = dict(args, **kw)
        return lib.gnn_node_union(a["ids_a"], a["n_a"], a["ids_b"], a["n_b"], a["id_bits"], a["out"], a["count"],
                                  a["map_a"], a["map_b"], fake, 1 << 20, None)

    assert call(n_a=-1) == BAD and b"bad size" in lib.gnn_last_error_string()
    assert call(n_b=2 ** 31) == BAD
    assert call(id_bits=16) == BAD and b"id_bits" in lib.gnn_last_error_string()
    for name in ("ids_a", "ids_b", "out", "count", "map_a", "map_b"):
        assert call(**{name: None}) == BAD, name
    # a side of size 0 needs no pointers, but the count always does
    assert call(n_a=0, n_b=0, ids_a=None, ids_b=None, out=None, map_a=None, map_b=None, count=None) == BAD


@pytest.mark.gpu
def test_node_union_short_workspace_and_mixed_dtypes(lib):
    a = torch.arange(10, device=DEV)
    count = torch.empty(1, dtype=torch.int64, device=DEV)
    m = torch.empty(10, dtype=torch.int64, device=DEV)
    out = torch.empty(20, dtype=torch.int64, device=DEV)
    ws = torch.empty(16, dtype=torch.uint8, device=DEV)
    rc = lib.gnn_node_union(a.data_ptr(), 10, a.data_ptr(), 10, 64, out.data_ptr(), count.data_ptr(), m.data_ptr(),
                            m.data_ptr(), ws.data_ptr(), 16, torch.cuda.current_stream().cuda_stream)
    assert rc == 5  # GNN_ERR_WORKSPACE
    with pytest.raises(_lib.GnnError):
        Fn.node_union(a, a.to(torch.int32))
