"""The gather-reduce kernels (csrc/sage.cu: the TMA ring; csrc/rowreduce.cuh: the vector-load kernel) held to a
float64 reference element by element, at every kernel variant the host dispatch can pick, and the tail-store
contract of the row-parallel output paths (gather and SpMM): a kernel writes the F columns of each output row and
nothing past them, so a padded buffer's pad columns and an adjacent output slice are left as they were.

Reference: the stored values reduced in float64 over the fanout.  Ids < 0 or >= N contribute nothing (mean still
divides by the fanout); under max a source without a valid id is -inf.  Bounds, per element:
  - fp32 mean / sum: |got - ref| <= (K + 2) * 2^-24 * scale * sum_k |x_k|  (scale = 1/K for mean, else 1)
  - bf16 outputs: the same bound (widened by the final rounding) plus 2^-8 * |ref|
  - max: the same bits, and the argmax is the first k that attains the max (where torch.max routes its gradient).

Every GPU test carries the `gpu` mark; `test_sweep_reaches_every_variant` needs no device."""
import contextlib

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from graphneuralnetwork_b200 import _lib, functional as Fn, layers
from graphneuralnetwork_b200.graph import CSRGraph
from graphneuralnetwork_b200.partition import ShardedTable

gpu = pytest.mark.gpu
DEV = "cuda"
U32 = 2.0 ** -24
ESZ = {torch.float32: 4, torch.bfloat16: 2}
SHORT = {torch.float32: "f32", torch.bfloat16: "bf16"}
SENTINEL = -96.5  # exact in fp32, bf16 and fp16; every pad column starts as it and must end as it
CONSUMER_THREADS = 160  # sage.cu kConsumerThreads


def _round_up(x, a):
    return (x + a - 1) // a * a


# ------------------------------------------------------------------------------ which kernel a call reaches
def gather_variant(dtype, F, ld, reduce, ldo=None, force_ldg=0, packed_add=-1, sharded=False, table_align=16,
                   out_align=16):
    """The kernel instantiation one block of `gather_reduce_impl` (csrc/sage.cu) launches, for a table of row
    stride `ld` and an output of row stride `ldo` (default `ld`) whose base pointers are aligned to
    `table_align` / `out_align` bytes:
      - TMA ring: ("tma", dtype, OP, NV, PK, SH, store) = `sage_tma_kernel<T, NV, OP, PK, SH>` and whether the
        reduced row leaves in 16-byte vectors ("vec16") or element by element ("scalar", `out_vec16 == 0`);
      - vector-load: ("ldg", dtype, OP, VEC, tiles), tiles = the (GROUP, CHUNKS) of each column tile of
        `row_reduce_kernel` (`pick_vec` / `launch_row_reduce_vec`, csrc/rowreduce.cuh).
    OP is SUM for mean and sum (mean is a scale), MAX for max.  This function restates the C++ host dispatch
    (sage.cu `gather_reduce_impl` / `launch_tma*`, rowreduce.cuh `pick_vec` / `launch_row_reduce*`): when that
    dispatch changes, this must change with it, or the test ids and the coverage test stop describing what runs."""
    esz = ESZ[dtype]
    ldo = ld if ldo is None else ldo
    op = "MAX" if reduce == "max" else "SUM"
    row_bytes = _round_up(F * esz, 16)
    tma = sharded or (not force_ldg and table_align % 16 == 0 and ld * esz % 16 == 0 and row_bytes <= ld * esz
                      and row_bytes >= 256 and row_bytes // 16 <= 4 * CONSUMER_THREADS)
    if tma:
        nvec, E = row_bytes // 16, 16 // esz
        pk = op != "MAX" and (esz == 2 if packed_add < 0 else packed_add != 0)
        vec16 = out_align % 16 == 0 and ldo * esz % 16 == 0 and nvec * E <= ldo
        return ("tma", SHORT[dtype], op, -(-nvec // CONSUMER_THREADS), int(pk), bool(sharded),
                "vec16" if vec16 else "scalar")
    v = 16 // esz
    while v > 1:
        fpad = _round_up(F, v)
        if table_align % (v * esz) == 0 and out_align % (v * esz) == 0 and ld % v == 0 and ldo % v == 0 \
                and fpad <= ld and fpad <= ldo:
            break
        v >>= 1
    vec = 8 if (esz == 2 and v == 8) else (4 if v >= 4 else v)
    tiles = []
    for c0 in range(0, F, 256 * vec):
        nv = -(-min(F - c0, 256 * vec) // vec)
        for lim, gc in ((4, (4, 1)), (8, (8, 1)), (16, (16, 1)), (32, (32, 1)), (64, (32, 2)), (96, (32, 3)),
                        (128, (32, 4)), (160, (32, 5)), (192, (32, 6)), (1 << 30, (32, 8))):
            if nv <= lim:
                tiles.append(gc)
                break
    return ("ldg", SHORT[dtype], op, vec, tuple(tiles))


def variant_id(v):
    if v[0] == "tma":
        return f"tma-{v[1]}-{v[2]}-NV{v[3]}-PK{v[4]}-{'sharded' if v[5] else 'plain'}-{v[6]}"
    return f"ldg-{v[1]}-{v[2]}-VEC{v[3]}-" + "+".join(f"G{g}C{c}" for g, c in v[4])


# ------------------------------------------------------------------------------ the sweep
# TMA ring: NV 1/2/3/4 per dtype; the table's row stride is F (already 16-byte rows)
TMA_F = {torch.float32: (64, 700, 1500, 2560), torch.bfloat16: (128, 1400, 3000, 5120)}
TMA_REDUCE = (("mean", 0), ("mean", 1), ("sum", 0), ("sum", 1), ("max", -1))
FANOUTS = (1, 7, 32, 33, 40)


def _tma_ldo(dtype, F, layout):
    """Output row stride: a 16-byte multiple with room past the last vector, or one that is not (scalar stores)."""
    E = 16 // ESZ[dtype]
    return _round_up(F, E) + E if layout == "vec16" else F + 1


def _tma_cases():
    out = []
    for dtype, Fs in TMA_F.items():
        for nv, F in enumerate(Fs, 1):
            for sharded in (False, True):
                layout = "scalar" if (nv + sharded) % 2 else "vec16"
                for reduce, pk in TMA_REDUCE:
                    v = gather_variant(dtype, F, F, reduce, ldo=_tma_ldo(dtype, F, layout), packed_add=pk,
                                       sharded=sharded)
                    out.append(pytest.param(dtype, F, reduce, pk, sharded, layout,
                                            id=f"F{F}-{reduce}-{variant_id(v)}"))
    return out


# vector-load kernel: (F, table row stride) per dtype; the stride picks VEC (odd: 1, 2 mod 4: 2, ...), F picks the
# (GROUP, CHUNKS) bucket of each column tile; the output has the table's row stride
LDG_SHAPES = {
    torch.float32: [(7, 12), (30, 32), (41, 44), (100, 104), (250, 252), (380, 384), (500, 504), (602, 608),
                    (700, 704), (1000, 1004), (2000, 2004),                       # VEC 4; 2000: two tiles
                    (41, 42), (602, 606), (1100, 1102),                           # VEC 2; 1100: three tiles
                    (7, 7), (300, 301), (602, 603)],                              # VEC 1; 300: two tiles
    torch.bfloat16: [(7, 8), (60, 64), (130, 136), (605, 608), (1000, 1008), (1400, 1408), (2100, 2104),  # VEC 8
                     (41, 44), (605, 612),                                        # VEC 4
                     (130, 134),                                                  # VEC 2
                     (7, 7), (300, 301)],                                         # VEC 1
}
LDG_FANOUTS = (1, 7, 33)


def _ldg_force(dtype, F, ld):
    return int(gather_variant(dtype, F, ld, "sum")[0] == "tma")


def _ldg_cases():
    out = []
    for dtype, shapes in LDG_SHAPES.items():
        for F, ld in shapes:
            for reduce in ("mean", "sum", "max"):
                v = gather_variant(dtype, F, ld, reduce, force_ldg=_ldg_force(dtype, F, ld))
                out.append(pytest.param(dtype, F, ld, reduce, id=f"F{F}-ld{ld}-{reduce}-{variant_id(v)}"))
    return out


TMA_CASES = _tma_cases()
LDG_CASES = _ldg_cases()


def test_sweep_reaches_every_variant():
    """The forward sweep launches every reachable `sage_tma_kernel` instantiation (dtype x OP x NV x PK, plain and
    sharded; PK is off for max), both TMA store forms, every VEC of the vector-load kernel for sum and for max,
    every (GROUP, CHUNKS) bucket, and max over two or more column tiles.  No device needed."""
    tma, stores, ldg, buckets, tiled_max = set(), set(), set(), set(), set()
    for p in TMA_CASES:
        dtype, F, reduce, pk, sharded, layout = p.values
        v = gather_variant(dtype, F, F, reduce, ldo=_tma_ldo(dtype, F, layout), packed_add=pk, sharded=sharded)
        assert v[0] == "tma", p.id
        tma.add(v[1:6])
        stores.add((v[1], v[6]))
    for p in LDG_CASES:
        dtype, F, ld, reduce = p.values
        v = gather_variant(dtype, F, ld, reduce, force_ldg=_ldg_force(dtype, F, ld))
        assert v[0] == "ldg", p.id
        ldg.add(v[1:4])
        buckets.update((v[1],) + t for t in v[4])
        if v[2] == "MAX" and len(v[4]) >= 2:
            tiled_max.add(v[1])
    want_tma = {(dt, op, nv, pk, sh) for dt in ("f32", "bf16") for op, pk in (("SUM", 0), ("SUM", 1), ("MAX", 0))
                for nv in (1, 2, 3, 4) for sh in (False, True)}
    assert want_tma <= tma, sorted(want_tma - tma)
    assert {(dt, s) for dt in ("f32", "bf16") for s in ("vec16", "scalar")} <= stores
    want_ldg = {(dt, op, vec) for dt, vecs in (("f32", (1, 2, 4)), ("bf16", (1, 2, 4, 8)))
                for op in ("SUM", "MAX") for vec in vecs}
    assert want_ldg <= ldg, sorted(want_ldg - ldg)
    all_gc = {(4, 1), (8, 1), (16, 1), (32, 1), (32, 2), (32, 3), (32, 4), (32, 5), (32, 6), (32, 8)}
    for dt in ("f32", "bf16"):
        assert {(dt,) + gc for gc in all_gc} <= buckets, (dt, sorted(all_gc - {b[1:] for b in buckets if b[0] == dt}))
    assert tiled_max == {"f32", "bf16"}
    # the helper agrees with the dispatch at the shapes the rest of the suite leans on
    assert gather_variant(torch.float32, 602, 604, "mean", ldo=604)[:4] == ("tma", "f32", "SUM", 1)
    assert gather_variant(torch.float32, 70, 70, "max")[:4] == ("ldg", "f32", "MAX", 2)


# ------------------------------------------------------------------------------ reference and bounds
@contextlib.contextmanager
def knob(key, value):
    old = _lib.get_tuning(key)
    _lib.set_tuning(key, value)
    try:
        yield
    finally:
        _lib.set_tuning(key, old)


def reduce_f64(table64, ids, n_src, fanout, reduce):
    """(ref, bound_terms, argmax) of one fixed-fanout block over the stored values `table64` [N, F] (float64);
    ids None = identity block.  bound_terms = scale * sum_k |x_k| (None for max)."""
    N, F = table64.shape
    ids = np.arange(n_src * fanout) if ids is None else np.asarray(ids, dtype=np.int64)
    valid = ((ids >= 0) & (ids < N)).reshape(n_src, fanout, 1)
    rows = table64[np.where(valid.ravel(), ids, 0)].reshape(n_src, fanout, F)
    if reduce == "max":
        x = np.where(valid, rows, -np.inf)
        return x.max(1), None, x.argmax(1)  # argmax: the first k attaining the max
    x = np.where(valid, rows, 0.0)
    scale = 1.0 / fanout if reduce == "mean" else 1.0
    return x.sum(1) * scale, np.abs(x).sum(1) * scale, None


def assert_within(got, ref, terms, K, dtype, what=""):
    """|got - ref| <= (K + 2) * 2^-24 * terms (+ the bf16 output rounding) for every element."""
    got = got.double().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, np.float64)
    tol = (K + 2) * U32 * terms
    if dtype == torch.bfloat16:
        tol = tol * (1 + 2.0 ** -8) + 2.0 ** -8 * np.abs(ref)
    err = np.abs(got - ref)
    bad = ~(err <= tol)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} elements outside the bound; first at "
                           f"{np.argwhere(bad)[0].tolist()}: got {got[bad][0]!r}, ref {ref[bad][0]!r}, "
                           f"tol {tol[bad][0]:.3e}")


def assert_max_exact(got, ref, argmax, ref_arg, what=""):
    got = got.double().cpu().numpy()
    assert np.array_equal(got, ref), f"{what}: max differs at {np.argwhere(got != ref)[0].tolist()}"
    if argmax is not None:
        arg = argmax.cpu().numpy()
        has = np.isfinite(ref)  # a source with a valid id; ties resolved to the first k
        assert np.array_equal(arg[has], ref_arg[has]), f"{what}: argmax differs"


def check_block(got, table64, ids, n_src, fanout, reduce, dtype, argmax=None, what=""):
    ref, terms, ref_arg = reduce_f64(table64, ids, n_src, fanout, reduce)
    if reduce == "max":
        assert_max_exact(got, ref, argmax, ref_arg, what)
    else:
        assert_within(got, ref, terms, fanout, dtype, what)


def sentinel_buffer(rows, cols, dtype):
    return torch.full((rows, cols), SENTINEL, dtype=dtype, device=DEV)


def assert_untouched(buf, keep, what=""):
    """Every element of `buf` outside the boolean [rows, cols] mask `keep` still holds the sentinel, bit for bit."""
    bits = {torch.float32: torch.int32, torch.bfloat16: torch.int16, torch.float16: torch.int16}[buf.dtype]
    want = torch.tensor(SENTINEL, dtype=buf.dtype).view(bits).item()
    outside = buf.view(bits)[~keep]
    bad = int((outside != want).sum())
    assert bad == 0, f"{what}: {bad} element(s) outside the output view were written"


def cols_mask(buf, *spans):
    keep = torch.zeros(buf.shape, dtype=torch.bool, device=buf.device)
    for c0, c1 in spans:
        keep[:, c0:c1] = True
    return keep


def make_table(rng, N, F, ld, dtype, ties=True):
    """[N, F] view of an [N, ld] buffer whose columns past F hold random values too (a column slice of a wider
    table); every third column is drawn from {-2..2} so that the max has ties.  Returns (view, stored float64)."""
    full = rng.standard_normal((N, ld))
    if ties:
        full[:, ::3] = rng.integers(-2, 3, size=full[:, ::3].shape)
    buf = torch.from_numpy(full).to(DEV, dtype)
    view = buf[:, :F]
    return view, view.double().cpu().numpy()


def make_ids(rng, N, n_src, fanout, bits):
    """Random ids with about one in eight invalid (-1, N, N + 7 and a large id past int32 for int64 blocks) and
    source 1 (of n_src >= 2) with no valid id at all."""
    ids = rng.integers(0, N, n_src * fanout)
    bad = [-1, N, N + 7] + ([2 ** 31 - 1] if bits == 32 else [2 ** 32 + 3, -(2 ** 40)])
    pos = rng.random(ids.size) < 0.125
    ids[pos] = rng.choice(bad, int(pos.sum()))
    ids[fanout:2 * fanout] = rng.choice(bad, fanout)
    return ids


def id_tensor(ids, bits):
    return None if ids is None else torch.from_numpy(ids).to(DEV, torch.int32 if bits == 32 else torch.int64)


# ------------------------------------------------------------------------------ forward sweep
_tma_inputs = {}


def _tma_setup(dtype, F):
    """Table, index blocks and shard split per (dtype, F), shared by the cases of that shape."""
    key = (dtype, F)
    if key not in _tma_inputs:
        rng = np.random.default_rng(F * 7 + ESZ[dtype])
        n_src = 48 if F * ESZ[dtype] <= 2800 else 16  # NV 3-4: a few wide rows
        N = n_src * max(FANOUTS) + 60
        table, t64 = make_table(rng, N, F, F, dtype)
        blocks = []
        for i, fanout in enumerate(FANOUTS):
            for kind in ("int32", "int64", "identity"):
                if kind == "identity":
                    blocks.append((kind, fanout, None, None))
                else:
                    bits = 32 if kind == "int32" else 64
                    ids = make_ids(rng, N, n_src, fanout, bits)
                    blocks.append((kind, fanout, ids, id_tensor(ids, bits)))
        cut = N // 3
        sharded = ShardedTable.local([table[:cut], table[cut:cut], table[cut:]])  # uneven, the middle one empty
        _tma_inputs.clear()
        _tma_inputs[key] = (n_src, table, t64, blocks, sharded)
    return _tma_inputs[key]


def _run_tma(table, sharded_table, ids_t, n_src, fanout, reduce, ldo, dtype, F, argmax_wanted):
    buf = sentinel_buffer(n_src, ldo, dtype)
    out = buf[:, :F]
    argmax = None
    if sharded_table is not None:
        Fn.gather_reduce_multi_raw(sharded_table, [(ids_t, n_src, fanout)], reduce, outs=[out])
    else:
        if argmax_wanted:
            argmax = torch.empty((n_src, ldo), dtype=torch.int32, device=DEV)[:, :F]
        Fn.gather_reduce_raw(table, ids_t, n_src, fanout, reduce, out=out, argmax=argmax)
    return buf, out, argmax


@gpu
@pytest.mark.parametrize("dtype,F,reduce,pk,sharded,layout", TMA_CASES)
def test_tma_ring_vs_f64(lib, dtype, F, reduce, pk, sharded, layout):
    """TMA ring, every (NV, OP, PK, SH) and both store forms: fanouts 1/7/32/33/40 (multi-chunk sources and
    balanced chunks), int32 / int64 / identity blocks, -1 and >= N ids and a source without a valid id (a ring
    stage with an empty mask).  Packed and unpacked adds give the same bits."""
    n_src, table, t64, blocks, st = _tma_setup(dtype, F)
    ldo = _tma_ldo(dtype, F, layout)
    for kind, fanout, ids, ids_t in blocks:
        what = f"{kind} fanout {fanout}"
        with knob("sage.packed_add", pk):
            buf, out, argmax = _run_tma(table, st if sharded else None, ids_t, n_src, fanout, reduce, ldo, dtype, F,
                                        reduce == "max")
        assert_untouched(buf, cols_mask(buf, (0, F)), what)
        check_block(out, t64, ids, n_src, fanout, reduce, dtype, argmax, what)
        if pk == 1:
            with knob("sage.packed_add", 0):
                _, out0, _ = _run_tma(table, st if sharded else None, ids_t, n_src, fanout, reduce, ldo, dtype, F,
                                      False)
            assert torch.equal(out.view(torch.int16 if ESZ[dtype] == 2 else torch.int32),
                               out0.view(torch.int16 if ESZ[dtype] == 2 else torch.int32)), what


@gpu
@pytest.mark.parametrize("dtype,F,ld,reduce", LDG_CASES)
def test_vector_load_vs_f64(lib, dtype, F, ld, reduce):
    """Vector-load kernel, every VEC and (GROUP, CHUNKS) bucket, column tiles (max offsets its argmax per tile),
    fanouts 1/7/33, int32 / int64 / identity blocks with invalid ids.  The output has the table's row stride and
    its columns past F must keep their sentinel."""
    rng = np.random.default_rng(F * 13 + ld)
    n_src = 24
    N = n_src * max(LDG_FANOUTS) + 40
    table, t64 = make_table(rng, N, F, ld, dtype)
    with knob("sage.force_ldg", _ldg_force(dtype, F, ld)):
        for fanout in LDG_FANOUTS:
            for kind in ("int32", "int64", "identity"):
                bits = 32 if kind == "int32" else 64
                ids = None if kind == "identity" else make_ids(rng, N, n_src, fanout, bits)
                buf = sentinel_buffer(n_src, ld, dtype)
                out = buf[:, :F]
                argmax = torch.empty((n_src, ld), dtype=torch.int32, device=DEV)[:, :F] if reduce == "max" else None
                Fn.gather_reduce_raw(table, id_tensor(ids, bits), n_src, fanout, reduce, out=out, argmax=argmax)
                what = f"{kind} fanout {fanout}"
                assert_untouched(buf, cols_mask(buf, (0, F)), what)
                check_block(out, t64, ids, n_src, fanout, reduce, dtype, argmax, what)


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("reduce", ["mean", "max"])
def test_four_block_launch_vs_f64(lib, dtype, reduce):
    """One launch of four blocks with different fanouts (one of them an identity block): every block against
    float64 directly, and against its single launch bit for bit."""
    rng = np.random.default_rng(5)
    F = 602
    N = 3000
    table, t64 = make_table(rng, N, F, _round_up(F, 16 // ESZ[dtype]), dtype)
    spec = [(1500, 10), (64, 25), (7, 1), (90, 33)]
    blocks, ids_np = [], []
    for i, (n_src, fanout) in enumerate(spec):
        ids = None if i == 3 else make_ids(rng, N, n_src, fanout, 32)
        ids_np.append(ids)
        blocks.append((id_tensor(ids, 32), n_src, fanout))
    outs = Fn.gather_reduce_multi_raw(table, blocks, reduce)
    for (ids_t, n_src, fanout), ids, o in zip(blocks, ids_np, outs):
        check_block(o, t64, ids, n_src, fanout, reduce, dtype, what=f"block fanout {fanout}")
        assert torch.equal(o, Fn.gather_reduce_raw(table, ids_t, n_src, fanout, reduce))


@gpu
@pytest.mark.parametrize("F", [605, 1402, 700])
@pytest.mark.parametrize("reduce", ["mean", "sum"])
def test_split_planes_vs_f64(lib, F, reduce):
    """fp16 hi / lo planes of the layer-0 gather: hi == fp16(out32) and lo == fp16(out32 - hi) bit for bit, where
    out32 is the fp32 gather of the same blocks in the same launch shape; hi + lo within the fp32 bound of float64
    (plus what 22 mantissa bits and an fp16 subnormal lo can carry); the columns past F and between the planes
    untouched."""
    rng = np.random.default_rng(F)
    N = 2000
    table, t64 = make_table(rng, N, F, _round_up(F, 4) + 4, torch.float32)
    spec = [(400, 10), (64, 1), (33, 33)]
    ids_np = [make_ids(rng, N, n, k, 32) for n, k in spec]
    blocks = [(id_tensor(ids, 32), n, k) for ids, (n, k) in zip(ids_np, spec)]
    ldh = _round_up(F, 4) + 4
    Hs = [torch.full((n, 2 * ldh + 8), SENTINEL, dtype=torch.float16, device=DEV) for n, _ in spec]
    Fn.gather_reduce_multi_split_raw(table, blocks, reduce, [H[:, :F] for H in Hs], ldh)
    out32 = Fn.gather_reduce_multi_raw(table, blocks, reduce)
    for H, o32, ids, (n, k) in zip(Hs, out32, ids_np, spec):
        what = f"fanout {k}"
        hi, lo = H[:, :F], H[:, ldh:ldh + F]
        assert torch.equal(hi.view(torch.int16), o32.half().view(torch.int16)), what
        assert torch.equal(lo.view(torch.int16), (o32 - hi.float()).half().view(torch.int16)), what
        assert_untouched(H, cols_mask(H, (0, F), (ldh, ldh + F)), what)
        ref, terms, _ = reduce_f64(t64, ids, n, k, reduce)
        got = (hi.double() + lo.double()).cpu().numpy()
        e32 = (k + 2) * U32 * terms
        tol = e32 + 2.0 ** -22 * (np.abs(ref) + e32) + 2.0 ** -25
        assert (np.abs(got - ref) <= tol).all(), what


# ------------------------------------------------------------------------------ backward
@gpu
@pytest.mark.parametrize("F", [7, 130, 602, 2000])
@pytest.mark.parametrize("reduce", ["mean", "sum"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_gather_backward_vs_f64(lib, F, reduce, dtype):
    """Table gradient of `gather_reduce` (the ordered transpose walk of gnn_gather_reduce_bwd_f32) against a float64
    index_add: one table row referenced 5000 times, -1 and >= N ids (no gradient, nothing corrupted)."""
    rng = np.random.default_rng(F + (7 if dtype == torch.bfloat16 else 0))
    N, n_src, fanout = 900, 1000, 7
    ids = make_ids(rng, N, n_src, fanout, 64)
    hub = rng.choice(n_src * fanout, 5000, replace=False)
    ids[hub] = 3
    table = torch.from_numpy(rng.standard_normal((N, F))).to(DEV, dtype).requires_grad_(True)
    g = torch.from_numpy(rng.standard_normal((n_src, F))).to(DEV, dtype)
    Fn.gather_reduce(table, id_tensor(ids, 64), n_src, fanout, reduce).backward(g)
    grad = table.grad
    assert grad.dtype == dtype
    scale = 1.0 / fanout if reduce == "mean" else 1.0
    valid = (ids >= 0) & (ids < N)
    src = torch.from_numpy(np.repeat(np.arange(n_src), fanout)[valid])
    dst = torch.from_numpy(ids[valid])
    g64 = g.double().cpu()
    ref = torch.zeros(N, F, dtype=torch.float64).index_add_(0, dst, g64[src] * scale).numpy()
    terms = torch.zeros(N, F, dtype=torch.float64).index_add_(0, dst, g64[src].abs() * scale).numpy()
    hits = np.bincount(ids[valid], minlength=N).reshape(N, 1)
    assert hits[3, 0] >= 5000
    assert_within(grad, ref, terms, hits, dtype, "d_table")


@gpu
@pytest.mark.parametrize("dtype,F,ld_force", [(torch.float32, 128, 0), (torch.bfloat16, 256, 0),
                                               (torch.float32, 301, 0), (torch.float32, 1100, 1),
                                               (torch.bfloat16, 2100, 1)])
def test_max_backward_identity_block_exact(lib, dtype, F, ld_force):
    """Max over a pre-gathered [n_src * fanout, F] input (identity block): the gradient is exactly g at the first
    argmax of every column and 0 elsewhere.  fp32 F 128 / bf16 F 256 run the TMA ring; F 301 (VEC 1), fp32 1100 and
    bf16 2100 (vector loads forced) run two or more column tiles."""
    rng = np.random.default_rng(F)
    n_src, fanout = 40, 9
    v = gather_variant(dtype, F, F, "max", force_ldg=ld_force)
    assert (v[0] == "tma") == (F in (128, 256)) and (v[0] == "tma" or len(v[4]) >= 2), v
    x64 = rng.standard_normal((n_src * fanout, F))
    x64[:, ::3] = rng.integers(-2, 3, size=x64[:, ::3].shape)  # ties
    x = torch.from_numpy(x64).to(DEV, dtype).requires_grad_(True)
    g = torch.from_numpy(rng.standard_normal((n_src, F))).to(DEV, dtype)
    with knob("sage.force_ldg", ld_force):
        out = Fn.gather_reduce(x, None, n_src, fanout, "max")
        out.backward(g)
    xs = x.detach().double().cpu().numpy().reshape(n_src, fanout, F)
    assert np.array_equal(out.detach().double().cpu().numpy(), xs.max(1))
    want = np.zeros((n_src, fanout, F))
    arg = xs.argmax(1)
    np.put_along_axis(want, arg[:, None, :], g.double().cpu().numpy()[:, None, :], axis=1)
    assert np.array_equal(x.grad.double().cpu().numpy().reshape(n_src, fanout, F), want)


@gpu
@pytest.mark.parametrize("U", [10, 64, 201])
@pytest.mark.parametrize("reduce", ["sum", "mean"])
def test_typed_gather_vs_f64(lib, U, reduce):
    """GATNE's typed gather [N, T, U] x [B, T, K] forward and backward against float64, with -1 and >= N ids."""
    rng = np.random.default_rng(U)
    N, T, B, K = 300, 3, 50, 7
    table64 = rng.standard_normal((N, T, U)).astype(np.float32).astype(np.float64)
    ids = rng.integers(0, N, (B, T, K))
    pos = rng.random(ids.shape) < 0.1
    ids[pos] = rng.choice([-1, N, N + 5], int(pos.sum()))
    t = torch.from_numpy(table64).to(DEV, torch.float32).requires_grad_(True)
    out = Fn.typed_gather_reduce(t, torch.from_numpy(ids).to(DEV), reduce)
    valid = (ids >= 0) & (ids < N)
    safe = np.where(valid, ids, 0)
    rows = table64[safe, np.arange(T)[None, :, None], :] * valid[..., None]  # [B, T, K, U]
    scale = 1.0 / K if reduce == "mean" else 1.0
    assert_within(out.detach(), rows.sum(2) * scale, np.abs(rows).sum(2) * scale, K, torch.float32, "forward")
    g = rng.standard_normal((B, T, U))
    out.backward(torch.from_numpy(g).to(DEV, torch.float32))
    g64 = g.astype(np.float32).astype(np.float64)
    ref = np.zeros((N, T, U))
    terms = np.zeros((N, T, U))
    hits = np.zeros((N, T, 1))
    b, tt, _ = np.nonzero(valid)
    nid = ids[valid]
    np.add.at(ref, (nid, tt), g64[b, tt] * scale)
    np.add.at(terms, (nid, tt), np.abs(g64[b, tt]) * scale)
    np.add.at(hits, (nid, tt), 1)
    assert_within(t.grad, ref, terms, hits, torch.float32, "backward")


# ------------------------------------------------------------------------------ tail-store contract
TAIL_SHAPES = [(torch.float32, 7), (torch.float32, 602), (torch.bfloat16, 605)]


@gpu
@pytest.mark.parametrize("dtype,F", TAIL_SHAPES)
@pytest.mark.parametrize("entry", ["tma", "vector_load", "multi", "sharded"])
@pytest.mark.parametrize("reduce", ["sum", "max"])
def test_gather_writes_only_its_columns(lib, dtype, F, entry, reduce):
    """An output view [rows, F] into a sentinel-filled [rows, F + pad] buffer: every element outside the view
    keeps the sentinel, whatever the table holds past its F columns.  `multi` also hands two blocks adjacent
    column slices of one buffer."""
    E = 16 // ESZ[dtype]
    if entry in ("tma", "sharded") and F * ESZ[dtype] < 256:
        pytest.skip("rows under 256 bytes never take the TMA path")
    rng = np.random.default_rng(F + len(entry))
    N, n_src, fanout = 500, 96, 9
    ld = _round_up(F, E) + E
    table, t64 = make_table(rng, N, F, ld, dtype)
    ids = make_ids(rng, N, n_src, fanout, 32)
    ids_t = id_tensor(ids, 32)
    ldo = _round_up(F, E) + E
    force = int(entry == "vector_load")
    if entry in ("tma", "vector_load"):
        want = gather_variant(dtype, F, ld, reduce, ldo=ldo, force_ldg=force)
        assert want[0] == ("tma" if entry == "tma" else "ldg"), want
    with knob("sage.force_ldg", force):
        if entry in ("tma", "vector_load"):
            buf = sentinel_buffer(n_src, ldo, dtype)
            Fn.gather_reduce_raw(table, ids_t, n_src, fanout, reduce, out=buf[:, :F])
            assert_untouched(buf, cols_mask(buf, (0, F)), entry)
            check_block(buf[:, :F], t64, ids, n_src, fanout, reduce, dtype, what=entry)
        elif entry == "multi":
            ids2 = make_ids(rng, N, n_src, 4, 32)
            Z = sentinel_buffer(n_src, 2 * F + E, dtype)
            W = sentinel_buffer(n_src, ldo, dtype)
            Fn.gather_reduce_multi_raw(table, [(ids_t, n_src, fanout), (id_tensor(ids2, 32), n_src, 4),
                                               (ids_t, n_src, fanout)], reduce,
                                       outs=[Z[:, :F], Z[:, F:2 * F], W[:, :F]])
            assert_untouched(Z, cols_mask(Z, (0, 2 * F)), "adjacent slices")
            assert_untouched(W, cols_mask(W, (0, F)), "padded output")
            check_block(Z[:, :F], t64, ids, n_src, fanout, reduce, dtype, what="slice 0")
            check_block(Z[:, F:2 * F], t64, ids2, n_src, 4, reduce, dtype, what="slice 1")
            check_block(W[:, :F], t64, ids, n_src, fanout, reduce, dtype, what="padded output")
        else:
            st = ShardedTable.local([table[:200], table[200:200], table[200:]])
            buf = sentinel_buffer(n_src, ldo, dtype)
            Fn.gather_reduce_multi_raw(st, [(ids_t, n_src, fanout)], reduce, outs=[buf[:, :F]])
            assert_untouched(buf, cols_mask(buf, (0, F)), entry)
            check_block(buf[:, :F], t64, ids, n_src, fanout, reduce, dtype, what=entry)


def _spmm_graph(rng, n, long_deg):
    deg = rng.poisson(9, size=n)
    deg[::7] = 0
    deg[5] = long_deg  # past spmm.long_row: the chunked long-row kernels on the planned path
    rowptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64)
    col = rng.integers(0, n, size=rowptr[-1]).astype(np.int32)
    val = rng.standard_normal(rowptr[-1]).astype(np.float32)
    return rowptr, col, val


@gpu
@pytest.mark.parametrize("dtype,F", TAIL_SHAPES)
@pytest.mark.parametrize("form", ["planned", "unplanned", "accumulate", "bias_relu", "ex", "ex_accumulate",
                                  "ex_bias_relu"])
def test_spmm_writes_only_its_columns(lib, dtype, F, form):
    """Y = A.X (planned with a chunked long row, unplanned, accumulating, with the bias/ReLU epilogue, and the
    row-subset entry spmm_ex) into an output view [n, F] of a sentinel-filled [n, F + pad] buffer: within the
    float64 bound, and no element past F read or written.  X's columns past F hold random values."""
    E = 16 // ESZ[dtype]
    rng = np.random.default_rng(F * 3 + len(form))
    n = 1200
    rowptr, col, val = _spmm_graph(rng, n, 9000)
    g = CSRGraph(torch.from_numpy(rowptr).to(DEV), torch.from_numpy(col).to(DEV), torch.from_numpy(val).to(DEV), n, n)
    ld = _round_up(F, E) + E
    X, X64 = make_table(rng, n, F, ld, dtype, ties=False)
    buf = sentinel_buffer(n, ld, dtype)
    out = buf[:, :F]
    accumulate = form.endswith("accumulate")
    epi = form.endswith("bias_relu")
    Y0 = np.zeros((n, F))
    if accumulate:
        out.copy_(torch.from_numpy(rng.standard_normal((n, F))).to(DEV, dtype))
        Y0 = out.double().cpu().numpy()
    b = rng.standard_normal(F).astype(np.float32) if epi else None
    bias = torch.from_numpy(b).to(DEV) if epi else None
    if form.startswith("ex"):
        Fn.spmm_ex(g, X, out, accumulate=accumulate, bias=bias, relu=epi)
    else:
        Fn.spmm_raw(g, X, out=out, planned=form != "unplanned", accumulate=accumulate, bias=bias, relu=epi)
    assert_untouched(buf, cols_mask(buf, (0, F)), form)
    A = sp.csr_matrix((val.astype(np.float64), col, rowptr), shape=(n, n))
    ref = A @ X64 + Y0
    terms = abs(A) @ np.abs(X64) + np.abs(Y0)
    deg = np.diff(rowptr).reshape(n, 1) + 2
    if epi:
        ref = np.maximum(ref + b, 0.0)
        terms = terms + np.abs(b)
    assert_within(out, ref, terms, deg, dtype, form)


@gpu
@pytest.mark.parametrize("reduce,force_ldg", [("max", 0), ("max", 1), ("mean", 0)])
def test_graphsage_inference_ignores_table_columns_past_f(lib, reduce, force_ldg):
    """GraphSage inference (the one-launch layer 0: [self | pooled] . [W_self ; W_agg] with zero weight rows under
    the pad columns) on an fp32 table whose columns between F and its row stride hold NaN: finite, and equal to
    the same model on pad_table(table)."""
    rng = np.random.default_rng(0)
    n, F_in, B, fan = 3000, 602, 48, [7, 4]
    buf = torch.full((n, 608), float("nan"), device=DEV)
    table = buf[:, :F_in]
    table.copy_(torch.from_numpy(rng.standard_normal((n, F_in)).astype(np.float32)))
    torch.manual_seed(1)
    model = layers.GraphSage(F_in, [128, 41], fan).to(DEV).eval()
    for layer in model.gcn:
        layer.aggr_neighbor_method = layer.aggregator.aggr_method = reduce
    model.tensor_core_gemm = False  # the fp32 product over the fused operand (max always takes it)
    blocks = [torch.from_numpy(rng.integers(0, n, s)).to(DEV, torch.int32) for s in (B, B * 7, B * 28)]
    with torch.no_grad(), knob("sage.force_ldg", force_ldg):
        got = model.forward_sampled(table, blocks)
        want = model.forward_sampled(Fn.pad_table(table), blocks)
    assert bool(torch.isfinite(got).all())
    assert torch.equal(got, want)
