#!/usr/bin/env python
"""Build HAN's metapath graphs on the device from relation matrices (torchrun, one rank per GPU): `CSRGraph.metapath`
for whole graphs and `PartitionedMetapaths.from_relations`, where each rank composes only its own row block.  One JSON
line per rank on stdout.

    torchrun --nproc-per-node N tools/metapath_build.py --check
    torchrun --nproc-per-node N tools/metapath_build.py --time [--nodes 2000000]

--check: the ACM-shaped relations that `han_dist_train.acm_like_metapaths` composes with scipy (3,025 papers, 3 of
  6,050 authors each, one of 56 subjects).  Device composition must equal those graphs bit for bit;
  `from_relations` must equal `from_global` over the device-composed graphs (bounds, every metapath block, union halo
  ids, per-metapath halo rows, slot shifts); a repeat must give the same bits.
--time: two seeded relations generated on the device at the node count of `han_dist_train.py --time`.
  paper-author: 3 authors per paper, author id floor(A * v^2) for uniform v (popular low ids: rows of up to a few
  thousand products), plus HUB_AUTHORS authors of HUB_PAPERS papers each (rows past the CTA sort: the bitmap path).
  paper-term: 2 of T terms per paper, term id floor(T * v^1.5).  Per metapath (with self-loops, as HAN trains):
  nnz of R, the product count Σ u_i, the output nnz, the rows each kernel path took, count and fill ms (CUDA events
  after a warm-up, median of repeats), and scipy's time for the same composition on the host (a row sample,
  extrapolated to all rows; scipy's sparse product runs on one core).  Then `from_relations` ms on this rank and the
  union halo against Σ of the per-metapath halos.  Device name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from graphneuralnetwork_b200.graph import CSRGraph, _pattern_count, _pattern_fill  # noqa: E402
from graphneuralnetwork_b200.partition import PartitionedMetapaths  # noqa: E402
from gcn_dist_train import device_info  # noqa: E402
from han_dist_train import acm_like_metapaths  # noqa: E402

HUB_AUTHORS, HUB_PAPERS = 2, 12000
WIDTH = 2 * 8 * 8  # M * heads * hidden of han_dist_train's model: the width the union's operator is built for


def acm_like_relations(dev, n=3025, seed=0):
    """The paper-author [n, 2n] and paper-subject [n, 56] relations `han_dist_train.acm_like_metapaths` composes (the
    same random draws), as device CSRs."""
    rng = np.random.default_rng(seed)
    authors = rng.integers(0, 2 * n, size=(n, 3))
    subj = rng.integers(0, 56, n)
    rows = torch.arange(n, dtype=torch.int64, device=dev)
    pa = CSRGraph.from_coo(rows.repeat_interleave(3), torch.from_numpy(authors.ravel()).to(dev), None, n, 2 * n)
    ps = CSRGraph.from_coo(rows, torch.from_numpy(subj).to(dev), None, n, 56)
    return [CSRGraph(pa.rowptr, pa.col, None, n, 2 * n), CSRGraph(ps.rowptr, ps.col, None, n, 56)]


def same_partition(a, b) -> bool:
    """Bounds, every metapath block, union halo ids, per-metapath halo rows and slot shifts equal, bit for bit."""
    return (a.bounds == b.bounds and len(a) == len(b)
            and all(torch.equal(x, y) for m in range(len(a)) for x, y in zip(a[m], b[m]))
            and torch.equal(a.union.plan.halo_ids, b.union.plan.halo_ids)
            and a.halo_rows_per_graph == b.halo_rows_per_graph and a.slot_shift == b.slot_shift)


def run_check(rank, world, dev):
    rels = acm_like_relations(dev)
    want = acm_like_metapaths(dev)
    got = [CSRGraph.metapath(R, self_loops=True) for R in rels]
    composed = all(torch.equal(g.rowptr, w.rowptr) and torch.equal(g.col, w.col) for g, w in zip(got, want))
    again = [CSRGraph.metapath(R, self_loops=True) for R in rels]
    repeat = all(torch.equal(g.col, h.col) and torch.equal(g.rowptr, h.rowptr) for g, h in zip(got, again))
    pm_rel = PartitionedMetapaths.from_relations(rels, rank, world, widths=[WIDTH])
    pm_glob = PartitionedMetapaths.from_global(got, rank, world, widths=[WIDTH])
    pm_again = PartitionedMetapaths.from_relations(rels, rank, world, widths=[WIDTH])
    partitioned = same_partition(pm_rel, pm_glob)
    repeat = repeat and same_partition(pm_rel, pm_again)
    line = {"mode": "check", "world": world, "rank": rank, "n": rels[0].n_rows, "nnz_R": [R.nnz for R in rels],
            "nnz": [g.nnz for g in got], "bounds": pm_rel.bounds, "halo_rows_union": pm_rel.halo_rows,
            "halo_rows_per_metapath": pm_rel.halo_rows_per_graph, "composed_equal": composed,
            "from_relations_equal": partitioned, "bitwise_repeat": repeat, "pass": composed and partitioned and repeat}
    for pm in (pm_rel, pm_glob, pm_again):
        pm.close()
    print(json.dumps(line), flush=True)


def time_relations(n, dev, seed=0):
    """(name, shape, CSR) of the two seeded relations of --time (see the module docstring)."""
    gen = torch.Generator(device=dev).manual_seed(seed)
    n_auth, n_term = n, n // 5
    rows = torch.arange(n, dtype=torch.int64, device=dev)
    a_rows = rows.repeat_interleave(3)
    a_cols = (n_auth * torch.rand(3 * n, generator=gen, device=dev, dtype=torch.float64) ** 2).long()
    hub_rows = torch.randint(0, n, (HUB_AUTHORS * HUB_PAPERS,), generator=gen, device=dev)
    hub_cols = n_auth + torch.arange(HUB_AUTHORS, device=dev).repeat_interleave(HUB_PAPERS)
    pa = CSRGraph.from_coo(torch.cat([a_rows, hub_rows]), torch.cat([a_cols.clamp_max(n_auth - 1), hub_cols]), None,
                           n, n_auth + HUB_AUTHORS)
    t_cols = (n_term * torch.rand(2 * n, generator=gen, device=dev, dtype=torch.float64) ** 1.5).long()
    pt = CSRGraph.from_coo(rows.repeat_interleave(2), t_cols.clamp_max(n_term - 1), None, n, n_term)
    return [("paper-author", [n, n_auth + HUB_AUTHORS], CSRGraph(pa.rowptr, pa.col, None, n, n_auth + HUB_AUTHORS)),
            ("paper-term", [n, n_term], CSRGraph(pt.rowptr, pt.col, None, n, n_term))]


def events_ms(fn, reps):
    """Median ms of `reps` calls, each between two CUDA events, after one warm-up call."""
    fn()
    out = []
    for _ in range(reps):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        fn()
        t1.record()
        torch.cuda.synchronize()
        out.append(t0.elapsed_time(t1))
    return round(statistics.median(out), 3)


def scipy_ms(R, sample_rows):
    """Host ms of scipy's ((R·Rᵀ + I) > 0).sort_indices() over `sample_rows` rows, and the extrapolation to all."""
    import scipy.sparse as sp
    n, x = R.n_rows, R.n_cols
    S = sp.csr_matrix((np.ones(R.nnz, dtype=np.float32), R.col.cpu().numpy(), R.rowptr.cpu().numpy()), shape=(n, x))
    St = S.T.tocsr()
    rows = np.random.default_rng(0).choice(n, size=min(sample_rows, n), replace=False)
    rows.sort()
    t0 = time.perf_counter()
    C = S[rows] @ St
    C = C + sp.csr_matrix((np.ones(len(rows), dtype=np.float32), (np.arange(len(rows)), rows)), shape=C.shape)
    C = sp.csr_matrix(C > 0)
    C.sort_indices()
    ms = (time.perf_counter() - t0) * 1e3
    return round(ms, 1), round(ms * n / len(rows), 1)


def run_time(a, rank, world, dev):
    info = device_info(dev)
    rels = time_relations(a.nodes, dev)
    lines = []
    for name, shape, R in rels:
        Rt = R.transpose()
        n = R.n_rows
        deg_x = torch.bincount(R.col.long(), minlength=R.n_cols)
        products = int((deg_x * deg_x).sum().item()) + n  # Σ u_i with the self-loop
        path_rows = torch.zeros(3, dtype=torch.int64, device=dev)
        rp = _pattern_count(R, Rt, 0, n, True, path_rows)
        nnz = int(rp[-1].item())
        count_ms = events_ms(lambda: _pattern_count(R, Rt, 0, n, True), a.reps)
        fill_ms = events_ms(lambda: _pattern_fill(R, Rt, 0, n, True, rp, nnz), a.reps)
        got = _pattern_fill(R, Rt, 0, n, True, rp, nnz)
        repeat = torch.equal(got, _pattern_fill(R, Rt, 0, n, True, rp, nnz))
        del got
        sample_ms, scipy_all_ms = scipy_ms(R, a.scipy_rows) if rank == 0 else (None, None)
        lines.append({"metapath": f"{name}-{name.split('-')[0]}", "relation_shape": shape, "nnz_R": R.nnz,
                      "products": products, "nnz": nnz, "path_rows": dict(zip(("warp_sort", "cta_sort", "bitmap"),
                                                                             path_rows.tolist())),
                      "count_ms": count_ms, "fill_ms": fill_ms, "bitwise_repeat": repeat,
                      "scipy_sample_rows": min(a.scipy_rows, n) if rank == 0 else None,
                      "scipy_sample_ms": sample_ms, "scipy_ms_extrapolated": scipy_all_ms})
        torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pm = PartitionedMetapaths.from_relations([R for _, _, R in rels], rank, world, widths=[WIDTH])
    torch.cuda.synchronize()
    build_ms = round((time.perf_counter() - t0) * 1e3, 1)
    line = {"mode": "time", "world": world, "rank": rank, **info, "n": a.nodes, "host_cores": os.cpu_count(),
            "hub_authors": HUB_AUTHORS, "hub_papers": HUB_PAPERS, "metapaths": lines, "bounds": pm.bounds,
            "rows_local": pm.n_local, "from_relations_ms": build_ms, "halo_rows_union": pm.halo_rows,
            "halo_rows_sum_per_metapath": sum(pm.halo_rows_per_graph), "halo_rows_per_metapath": pm.halo_rows_per_graph,
            "peak_mem_gb": round(torch.cuda.max_memory_allocated(dev) / 1e9, 2)}
    pm.close()
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    mode = ap.add_mutually_exclusive_group(required=True)
    mode.add_argument("--check", action="store_true")
    mode.add_argument("--time", action="store_true")
    ap.add_argument("--nodes", type=int, default=2_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scipy-rows", type=int, default=50_000, help="--time: rows of the host scipy sample")
    a = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    try:
        run_check(rank, world, dev) if a.check else run_time(a, rank, world, dev)
    finally:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
