#!/usr/bin/env python
"""De-duplicating GraphSAGE minibatches built on the device (`functional.dedup_layer_nodes`) and consumed by
`GraphSAGE.forward_sampled`, against the reference's collate layout.  One JSON line on stdout (and appended to --out).

    python tools/sage_v2_batch.py --check
    python tools/sage_v2_batch.py --time [--out profiles/sage_v2_batch_time_1gpu.jsonl]

--check: on a 2,000-node skewed graph, for L = 1, 2, 3: the builder against `oracle.sage_dedup.layer_adj_nodes_v2`
  fed with the same device draws (node sets, maps and outer draws bit for bit); `forward_sampled` against `forward` on
  the same batch gathered on the host (logits and every weight gradient bit for bit, MEAN, MAX and gcn=True, F = 602);
  a repeat of the builder (same bits).
--time: the Reddit shape (232,965 nodes, mean degree 492, F = 602 fp32, B = 1024, L = 2, k = 10, hidden 128, 41
  classes).  Per batch: the builder's ms (host clock around the call and a device synchronise: it includes the one
  count read), `forward_sampled` forward + backward ms, and for comparison the reference's collate path from the same
  ids: the vectorised host feature gather (`X[S_0]`, `X[outer draws]` as [n0, k, F] on the CPU), its host-to-device
  copy, and `forward` forward + backward.  Also the host union/remap of the same draws in Python (the oracle), |S_1|,
  |S_0| and the bytes `neigh_feats` would have had.  Medians over --reps batches after --warmup.  The 561 MB table is
  larger than L2, and the gathers are not flushed between reps.  Device name and power limit are read in the run."""
import argparse
import copy
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

from graphneuralnetwork_b200 import functional as Fn, layers, synthetic as S  # noqa: E402
from gcn_dist_train import device_info  # noqa: E402
from oracle.sage_dedup import layer_adj_nodes_v2  # noqa: E402


def _adj_lists(g):
    rp, col = g.rowptr.cpu().numpy(), g.col.cpu().numpy()
    return {i: set(col[rp[i]:rp[i + 1]].tolist()) for i in range(g.n_rows)}


def _host_batch(table_cpu, b):
    """The reference collate's tensors from the batch's ids: X[S_0] and X[outer draws] gathered on the host."""
    ids = b.outer_neighbors.cpu()
    center = table_cpu.index_select(0, b.nodes[0].cpu())
    neigh = table_cpu.index_select(0, ids.reshape(-1)).view(*ids.shape, -1)
    return center, neigh


def run_check(dev):
    g = S.powerlaw_csr(2000, 12.0, seed=7, device=dev, with_values=False)
    adj = _adj_lists(g)
    k, seed = 5, 1234
    batch = np.random.default_rng(0).choice(2000, 64, replace=False).tolist()
    res = {}
    for L in (1, 2, 3):
        b = Fn.dedup_layer_nodes(g, batch, L, k, seed)
        draws_ok = []

        def draws(level, nodes):
            d = Fn.sample_neighbors(g, torch.tensor(nodes, dtype=torch.int64, device=dev), k,
                                    seed + 0x9E3779B9 * (L - level), torch.int64)
            draws_ok.append(torch.equal(d.view(-1, k), b.neighbors[level]))
            return d.cpu().numpy()

        nodes, cm, nm, outer = layer_adj_nodes_v2(adj, batch, L, k, draws)
        res[f"builder_L{L}"] = bool(all(draws_ok) and b.counts == [len(x) for x in nodes]
                                    and all(np.array_equal(x.cpu().numpy(), y) for x, y in zip(b.nodes, nodes))
                                    and np.array_equal(b.center_map.cpu().numpy(), cm)
                                    and np.array_equal(b.neigh_map.cpu().numpy(), nm)
                                    and np.array_equal(b.outer_neighbors.cpu().numpy(), outer))
        again = Fn.dedup_layer_nodes(g, batch, L, k, seed)
        res[f"repeat_L{L}"] = bool(again.counts == b.counts and all(
            torch.equal(x, y) for x, y in zip(again.nodes + again.neighbors + [again.center_map, again.neigh_map],
                                              b.nodes + b.neighbors + [b.center_map, b.neigh_map])))
    table_cpu = torch.from_numpy(np.random.default_rng(1).standard_normal((2000, 602), dtype=np.float32))
    table = Fn.pad_table(table_cpu.to(dev))
    labels = torch.from_numpy(np.random.default_rng(2).integers(0, 7, 64)).to(dev)
    # MAX trains at L = 1 only: `forward` has no max backward into a gathered layer output
    for agg, gcn, L, grads in (("MEAN", False, 2, True), ("MEAN", True, 2, True), ("MEAN", False, 3, True),
                               ("MAX", False, 1, True), ("MAX", False, 2, False), ("MAX", True, 2, False)):
        b = Fn.dedup_layer_nodes(g, batch, L, k, seed + 1)
        torch.manual_seed(0)
        m1 = layers.GraphSAGE(L, 602, 128, gcn=gcn, agg_func=agg, Unsupervised=False, class_size=7).to(dev)
        m2 = copy.deepcopy(m1)
        center, neigh = _host_batch(table_cpu, b)
        with torch.set_grad_enabled(grads):
            _, y1 = m1(center.to(dev), b.center_map, neigh.to(dev), b.neigh_map, None, None, None, None, None)
            _, y2 = m2.forward_sampled(table, b)
        ok = torch.equal(y1, y2)
        if grads:
            torch.nn.functional.cross_entropy(y1, labels).backward()
            torch.nn.functional.cross_entropy(y2, labels).backward()
            ok = ok and all(torch.equal(p.grad, q.grad) for p, q in zip(m1.parameters(), m2.parameters()))
        res[f"forward_sampled_{agg}{'_gcn' if gcn else ''}_L{L}{'_grads' if grads else ''}"] = bool(ok)
    return {"mode": "check", **res, "all_ok": all(res.values())}


def _ms(fn, dev):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize(dev)
    return (time.perf_counter() - t0) * 1e3, out


def run_time(a, dev):
    info = device_info(dev)
    n, F, B, L, k = S.REDDIT["n"], S.REDDIT["feats"], S.REDDIT["batch"], 2, 10
    g = S.powerlaw_csr(n, 492.0, seed=0, device=dev, with_values=False)  # the Reddit-shaped adjacency of bench.py
    table_cpu = torch.from_numpy(np.random.default_rng(0).standard_normal((n, F), dtype=np.float32))
    table = Fn.pad_table(table_cpu.to(dev))
    torch.manual_seed(0)
    m_dev = layers.GraphSAGE(L, F, 128, agg_func="MEAN", Unsupervised=False, class_size=41).to(dev)
    m_host = copy.deepcopy(m_dev)
    perm = np.random.default_rng(1).permutation(n)
    rows = {k_: [] for k_ in ("builder_ms", "forward_sampled_fwd_bwd_ms", "host_gather_ms", "h2d_ms",
                              "forward_fwd_bwd_ms", "host_union_remap_ms", "s1", "s0", "bitwise_equal_logits")}
    for it in range(a.warmup + a.reps):
        batch = perm[it * B:(it + 1) * B].tolist()
        labels = torch.from_numpy(np.random.default_rng(it).integers(0, 41, B)).to(dev)
        t_build, b = _ms(lambda: Fn.dedup_layer_nodes(g, batch, L, k, seed=it), dev)

        def step_dev():
            m_dev.zero_grad()
            _, y = m_dev.forward_sampled(table, b)
            torch.nn.functional.cross_entropy(y, labels).backward()
            return y.detach()
        t_dev, y_dev = _ms(step_dev, dev)
        t0 = time.perf_counter()
        center, neigh = _host_batch(table_cpu, b)
        t_gather = (time.perf_counter() - t0) * 1e3
        t_h2d, (center_d, neigh_d) = _ms(lambda: (center.to(dev), neigh.to(dev)), dev)

        def step_host():
            m_host.zero_grad()
            _, y = m_host(center_d, b.center_map, neigh_d, b.neigh_map, None, None, None, None, None)
            torch.nn.functional.cross_entropy(y, labels).backward()
            return y.detach()
        t_host, y_host = _ms(step_host, dev)
        drawn = {lvl: b.neighbors[lvl].cpu().numpy() for lvl in range(L)}
        t_union = _host_union_ms(batch, L, k, drawn)
        if it >= a.warmup:
            for key, v in (("builder_ms", t_build), ("forward_sampled_fwd_bwd_ms", t_dev), ("host_gather_ms", t_gather),
                           ("h2d_ms", t_h2d), ("forward_fwd_bwd_ms", t_host), ("host_union_remap_ms", t_union),
                           ("s1", b.counts[1]), ("s0", b.counts[0]), ("bitwise_equal_logits", torch.equal(y_dev, y_host))):
                rows[key].append(v)
        del center, neigh, center_d, neigh_d
    med = {key: round(statistics.median(v), 3) for key, v in rows.items()
           if key not in ("s1", "s0", "bitwise_equal_logits")}
    s0 = rows["s0"]
    host_total = med["host_gather_ms"] + med["h2d_ms"] + med["forward_fwd_bwd_ms"]
    dev_total = med["builder_ms"] + med["forward_sampled_fwd_bwd_ms"]
    return {"mode": "time", **info, "n": n, "F": F, "B": B, "L": L, "k": k, "hidden": 128, "classes": 41,
            "reps": a.reps, "warmup": a.warmup, **med,
            "device_path_ms": round(dev_total, 3), "host_collate_path_ms": round(host_total, 3),
            "host_path_excludes": "the host sampling and union (host_union_remap_ms, measured apart)",
            "s1_median": int(statistics.median(rows["s1"])), "s0_median": int(statistics.median(s0)),
            "s0_min": min(s0), "s0_max": max(s0),
            "neigh_feats_bytes_median": int(statistics.median(s0)) * k * F * 4,
            "bitwise_equal_logits": all(rows["bitwise_equal_logits"]), "host_cores": os.cpu_count()}


def _host_union_ms(batch, L, k, drawn):
    """The reference collate's union and remap in Python over the same draws (the oracle without its membership
    check): what the device builder replaces, apart from the sampling itself."""
    t0 = time.perf_counter()
    sets, samples = [list(batch)], []
    for lvl in range(L - 1, 0, -1):
        d = drawn[lvl]
        samples.insert(0, d)
        sets.insert(0, sorted(set(sets[0]) | set(d.reshape(-1).tolist())))
    n0 = len(sets[0])
    cm = np.full((L - 1, n0), -1, np.int64)
    nm = np.full((L - 1, n0, k), -1, np.int64)
    for i in range(L - 1):
        pos = {v: p for p, v in enumerate(sets[i])}
        cm[i, :len(sets[i + 1])] = [pos[v] for v in sets[i + 1]]
        nm[i, :len(sets[i + 1])] = np.vectorize(pos.__getitem__)(samples[i])
    return (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    mode = ap.add_mutually_exclusive_group(required=True)
    mode.add_argument("--check", action="store_true")
    mode.add_argument("--time", action="store_true")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="append the JSON line to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sage_v2_batch.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    line = run_check(dev) if a.check else run_time(a, dev)
    print(json.dumps(line), flush=True)
    if a.out:
        with open(a.out, "a") as f:
            f.write(json.dumps(line) + "\n")
    if a.check and not line["all_ok"]:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
