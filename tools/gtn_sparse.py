#!/usr/bin/env python
"""GTN on a sparse RelationStack against the dense drop-in (one GPU).  One JSON line per configuration on stdout.

    python tools/gtn_sparse.py --check
    python tools/gtn_sparse.py --time [--out profiles/gtn_sparse_time_1gpu.jsonl]

--check: a small DBLP-shaped heterograph (the generator below at 1/20 scale).  For 1, 2 and 3 layers, the logits
  (1e-5 relative) and every parameter gradient (5e-5: both sides are fp32, and the dense bmm chain's own rounding
  dominates) of `GTN_Model.forward(RelationStack, ...)` against the dense drop-in on the same GPU, and the logits
  against oracle/gtn_sparse.py in float64 (1e-5 relative).
--time: a DBLP-shaped synthetic heterograph.  The published DBLP figures (not part of the reference): 4,057 authors,
  14,328 papers, 20 venues, 67,946 edges over the relations PA, AP, PC, CP, plus the identity; 334 features.  Here:
  one venue per paper, drawn with a Zipf-like skew over the venues; 19,645 paper-author edges (67,946 / 2 - 14,328),
  every paper with at least one author and authors drawn with a skew (a few prolific authors).  For 2 and 3 layers
  at C = 2: nnz and nnz/N^2 of every P_l, the pattern build time (once per stack), the sparse forward+backward step,
  and the dense drop-in step on the same GPU in the same run, the two alternated.  Then one scale at which the dense
  [C, N, N] does not fit (10x DBLP, 1 and 2 layers), sparse only.  Device name and power limit are read in the same run."""
import argparse
import gc
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

from graphneuralnetwork_b200 import _lib, layers  # noqa: E402
from graphneuralnetwork_b200.graph import CSRGraph  # noqa: E402
from graphneuralnetwork_b200.layers.gtn import RelationStack  # noqa: E402
from gcn_dist_train import device_info  # noqa: E402

DBLP = {"authors": 4057, "papers": 14328, "venues": 20, "pa_edges": 19645, "feats": 334, "classes": 4}


def dblp_like(dev, scale=1.0, seed=0):
    """([PA, AP, PC, CP, I] as value-1 CSRGraphs [N, N], N): node ids authors, then papers, then venues."""
    rng = np.random.default_rng(seed)
    na, npap, nv = (int(round(DBLP[k] * scale)) for k in ("authors", "papers", "venues"))
    n_pa = int(round(DBLP["pa_edges"] * scale))
    n = na + npap + nv
    venue_w = 1.0 / np.arange(1, nv + 1) ** 1.1
    venue = rng.choice(nv, npap, p=venue_w / venue_w.sum())
    author_w = 1.0 / np.arange(1, na + 1) ** 0.8
    extra = rng.choice(npap, n_pa - npap)  # papers with more than one author
    pap = np.concatenate([np.arange(npap), extra])
    auth = rng.choice(na, len(pap), p=author_w / author_w.sum())
    key = np.unique(pap.astype(np.int64) * na + auth)  # one edge per (paper, author)
    pap, auth = key // na, key % na
    p_ids, a_ids, v_ids = pap + na, auth, venue + na + npap

    def rel(r, c):
        r, c = torch.from_numpy(np.asarray(r, np.int64)).to(dev), torch.from_numpy(np.asarray(c, np.int64)).to(dev)
        return CSRGraph.from_coo(r, c, torch.ones(r.numel(), device=dev), n, n)

    eye = np.arange(n)
    papers = np.arange(npap) + na
    return [rel(p_ids, a_ids), rel(a_ids, p_ids), rel(papers, v_ids), rel(v_ids, papers), rel(eye, eye)], n


def dense_of(rels, n, dev):
    A = torch.zeros((n, n, len(rels)), dtype=torch.float32, device=dev)
    for k, g in enumerate(rels):
        A[g.edge_rows().long(), g.col.long(), k] = g.val
    return A


def _model(K, C, L, w_in, seed, dev):
    torch.manual_seed(seed)
    m = layers.GTN_Model(K, C, w_in, 64, DBLP["classes"], L, True)
    for mod in m.modules():
        if isinstance(mod, layers.GTConv):
            torch.nn.init.normal_(mod.weight, std=0.5)
    return m.to(dev)


def _step(model, A, X, target, labels):
    model.zero_grad(set_to_none=True)
    y, _ = model(A, X, target)
    torch.nn.functional.cross_entropy(y, labels).backward()
    return y.detach()


def _inputs(n, w_in, dev, seed=1):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(n, w_in, generator=g).to(dev)
    target = torch.arange(0, n, 3, device=dev)
    labels = torch.randint(0, DBLP["classes"], (target.numel(),), generator=g).to(dev)
    return X, target, labels


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


def check(dev):
    from oracle import gtn_sparse as O
    out, ok = [], True
    rels, n = dblp_like(dev, scale=0.05, seed=3)
    A = dense_of(rels, n, dev)
    stack = RelationStack.from_relations(rels)
    X, target, labels = _inputs(n, 16, dev)
    for L in (1, 2, 3):
        dense, sparse = _model(5, 2, L, 16, L, dev), _model(5, 2, L, 16, L, dev)
        yd, ys = _step(dense, A, X, target, labels), _step(sparse, stack, X, target, labels)
        grads = {name: rel(ps.grad, pd.grad) for (name, pd), (_, ps) in zip(dense.named_parameters(),
                                                                              sparse.named_parameters())
                 if pd.grad is not None}
        params = {k: v.detach().cpu().numpy() for k, v in sparse.state_dict().items()}
        y64 = O.gtn_forward(A.cpu().numpy(), X.cpu().numpy(), target.cpu().numpy(), params, 2, L)
        r = {"mode": "check", "layers": L, "n": n, "logits_vs_dense": rel(ys, yd),
             "logits_vs_oracle_f64": rel(ys, torch.from_numpy(y64)), "worst_grad_vs_dense": max(grads.values())}
        r["pass"] = r["logits_vs_dense"] < 1e-5 and r["logits_vs_oracle_f64"] < 1e-5 and r["worst_grad_vs_dense"] < 5e-5
        ok &= r["pass"]
        out.append(r)
    return out, ok


def _time(fn, reps):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return ts


def time_run(dev, reps):
    info = device_info(dev)
    out = []
    rels, n = dblp_like(dev)
    X, target, labels = _inputs(n, DBLP["feats"], dev)
    A = dense_of(rels, n, dev)
    for L in (2, 3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        stack = RelationStack.from_relations(rels)
        stack.patterns(L)
        stack.gcn_pattern(L)
        torch.cuda.synchronize()
        build_ms = (time.perf_counter() - t0) * 1e3
        P = stack.patterns(L)[0]
        dense, sparse = _model(5, 2, L, DBLP["feats"], L, dev), _model(5, 2, L, DBLP["feats"], L, dev)
        yd, ys = _step(dense, A, X, target, labels), _step(sparse, stack, X, target, labels)  # warm-up
        sp_ms, de_ms = [], []
        for _ in range(reps):  # alternated
            sp_ms += _time(lambda: _step(sparse, stack, X, target, labels), 1)
            de_ms += _time(lambda: _step(dense, A, X, target, labels), 1)
        r = {"mode": "time", "shape": "dblp", "n": n, "K": 5, "C": 2, "layers": L, "feats": DBLP["feats"],
             "nnz_U": stack.U.nnz, "nnz_P": [p.nnz for p in P], "density_P": [p.nnz / n / n for p in P],
             "pattern_build_ms": build_ms, "sparse_step_ms_median": statistics.median(sp_ms),
             "dense_step_ms_median": statistics.median(de_ms), "sparse_step_ms": sp_ms, "dense_step_ms": de_ms,
             "logits_rel_vs_dense": rel(ys, yd), "reps": reps, **info}
        out.append(r)
        print(json.dumps(r), flush=True)
        del stack, dense, sparse, yd, ys, P
    del A, rels
    gc.collect()
    torch.cuda.empty_cache()
    # 10x DBLP: dense [C, N, N] fp32 would take 2*N^2*4 bytes
    rels, n = dblp_like(dev, scale=10.0, seed=1)
    X, target, labels = _inputs(n, DBLP["feats"], dev)
    for L in (1, 2):
        r = {"mode": "time", "shape": "dblp_x10", "n": n, "K": 5, "C": 2, "layers": L,
             "dense_CNN_bytes": 2 * n * n * 4, **info}
        try:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            stack = RelationStack.from_relations(rels, max_nnz=1_500_000_000)
            stack.patterns(L)
            stack.gcn_pattern(L)
            torch.cuda.synchronize()
            r["pattern_build_ms"] = (time.perf_counter() - t0) * 1e3
            P = stack.patterns(L)[0]
            r.update(nnz_U=stack.U.nnz, nnz_P=[p.nnz for p in P], density_P=[p.nnz / n / n for p in P])
            sparse = _model(5, 2, L, DBLP["feats"], L, dev)
            _step(sparse, stack, X, target, labels)
            ms = _time(lambda: _step(sparse, stack, X, target, labels), reps)
            r.update(sparse_step_ms_median=statistics.median(ms), sparse_step_ms=ms,
                     peak_mem_gb=torch.cuda.max_memory_allocated(dev) / 1e9)
            del stack, sparse, P
        except (_lib.GnnError, torch.OutOfMemoryError) as e:
            r["refused"] = f"{type(e).__name__}: {str(e)[:200]}"
        gc.collect()
        torch.cuda.empty_cache()
        out.append(r)
        print(json.dumps(r), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--time", action="store_true")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gtn_sparse: needs a CUDA device (the sparse path has no CPU fallback)")
    dev = torch.device("cuda:0")
    ok = True
    rows = []
    if args.check:
        res, ok = check(dev)
        for r in res:
            print(json.dumps(r), flush=True)
    if args.time:
        rows = time_run(dev, args.reps)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                for r in rows:
                    f.write(json.dumps(r) + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
