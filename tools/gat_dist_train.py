#!/usr/bin/env python
"""Full-graph GAT training across GPUs (torchrun, one rank per GPU): the drop-in `GAT` on a
`partition.PartitionedGraph`, replicated weights, the global loss rule and one gradient all-reduce per step.
One JSON line per rank and configuration on stdout.

    torchrun --nproc-per-node N tools/gat_dist_train.py --check [--dtype fp32|bf16] [--transports p2p ce nccl]
    torchrun --nproc-per-node N tools/gat_dist_train.py --time [--nodes 20000000] [--features 128 --heads 8 --hidden 8]

--check (small graphs every rank holds, with self-loops: a Cora-like graph and a 200 k-row power-law graph; 8 heads x 8,
  41 classes): every rank also trains the same seeded GAT on its GPU over the WHOLE graph and compares its own rows of
  the logits, every gradient at step 1 (after the all-reduce) and the weights after 3 Adam steps; the 3-step run is
  repeated and must be bit-identical.  Feature dropout is off (`model.dropout = 0`); the attention dropout of the
  heads stays 0.6.  Both runs draw identical attention-dropout streams: the host seed (torch.manual_seed) and the
  per-device counters of functional._drop_counters are reset before every run, and each rank's block draws the
  whole graph's mask for its edges (edge_slot_base).  --dtype bf16: the model, the features and the partition are
  bf16 and the 1-GPU model is the same seeded bf16 model, under gcn_dist_train.CHECK_BOUNDS["bf16"].
--time (large power-law graph plus self-loops, each rank generates only its own row block): ms per training step
  (forward + backward + gradient all-reduce + Adam) and per forward, ms of the two halo exchanges alone
  (`exchange_only`, widths H*F' and classes), and a float64 spot check of sampled first-layer output rows.  The fp32
  and the bf16 model are timed at the same size in one run, their steps alternated; one line per dtype with its halo
  bytes and the peak memory of its step.  Device name and power limit are read in the same run."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from graphneuralnetwork_b200 import functional as Fn  # noqa: E402
from graphneuralnetwork_b200 import synthetic as S  # noqa: E402
from graphneuralnetwork_b200.graph import CSRGraph  # noqa: E402
from graphneuralnetwork_b200.layers import GAT, SpGAT  # noqa: E402
from graphneuralnetwork_b200.layers.gat import _fused_heads  # noqa: E402
from graphneuralnetwork_b200.partition import (PartitionedGraph, allreduce_gradients, broadcast_parameters,  # noqa: E402
                                               global_count, partitioned_cross_entropy)
from gcn_dist_train import DTYPES, check_metrics, device_info, halo_bytes, peak_step_gb, timed_ms  # noqa: E402

MODELS = {"GAT": GAT, "SpGAT": SpGAT}


def with_self_loops(rowptr, col, row_offset):
    """Insert the self-loop (global id row_offset + i) as the first edge of every row i."""
    n = rowptr.numel() - 1
    dev = rowptr.device
    new_rowptr = rowptr + torch.arange(n + 1, dtype=torch.int64, device=dev)
    new_col = torch.empty(col.numel() + n, dtype=torch.int32, device=dev)
    is_loop = torch.zeros(new_col.numel(), dtype=torch.bool, device=dev)
    is_loop[new_rowptr[:-1]] = True
    new_col[is_loop] = (torch.arange(n, dtype=torch.int64, device=dev) + row_offset).to(torch.int32)
    new_col[~is_loop] = col
    return new_rowptr, new_col


def pattern_with_loops(n, edges, dev):
    """Pattern CSR of an undirected edge list plus self-loops (sorted columns)."""
    import scipy.sparse as sp
    e = np.asarray(edges)
    A = sp.coo_matrix((np.ones(len(e)), (e[:, 0], e[:, 1])), shape=(n, n))
    A = sp.csr_matrix(((A + A.T + sp.eye(n)) > 0).astype(np.float32))
    A.sort_indices()
    return CSRGraph(torch.from_numpy(A.indptr.astype(np.int64)).to(dev), torch.from_numpy(A.indices.astype(np.int32)).to(dev),
                    None, n, n)


def reset_streams(seed=0):
    """Identical dropout streams for every run: torch's generators and the attention-dropout counters."""
    torch.manual_seed(seed)
    Fn._drop_counters.clear()


def train(model, X, adj, target, idx, n_train, steps, group=None):
    """`steps` Adam steps; returns (logits of step 1, gradients of step 1, final weights).  n_train None: the
    1-GPU model over the whole graph; else the partitioned model (loss rule + gradient all-reduce)."""
    opt = torch.optim.Adam(model.parameters(), lr=0.005, weight_decay=5e-4)
    model.train()
    logits1 = grads1 = None
    for s in range(steps):
        opt.zero_grad(set_to_none=True)
        out = model(X, adj)
        if n_train is None:
            loss = torch.nn.functional.cross_entropy(out[idx], target[idx])
        else:
            loss = partitioned_cross_entropy(out[idx], target[idx], n_train)
        loss.backward()
        if n_train is not None and dist.is_initialized():
            allreduce_gradients(model, group)
        if s == 0:
            logits1 = out.detach().clone()
            grads1 = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
        opt.step()
    return logits1, grads1, {k: v.detach().clone() for k, v in model.state_dict().items()}


def make_model(cls, F_in, a):
    m = MODELS[cls](F_in, a.hidden, a.classes, 0.6, 0.2, a.heads)
    m.dropout = 0.0  # feature dropout off; the heads keep their attention dropout (0.6)
    return m


def run_check(a, rank, world, dev):
    graphs = [("cora_like", S.CORA["n"], lambda: pattern_with_loops(S.CORA["n"], S.cora_like_edges(seed=0), dev), 301)]
    n_pl = 200_000
    g_pl = S.powerlaw_csr(n_pl, 10.0, seed=3, device=dev)
    rp, cc = with_self_loops(g_pl.rowptr, g_pl.col, 0)
    graphs.append(("powerlaw_200k", n_pl, lambda: CSRGraph(rp, cc, None, n_pl, n_pl), 37))
    for name, n, make, F_in in graphs:
        g = make()
        gen = torch.Generator().manual_seed(11)
        dt = DTYPES[a.dtype]
        X = (torch.rand(n, F_in, generator=gen) * 2 - 1).to(dev).to(dt)
        labels = torch.randint(0, a.classes, (n,), generator=gen).to(dev)
        idx_train = torch.randperm(n, generator=gen)[: max(n * 2 // 5, 1)].sort().values.to(dev)
        for cls in a.models:
            torch.manual_seed(0)
            ref = make_model(cls, F_in, a).to(dev).to(dt)
            init = {k: v.clone() for k, v in ref.state_dict().items()}
            reset_streams()
            r_logits, r_grads, r_w = train(ref, X, g, labels, idx_train, None, 3)
            for transport in (a.transports if world > 1 else ["none"]):
                pg = PartitionedGraph.from_global(g, rank, world, widths=[a.heads * a.hidden, a.classes],
                                                  transport=transport if world > 1 else "p2p", dtype=dt)
                lo, hi = pg.row_range
                X_loc, y_loc = X[lo:hi].contiguous(), labels[lo:hi]
                idx_loc = pg.local_index(idx_train)
                n_train = global_count(idx_loc.numel(), dev) if world > 1 else idx_loc.numel()
                runs = []
                for _ in range(2):
                    model = make_model(cls, F_in, a).to(dev).to(dt)
                    if rank == 0:
                        model.load_state_dict(init)
                    if world > 1:
                        broadcast_parameters(model)
                    reset_streams()
                    runs.append(train(model, X_loc, pg, y_loc, idx_loc, n_train, 3))
                for op in pg.ops.values():
                    op.check_status()
                (logits, grads, w), (logits_b, grads_b, w_b) = runs
                line = {"mode": "check", "model": cls, "graph": name, "n": n, "nnz": g.nnz,
                        "widths": [F_in, a.heads * a.hidden, a.classes], "world": world, "rank": rank,
                        "transport": pg.ops[a.classes].transport, "edge_slot_base": pg.edge_slot_base,
                        "n_halo": pg.plan.n_halo}
                line.update(check_metrics(a.dtype, logits, r_logits[lo:hi], grads, r_grads, w, r_w,
                                          torch.equal(logits, logits_b)
                                          and all(torch.equal(grads[k], grads_b[k]) for k in grads)
                                          and all(torch.equal(w[k], w_b[k]) for k in w)))
                print(json.dumps(line), flush=True)
                pg.close()
                del pg, runs
            del ref
        del g


def layer1_reference(csr, rows, lo, W, a_src, a_dst, H, Fp, F_in):
    """float64 first-layer output (ELU of the attention-weighted Wh, all heads) of the local rows `rows`; the block's
    CSR holds global column ids, X = hashed_features of the global ids."""
    out = []
    W64, as64, ad64 = W.double(), a_src.double(), a_dst.double()
    for r in rows.tolist():
        cols = csr.col[csr.rowptr[r]:csr.rowptr[r + 1]].to(torch.int64)
        Whj = (S.hashed_features(cols, F_in).double() @ W64).view(-1, H, Fp)
        Whi = (S.hashed_features(torch.tensor([lo + r], device=cols.device), F_in).double() @ W64).view(H, Fp)
        z = (Whi * as64).sum(-1)[None, :] + (Whj * ad64[None]).sum(-1)
        att = torch.softmax(torch.nn.functional.leaky_relu(z, 0.2), dim=0)
        out.append(torch.nn.functional.elu((att[:, :, None] * Whj).sum(0).reshape(-1)))
    return torch.stack(out)


def run_time(a, rank, world, dev):
    from spmm_dist import build_rank_block
    F_in, H, Fp, C = a.features, a.heads, a.hidden, a.classes
    info = device_info(dev)
    csr0, bounds, nnz_total = build_rank_block(a.nodes, a.deg, rank, world, dev)
    lo, hi = bounds[rank], bounds[rank + 1]
    n_loc = hi - lo
    rp, cc = with_self_loops(csr0.rowptr, csr0.col, lo)
    del csr0
    csr = CSRGraph(rp, cc, None, n_loc, a.nodes)
    X32 = S.hashed_feature_block(lo, hi, F_in, dev)
    labels = (torch.arange(lo, hi, device=dev) * 2654435761 % C).to(torch.int64)
    idx_loc = torch.arange(0, n_loc, 3, device=dev)  # every third row trains
    n_train = global_count(idx_loc.numel(), dev) if world > 1 else idx_loc.numel()
    runs = {}
    for name in a.time_dtypes:
        dt = DTYPES[name]
        pg = PartitionedGraph(csr.rowptr, csr.col, None, bounds, rank, world, widths=[H * Fp, C], device=dev, waves=1,
                              transport=a.transport, dtype=dt)
        torch.manual_seed(0)
        model = GAT(F_in, Fp, C, 0.6, 0.2, H).to(dev).to(dt)
        model.dropout = 0.0
        if world > 1:
            broadcast_parameters(model)
        opt = torch.optim.Adam(model.parameters(), lr=0.005)
        X = X32.to(dt)

        def step(model=model, opt=opt, X=X, pg=pg):
            model.train()
            opt.zero_grad(set_to_none=True)
            out = model(X, pg)
            partitioned_cross_entropy(out[idx_loc].float(), labels[idx_loc], n_train).backward()
            if world > 1:
                allreduce_gradients(model)
            opt.step()

        def forward(model=model, X=X, pg=pg):
            model.train()
            with torch.no_grad():
                model(X, pg)

        Wh1, Wh2 = torch.randn(n_loc, H * Fp, device=dev).to(dt), torch.randn(n_loc, C, device=dev).to(dt)

        def exchange(pg=pg, Wh1=Wh1, Wh2=Wh2):
            pg.op(H * Fp).exchange_only(Wh1)
            pg.op(C).exchange_only(Wh2)

        runs[name] = {"pg": pg, "model": model, "X": X, "step": step, "forward": forward, "exchange": exchange,
                      "train_step_ms": [], "forward_ms": [], "exchange_only_ms": []}
    for r in runs.values():  # warm every shape before the first timed window
        r["step"]()
        r["forward"]()
    for _ in range(2):  # the dtypes alternate: fp32 steps, bf16 steps, fp32 steps, ...
        for r in runs.values():
            r["train_step_ms"].append(timed_ms(r["step"], a.steps, a.warmup, world, dev))
            r["forward_ms"].append(timed_ms(r["forward"], a.steps, a.warmup, world, dev))
            if world > 1:
                r["exchange_only_ms"].append(timed_ms(r["exchange"], a.steps, a.warmup, world, dev))
    rows = S.spmm_check_rows(csr, 256, 17 + rank)
    for name, r in runs.items():
        pg, model = r["pg"], r["model"]
        r["peak_step_gb"] = peak_step_gb(r["step"], dev)
        # float64 spot check of sampled first-layer rows (eval mode: no dropout)
        model.eval()
        heads = list(model.attentions)
        with torch.no_grad():
            halves = [h._halves() for h in heads]
            Y1 = _fused_heads(r["X"], pg, [h.W for h in heads], [x[0] for x in halves], [x[1] for x in halves], 0.2,
                              model._mode, 1, 0.0, False)
            W = torch.cat([h.W for h in heads], dim=1)
            ref = layer1_reference(csr, rows, lo, W, torch.stack([x[0] for x in halves]),
                                   torch.stack([x[1] for x in halves]), H, Fp, F_in)
            err = float((Y1[rows].double() - ref).abs().max().item()) / max(float(ref.abs().max().item()), 1e-30)
        for o in pg.ops.values():
            o.check_status()
        line = {"mode": "time", "dtype": name, "world": world, "rank": rank, **info, "n": a.nodes,
                "nnz": nnz_total + a.nodes, "rows_local": n_loc, "widths": [F_in, H * Fp, C], "heads": H,
                "transport": a.transport, "n_halo": pg.plan.n_halo, "edge_slot_base": pg.edge_slot_base,
                "halo_bytes_per_exchange": halo_bytes(pg),
                "peak_mem_gb": round(torch.cuda.max_memory_allocated(dev) / 1e9, 2), "peak_step_gb": r["peak_step_gb"],
                "train_step_ms": min(r["train_step_ms"]), "forward_ms": min(r["forward_ms"]),
                "exchange_only_ms": min(r["exchange_only_ms"]) if r["exchange_only_ms"] else None,
                "rounds_ms": {k: r[k] for k in ("train_step_ms", "forward_ms", "exchange_only_ms")},
                "layer1_sampled_rel_err": err, "layer1_ok": err <= (1e-5 if name == "fp32" else 1e-2)}
        print(json.dumps(line), flush=True)
    for r in runs.values():
        r["pg"].close()


def main():
    ap = argparse.ArgumentParser()
    mode = ap.add_mutually_exclusive_group(required=True)
    mode.add_argument("--check", action="store_true")
    mode.add_argument("--time", action="store_true")
    ap.add_argument("--transports", nargs="+", default=["p2p", "ce", "nccl"])
    ap.add_argument("--models", nargs="+", default=["GAT", "SpGAT"], choices=sorted(MODELS))
    ap.add_argument("--transport", default="p2p")
    ap.add_argument("--nodes", type=int, default=20_000_000)
    ap.add_argument("--deg", type=float, default=13.55)
    ap.add_argument("--features", type=int, default=128)
    ap.add_argument("--heads", type=int, default=8)
    ap.add_argument("--hidden", type=int, default=8)
    ap.add_argument("--classes", type=int, default=41)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--dtype", choices=sorted(DTYPES), default="fp32", help="--check: the features' and model's dtype")
    ap.add_argument("--time-dtypes", nargs="+", choices=sorted(DTYPES), default=["fp32", "bf16"],
                    help="--time: the dtypes whose steps alternate in one run")
    a = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    try:
        run_check(a, rank, world, dev) if a.check else run_time(a, rank, world, dev)
    finally:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
