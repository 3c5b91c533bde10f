#!/usr/bin/env python
"""Full-graph HAN training across GPUs (torchrun, one rank per GPU): the drop-in `HANModel` on a
`partition.PartitionedMetapaths`, replicated weights, the global loss rule and one gradient all-reduce per step.
One JSON line per rank and configuration on stdout.

    torchrun --nproc-per-node N tools/han_dist_train.py --check [--dtype fp32|bf16] [--transports p2p ce nccl]
    torchrun --nproc-per-node N tools/han_dist_train.py --time [--nodes 2000000 --degs 4 16 48]

--check (ACM-shaped synthetic metapaths every rank holds, with self-loops: 3,025 nodes, a sparse paper-author-paper
  graph and a dense paper-subject-paper graph; 8 heads x 8, 3 classes): every rank also trains the same seeded
  HANModel on its GPU over the WHOLE graphs (one block holding every row, which the GPU tests hold bit-identical to
  HANModel over the plain graphs) and compares its own rows of the logits, every gradient at step 1 (after the
  all-reduce) and the weights after 3 Adam steps; the 3-step run is repeated and must be bit-identical.  Dropout is
  off: a GATConv's one `dropout` sets its feature and its attention dropout, and a rank draws its feature masks over
  its own rows.  (The GPU tests hold a rank block's attention-dropout mask to the whole set's, and HANModel on a
  one-rank partition to one GPU with dropout 0.6.)  --dtype bf16: the model, the features and the partitions are
  bf16 and the 1-GPU run is the same seeded bf16 model over the whole graphs as one block, under
  gcn_dist_train.CHECK_BOUNDS["bf16"].
--time (a synthetic set of power-law metapaths of different mean degrees plus self-loops, generated on the device on
  every rank; dropout 0.6): ms per training step (forward + backward + gradient all-reduce + Adam) and per forward,
  ms of the stacked-Wh halo exchange alone, peak memory, the union halo rows against Σ of the per-metapath halo rows, and a
  float64 spot check of sampled first-layer rows of metapath 0.  The fp32 and the bf16 model are timed at the same
  size in one run, their steps alternated; one line per dtype with its halo bytes and the peak memory of its step.
  Device name and power limit are read in the same run."""
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
from graphneuralnetwork_b200.layers.han import HANModel  # noqa: E402
from graphneuralnetwork_b200.partition import (PartitionedMetapaths, allreduce_gradients,  # noqa: E402
                                               broadcast_parameters, global_count, partitioned_cross_entropy)
from gat_dist_train import reset_streams, with_self_loops  # noqa: E402
from gcn_dist_train import DTYPES, check_metrics, device_info, halo_bytes, peak_step_gb, timed_ms  # noqa: E402


def acm_like_metapaths(dev, n=3025, seed=0):
    """Two symmetric metapath patterns with self-loops over n nodes, ACM-shaped: P-A-P (each paper shares an author
    with a few others) and P-S-P (papers grouped by one of 56 subjects: dense blocks)."""
    import scipy.sparse as sp
    rng = np.random.default_rng(seed)
    authors = rng.integers(0, 2 * n, size=(n, 3))
    pa = sp.csr_matrix((np.ones(authors.size), (np.repeat(np.arange(n), 3), authors.ravel())), shape=(n, 2 * n))
    subj = sp.csr_matrix((np.ones(n), (np.arange(n), rng.integers(0, 56, n))), shape=(n, 56))
    out = []
    for B in (pa, subj):
        A = sp.csr_matrix(((B @ B.T + sp.eye(n)) > 0).astype(np.float32))
        A.sort_indices()
        out.append(CSRGraph(torch.from_numpy(A.indptr.astype(np.int64)).to(dev),
                            torch.from_numpy(A.indices.astype(np.int32)).to(dev), None, n, n))
    return out


def train(model, graphs, X, target, idx, n_train, steps, group=None):
    """`steps` Adam steps; returns (logits of step 1, gradients of step 1, final weights).  n_train None: the
    1-GPU model over the whole graphs; else the partitioned model (loss rule + gradient all-reduce)."""
    opt = torch.optim.Adam(model.parameters(), lr=0.005, weight_decay=1e-3)
    model.train()
    logits1 = grads1 = None
    for s in range(steps):
        opt.zero_grad(set_to_none=True)
        out = model(graphs, X)
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


def make_model(M, F_in, a, dropout):
    return HANModel(M, F_in, a.hidden, a.classes, [a.heads], dropout)


def run_check(a, rank, world, dev):
    graphs = acm_like_metapaths(dev)
    n, M, F_in = graphs[0].n_rows, len(graphs), 334
    width = M * a.heads * a.hidden
    gen = torch.Generator().manual_seed(11)
    dt = DTYPES[a.dtype]
    X = (torch.rand(n, F_in, generator=gen) * 2 - 1).to(dev).to(dt)
    labels = torch.randint(0, a.classes, (n,), generator=gen).to(dev)
    idx_train = torch.randperm(n, generator=gen)[: n // 5].sort().values.to(dev)
    torch.manual_seed(0)
    ref = make_model(M, F_in, a, 0.0).to(dev).to(dt)
    init = {k: v.clone() for k, v in ref.state_dict().items()}
    # the 1-GPU run: the whole graphs as one block (tests/test_gpu_partition_han.py holds this equal, bit for bit, to
    # HANModel over the plain graphs in fp32; tests/test_gpu_partition_bf16.py within bf16 tolerance in bf16, whose
    # semantic attention differs on a partition)
    whole = PartitionedMetapaths.from_global(graphs, 0, 1, widths=[width], dtype=dt)
    reset_streams()
    r_logits, r_grads, r_w = train(ref, whole, X, labels, idx_train, None, 3)
    whole.close()
    for transport in (a.transports if world > 1 else ["none"]):
        pm = PartitionedMetapaths.from_global(graphs, rank, world, widths=[width],
                                              transport=transport if world > 1 else "p2p", dtype=dt)
        lo, hi = pm.row_range
        X_loc, y_loc = X[lo:hi].contiguous(), labels[lo:hi]
        idx_loc = pm.local_index(idx_train)
        n_train = global_count(idx_loc.numel(), dev) if world > 1 else idx_loc.numel()
        runs = []
        for _ in range(2):
            model = make_model(M, F_in, a, 0.0).to(dev).to(dt)
            if rank == 0:
                model.load_state_dict(init)
            if world > 1:
                broadcast_parameters(model)
            reset_streams()
            runs.append(train(model, pm, X_loc, y_loc, idx_loc, n_train, 3))
        for op in pm.union.ops.values():
            op.check_status()
        (logits, grads, w), (logits_b, grads_b, w_b) = runs
        line = {"mode": "check", "model": "HAN", "graph": "acm_like", "n": n, "nnz": [g.nnz for g in graphs],
                "widths": [F_in, width, a.classes], "world": world, "rank": rank,
                "transport": pm.op(width).transport, "slot_shift": pm.slot_shift,
                "halo_rows_union": pm.halo_rows, "halo_rows_per_metapath": pm.halo_rows_per_graph}
        line.update(check_metrics(a.dtype, logits, r_logits[lo:hi], grads, r_grads, w, r_w,
                                  torch.equal(logits, logits_b)
                                  and all(torch.equal(grads[k], grads_b[k]) for k in grads)
                                  and all(torch.equal(w[k], w_b[k]) for k in w)))
        print(json.dumps(line), flush=True)
        pm.close()
        del pm, runs


def powerlaw_with_loops(n, deg, seed, dev):
    g = S.powerlaw_csr(n, deg, seed=seed, device=dev)
    rp, cc = with_self_loops(g.rowptr, g.col, 0)
    return CSRGraph(rp, cc, None, n, n)


def layer1_reference(g, rows, X, W, a_src, a_dst, H, Fp):
    """float64 output of metapath 0's attention (ELU twice, all heads) for the global rows `rows`."""
    out = []
    W64, as64, ad64 = W.double(), a_src.double(), a_dst.double()
    for r in rows.tolist():
        cols = g.col[g.rowptr[r]:g.rowptr[r + 1]].long()
        Whj = (X[cols].double() @ W64).view(-1, H, Fp)
        Whi = (X[r].double() @ W64).view(H, Fp)
        z = (Whi * as64).sum(-1)[None, :] + (Whj * ad64[None]).sum(-1)
        att = torch.softmax(torch.nn.functional.leaky_relu(z, 0.2), dim=0)
        out.append(torch.nn.functional.elu(torch.nn.functional.elu((att[:, :, None] * Whj).sum(0).reshape(-1))))
    return torch.stack(out)


def run_time(a, rank, world, dev):
    H, Fp, C, F_in = a.heads, a.hidden, a.classes, a.features
    info = device_info(dev)
    graphs = [powerlaw_with_loops(a.nodes, d, 7 + m, dev) for m, d in enumerate(a.degs)]
    M = len(graphs)
    width = M * H * Fp
    runs = {}
    for name in a.time_dtypes:
        dt = DTYPES[name]
        pm = PartitionedMetapaths.from_global(graphs, rank, world, widths=[width], transport=a.transport, dtype=dt)
        lo, hi = pm.row_range
        n_loc = hi - lo
        X = S.hashed_feature_block(lo, hi, F_in, dev).to(dt)
        labels = (torch.arange(lo, hi, device=dev) * 2654435761 % C).to(torch.int64)
        idx_loc = torch.arange(0, n_loc, 3, device=dev)  # every third row trains
        torch.manual_seed(0)
        model = make_model(M, F_in, a, 0.6).to(dev).to(dt)
        if world > 1:
            broadcast_parameters(model)
        n_train = global_count(idx_loc.numel(), dev) if world > 1 else idx_loc.numel()
        opt = torch.optim.Adam(model.parameters(), lr=0.005)

        def step(model=model, opt=opt, X=X, pm=pm, labels=labels, idx_loc=idx_loc, n_train=n_train):
            model.train()
            opt.zero_grad(set_to_none=True)
            out = model(pm, X)
            partitioned_cross_entropy(out[idx_loc].float(), labels[idx_loc], n_train).backward()
            if world > 1:
                allreduce_gradients(model)
            opt.step()

        def forward(model=model, X=X, pm=pm):
            model.train()
            with torch.no_grad():
                model(pm, X)

        Wh = torch.randn(n_loc, width, device=dev).to(dt)

        def exchange(pm=pm, Wh=Wh):
            pm.op(width).exchange_only(Wh)

        runs[name] = {"pm": pm, "model": model, "X": X, "step": step, "forward": forward, "exchange": exchange,
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
    for name, r in runs.items():
        pm, model, X = r["pm"], r["model"], r["X"]
        lo, hi = pm.row_range
        n_loc = hi - lo
        r["peak_step_gb"] = peak_step_gb(r["step"], dev)
        # float64 spot check of sampled first-layer rows of metapath 0 (eval mode: no dropout)
        model.eval()
        layer = model.layers[0]
        conv0 = list(layer.gat_layers)[0]
        heads = list(conv0.attentions)
        with torch.no_grad():
            Xg = S.hashed_feature_block(0, a.nodes, F_in, dev).to(X.dtype)
            W = torch.cat([hd.W for hd in heads], dim=1)
            Wh_loc = torch.cat([X @ torch.cat([hd.W for hd in c.attentions], dim=1) for c in layer.gat_layers], dim=1)
            g, shift = pm.attention()
            Wh_c = Fn.halo_exchange(pm.union, Wh_loc)
            a_all = torch.stack([torch.stack([hd.a[:, 0] for hd in c.attentions]) for c in layer.gat_layers]).float()
            nc = Wh_c.shape[0]
            Wh4 = Wh_c.view(nc, M, H, Fp).float()
            s = (Wh4[:n_loc] * a_all[None, :, :, :Fp]).sum(-1).permute(1, 0, 2).reshape(M * n_loc, H)
            t = (Wh4 * a_all[None, :, :, Fp:]).sum(-1).permute(1, 0, 2).reshape(M * nc, H)
            z = Fn.gat_aggregate(g, Wh_c, s, t, H, Fp, 0.2, elu=2, batch=M)
            gen = torch.Generator(device="cpu").manual_seed(17 + rank)
            rows = torch.randint(0, max(n_loc, 1), (256,), generator=gen).to(dev)
            ref = layer1_reference(graphs[0], rows + lo, Xg, W, torch.stack([hd.a[:Fp, 0] for hd in heads]),
                                   torch.stack([hd.a[Fp:, 0] for hd in heads]), H, Fp)
            got = z[rows, :H * Fp].double()
            err = float((got - ref).abs().max().item()) / max(float(ref.abs().max().item()), 1e-30)
            del Xg
        for o in pm.union.ops.values():
            o.check_status()
        line = {"mode": "time", "dtype": name, "world": world, "rank": rank, **info, "n": a.nodes, "degs": a.degs,
                "nnz": [g.nnz for g in graphs], "rows_local": n_loc, "widths": [F_in, width, C], "heads": H,
                "transport": a.transport, "halo_rows_union": pm.halo_rows,
                "halo_rows_sum_per_metapath": sum(pm.halo_rows_per_graph),
                "halo_bytes_per_exchange": halo_bytes(pm.union),
                "peak_mem_gb": round(torch.cuda.max_memory_allocated(dev) / 1e9, 2), "peak_step_gb": r["peak_step_gb"],
                "train_step_ms": min(r["train_step_ms"]), "forward_ms": min(r["forward_ms"]),
                "exchange_only_ms": min(r["exchange_only_ms"]) if r["exchange_only_ms"] else None,
                "rounds_ms": {k: r[k] for k in ("train_step_ms", "forward_ms", "exchange_only_ms")},
                "layer1_sampled_rel_err": err, "layer1_ok": err <= (1e-5 if name == "fp32" else 1e-2)}
        print(json.dumps(line), flush=True)
    for r in runs.values():
        r["pm"].close()


def main():
    ap = argparse.ArgumentParser()
    mode = ap.add_mutually_exclusive_group(required=True)
    mode.add_argument("--check", action="store_true")
    mode.add_argument("--time", action="store_true")
    ap.add_argument("--transports", nargs="+", default=["p2p", "ce", "nccl"])
    ap.add_argument("--transport", default="p2p")
    ap.add_argument("--nodes", type=int, default=2_000_000)
    ap.add_argument("--degs", type=float, nargs="+", default=[4.0, 16.0, 48.0])
    ap.add_argument("--features", type=int, default=128)
    ap.add_argument("--heads", type=int, default=8)
    ap.add_argument("--hidden", type=int, default=8)
    ap.add_argument("--classes", type=int, default=3)
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
