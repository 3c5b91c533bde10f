#!/usr/bin/env python
"""Full-graph GCN training across GPUs (torchrun, one rank per GPU): the drop-in `GCN_Model` on a
`partition.PartitionedGraph`, replicated weights, the global loss rule and one gradient all-reduce per step.
One JSON line per rank and configuration on stdout.

    torchrun --nproc-per-node N tools/gcn_dist_train.py --check [--dtype fp32|bf16] [--transports p2p ce nccl]
                                                        [--configs 1:auto 4:2 auto:auto]
    torchrun --nproc-per-node N tools/gcn_dist_train.py --time [--nodes 20000000] [--features 128 --hidden 64 --classes 41]

--check (small graphs every rank holds: a Cora-like graph and a 200 k-row power-law graph, odd widths, dropout 0):
  every rank also trains the same seeded GCN_Model on its GPU over the WHOLE graph and compares its own rows of the
  logits, every gradient at step 1 (after the all-reduce) and the weights after 3 Adam steps; the 3-step run is
  repeated and must be bit-identical.  --dtype bf16: the model, the features and the partition are bf16 and the 1-GPU
  model is the same seeded bf16 model; the bounds are then bf16's (CHECK_BOUNDS).
--time (large graph, each rank generates only its own row block, as bench.py's partitioned-SpMM config does): ms per
  training step (forward + backward + gradient all-reduce + Adam) and per forward, the schedule chosen, a float64
  spot check of sampled first-layer output rows, and the fused bias/ReLU epilogue against the unfused
  `op.forward` + torch bias + ReLU on the same plan, alternated in one run.  The fp32 and the bf16 model (features,
  weights and partition in that dtype) are timed at the same size in one run, their steps alternated; one line per
  dtype with its halo bytes and the peak memory of its step.  Device name and power limit are read in the same
  run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from graphneuralnetwork_b200 import synthetic as S  # noqa: E402
from graphneuralnetwork_b200.graph import CSRGraph  # noqa: E402
from graphneuralnetwork_b200.layers import GCN_Model  # noqa: E402
from graphneuralnetwork_b200.partition import (PartitionedGraph, allreduce_gradients, broadcast_parameters,  # noqa: E402
                                               global_count, partitioned_cross_entropy)


def device_info(dev):
    """Device name and power limit, read in the run that measures."""
    info = {"device": torch.cuda.get_device_name(dev)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(dev.index)],
                           capture_output=True, text=True, timeout=30)
        info["power_limit"] = r.stdout.strip() or None
    except Exception as e:  # the numbers stay valid, their context is then incomplete
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}
# --check bounds per dtype.  fp32: max-normalised errors against the 1-GPU fp32 model.  bf16: logits 1e-2 and step-1
# gradients 3e-2 (the bf16 tolerances of the single-GPU parity tests); the weights after 3 Adam steps are bounded in
# norm, ‖w - w_ref‖₂ / ‖w_ref‖₂ <= 5e-2 over all parameters.  Adam's first steps move a weight by about lr whatever the
# size of its gradient, so an entry whose gradient is near zero may step in opposite directions in two bf16 runs that
# reduce in different orders: such entries set the max-normalised error (reported as weights_rel_err, up to
# 2·steps·lr / max|w|) but contribute little to the norm.
CHECK_BOUNDS = {"fp32": {"logits": 1e-5, "grad": 2e-5, "weights": 1e-4, "weights_norm": None},
                "bf16": {"logits": 1e-2, "grad": 3e-2, "weights": None, "weights_norm": 5e-2}}


def check_metrics(dtype, logits, r_logits, grads, r_grads, w, r_w, repeat):
    """The --check fields of one run against the 1-GPU run, with `ok` under CHECK_BOUNDS[dtype]."""
    b = CHECK_BOUNDS[dtype]
    num = sum(float((w[k].double() - r_w[k].double()).pow(2).sum()) for k in r_w)
    den = sum(float(r_w[k].double().pow(2).sum()) for k in r_w)
    m = {"dtype": dtype, "logits_rel_err": rel(logits, r_logits),
         "grad_rel_err": max(rel(grads[k], r_grads[k]) for k in r_grads),
         "weights_rel_err": max(rel(w[k], r_w[k]) for k in r_w),
         "weights_norm_rel_err": (num / max(den, 1e-300)) ** 0.5, "bitwise_repeat": bool(repeat)}
    m["weights_bound"] = b["weights_norm"] if b["weights"] is None else b["weights"]
    w_ok = (m["weights_rel_err"] <= b["weights"]) if b["weights"] is not None else \
        (m["weights_norm_rel_err"] <= b["weights_norm"])
    m["ok"] = m["logits_rel_err"] <= b["logits"] and m["grad_rel_err"] <= b["grad"] and w_ok and m["bitwise_repeat"]
    return m


def timed_ms(fn, steps, warmup, world, dev):
    """Mean ms per call over `steps` calls after `warmup` (CUDA events; the slowest rank's figure)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    t = torch.tensor([t0.elapsed_time(t1) / steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return round(float(t.item()), 3)


def peak_step_gb(fn, dev):
    """Peak memory while `fn` runs, above what was allocated before it (GB): the step's own working set."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    fn()
    torch.cuda.synchronize()
    return round((torch.cuda.max_memory_allocated(dev) - base) / 1e9, 3)


def halo_bytes(pg):
    """Bytes one exchange moves into this rank, per feature width (forward; the gradient return moves as many)."""
    return {str(F): op.halo_bytes_received if hasattr(op, "halo_bytes_received") else 0 for F, op in pg.ops.items()}


def parse_config(cfg):
    k, c0 = cfg.split(":")
    return (None if k == "auto" else int(k)), (None if c0 == "auto" else int(c0))


def gcn_csr(n, edges, dev):
    """Â = D^-1/2 (A + I) D^-1/2 of an undirected edge list, as a CSRGraph (float64 normalisation)."""
    import scipy.sparse as sp
    e = np.asarray(edges)
    A = sp.coo_matrix((np.ones(len(e)), (e[:, 0], e[:, 1])), shape=(n, n))
    A = ((A + A.T) > 0).astype(np.float64) + sp.eye(n)
    d = np.asarray(A.sum(1)).ravel() ** -0.5
    A = sp.csr_matrix(sp.diags(d) @ A @ sp.diags(d))
    A.sort_indices()
    return CSRGraph(torch.from_numpy(A.indptr.astype(np.int64)).to(dev), torch.from_numpy(A.indices.astype(np.int32)).to(dev),
                    torch.from_numpy(A.data.astype(np.float32)).to(dev), n, n)


def rel(a, b):
    return float((a.double() - b.double()).abs().max().item()) / max(float(b.double().abs().max().item()), 1e-30)


def train(model, X, adj, target, idx, n_train, steps, group=None):
    """`steps` Adam steps; returns (logits of step 1, gradients of step 1, final weights).  n_train None: the
    1-GPU model over the whole graph; else the partitioned model (loss rule + gradient all-reduce)."""
    opt = torch.optim.Adam(model.parameters(), lr=0.01, weight_decay=5e-4)
    logits1 = grads1 = None
    for s in range(steps):
        opt.zero_grad(set_to_none=True)
        out = model(X, adj)
        if n_train is None:  # one GPU: the reference's loss, CrossEntropyLoss over idx_train (GCN/train_eval.py:45)
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


def run_check(a, rank, world, dev):
    F_HID, F_CLS = 16, 41
    graphs = []
    cora = S.cora_like_edges(seed=0)
    graphs.append(("cora_like", S.CORA["n"], lambda: gcn_csr(S.CORA["n"], cora, dev), 301))
    graphs.append(("powerlaw_200k", 200_000, lambda: S.powerlaw_csr(200_000, 10.0, seed=3, device=dev), 37))
    for name, n, make, F_in in graphs:
        g = make()
        gen = torch.Generator().manual_seed(11)
        dt = DTYPES[a.dtype]
        X = (torch.rand(n, F_in, generator=gen) * 2 - 1).to(dev).to(dt)
        labels = torch.randint(0, F_CLS, (n,), generator=gen).to(dev)
        idx_train = torch.randperm(n, generator=gen)[: max(n * 2 // 5, 1)].sort().values.to(dev)
        for layers in a.layers:
            torch.manual_seed(0)
            ref = GCN_Model(F_in, F_HID, F_CLS, layers, 0.0).to(dev).to(dt)
            init = {k: v.clone() for k, v in ref.state_dict().items()}
            r_logits, r_grads, r_w = train(ref, X, g, labels, idx_train, None, 3)
            for transport in (a.transports if world > 1 else ["none"]):
                for cfg in (a.configs if world > 1 else ["1:auto"]):
                    K, c0 = parse_config(cfg)
                    pg = PartitionedGraph.from_global(g, rank, world, widths=[F_HID, F_CLS], waves=K,
                                                      two_pass_chunks=c0, transport=transport if world > 1 else "p2p",
                                                      dtype=dt)
                    lo, hi = pg.row_range
                    X_loc, y_loc = X[lo:hi].contiguous(), labels[lo:hi]
                    idx_loc = pg.local_index(idx_train)
                    n_train = global_count(idx_loc.numel(), dev) if world > 1 else idx_loc.numel()
                    runs = []
                    for _ in range(2):
                        model = GCN_Model(F_in, F_HID, F_CLS, layers, 0.0).to(dev).to(dt)
                        if rank == 0:
                            model.load_state_dict(init)
                        if world > 1:
                            broadcast_parameters(model)
                        runs.append(train(model, X_loc, pg, y_loc, idx_loc, n_train, 3))
                    for op in pg.ops.values():
                        op.check_status()
                    (logits, grads, w), (logits_b, grads_b, w_b) = runs
                    line = {"mode": "check", "graph": name, "n": n, "nnz": int(g.rowptr[-1].item()), "layers": layers,
                            "widths": [F_in, F_HID, F_CLS], "world": world, "rank": rank, "transport": pg.ops[F_HID].transport,
                            "config": cfg, "waves": pg.plan.waves, "two_pass_chunks": pg.plan.two_pass_chunks,
                            "p1_epilogue_skip": 0 if pg.plan.p1 is None else pg.plan.p1.epilogue_skip}
                    line.update(check_metrics(a.dtype, logits, r_logits[lo:hi], grads, r_grads, w, r_w,
                                              torch.equal(logits, logits_b)
                                              and all(torch.equal(grads[k], grads_b[k]) for k in grads)
                                              and all(torch.equal(w[k], w_b[k]) for k in w)))
                    print(json.dumps(line), flush=True)
                    pg.close()
                    del pg, runs
            del ref
        del g


def run_time(a, rank, world, dev):
    from spmm_dist import build_rank_block
    F_in, H, C = a.features, a.hidden, a.classes
    info = device_info(dev)
    csr, bounds, nnz_total = build_rank_block(a.nodes, a.deg, rank, world, dev)
    lo, hi = bounds[rank], bounds[rank + 1]
    n_loc = hi - lo
    X32 = S.hashed_feature_block(lo, hi, F_in, dev)
    labels = (torch.arange(lo, hi, device=dev) * 2654435761 % C).to(torch.int64)
    idx_loc = torch.arange(0, n_loc, 3, device=dev)  # every third row trains
    n_train = global_count(idx_loc.numel(), dev) if world > 1 else idx_loc.numel()
    nnz_loc = int(csr.rowptr[-1].item())
    gb = lambda b: round(b / 1e9, 2)  # noqa: E731
    rows = S.spmm_check_rows(csr, 2048, 17 + rank)
    ax = S.spmm_sampled_reference(csr, rows, F_in)  # the block's CSR holds global column ids
    runs = {}
    for name in a.time_dtypes:
        dt = DTYPES[name]
        esz = 4 if dt == torch.float32 else 2
        # footprint of one rank, 2 layers: the CSR and its two transposes (backward), X, and per layer S = XWᵀ,
        # Y (saved for the ReLU mask), their gradients and the halo buffers; the largest share is 1/world
        foot = {"csr_gb": gb(nnz_loc * 8 + (n_loc + 1) * 8), "transposes_gb": gb(2 * (nnz_loc * 8 + (n_loc + 1) * 8)),
                "x_gb": gb(n_loc * F_in * esz), "activations_gb": gb(n_loc * (4 * H + 4 * C) * esz)}
        foot["total_gb"] = round(sum(foot.values()), 2)
        pg = PartitionedGraph(csr.rowptr, csr.col, csr.val, bounds, rank, world, widths=[H, C], device=dev, waves=None,
                              transport=a.transport, dtype=dt)
        torch.manual_seed(0)
        model = GCN_Model(F_in, H, C, 2, 0.0).to(dev).to(dt)
        if world > 1:
            broadcast_parameters(model)
        opt = torch.optim.Adam(model.parameters(), lr=0.01)
        X = X32.to(dt)

        def step(model=model, opt=opt, X=X, pg=pg):
            opt.zero_grad(set_to_none=True)
            out = model(X, pg)
            partitioned_cross_entropy(out[idx_loc].float(), labels[idx_loc], n_train).backward()
            if world > 1:
                allreduce_gradients(model)
            opt.step()

        def forward(model=model, X=X, pg=pg):
            with torch.no_grad():
                model(X, pg)

        Sh, Sc = torch.randn(n_loc, H, device=dev).to(dt), torch.randn(n_loc, C, device=dev).to(dt)

        def exchange(pg=pg, Sh=Sh, Sc=Sc):
            pg.op(H).exchange_only(Sh)
            pg.op(C).exchange_only(Sc)

        runs[name] = {"pg": pg, "model": model, "X": X, "step": step, "forward": forward, "exchange": exchange,
                      "foot": foot, "train_step_ms": [], "forward_ms": [], "exchange_only_ms": []}
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
        pg, model = r["pg"], r["model"]
        r["peak_step_gb"] = peak_step_gb(r["step"], dev)
        # float64 spot check of sampled first-layer rows: relu((Â·X)[rows] Wᵀ + b), Â·X recomputed from the global ids
        layer0 = model.gcn_blocks.gcn0
        with torch.no_grad():
            Y1 = layer0(r["X"], pg, fused_relu=True)
        ref = torch.clamp_min(ax @ layer0.dense.weight.detach().double().T + layer0.bias.detach().double(), 0.0)
        err = float((Y1[rows].double() - ref).abs().max().item()) / max(float(ref.abs().max().item()), 1e-30)
        for o in pg.ops.values():
            o.check_status()
        line = {"mode": "time", "dtype": name, "world": world, "rank": rank, **info, "n": a.nodes, "nnz": nnz_total,
                "rows_local": n_loc, "widths": [F_in, H, C], "transport": a.transport, "waves": pg.plan.waves,
                "two_pass_chunks": pg.plan.two_pass_chunks,
                "p1_epilogue_skip": 0 if pg.plan.p1 is None else pg.plan.p1.epilogue_skip,
                "halo_bytes_per_exchange": halo_bytes(pg), "footprint_rank": r["foot"],
                "peak_mem_gb": round(torch.cuda.max_memory_allocated(dev) / 1e9, 2), "peak_step_gb": r["peak_step_gb"],
                "train_step_ms": min(r["train_step_ms"]), "forward_ms": min(r["forward_ms"]),
                "exchange_only_ms": min(r["exchange_only_ms"]) if r["exchange_only_ms"] else None,
                "rounds_ms": {k: r[k] for k in ("train_step_ms", "forward_ms", "exchange_only_ms")},
                "layer1_sampled_rel_err": err, "layer1_ok": err <= (1e-5 if name == "fp32" else 1e-2)}
        print(json.dumps(line), flush=True)
    if "fp32" in runs:
        epilogue_ab(a, runs["fp32"], world, dev)
    for r in runs.values():
        r["pg"].close()


def epilogue_ab(a, r, world, dev):
    """The fused bias/ReLU epilogue against op.forward + torch bias + ReLU on the same fp32 plan, alternated."""
    H = a.hidden
    layer0 = r["model"].gcn_blocks.gcn0
    op = r["pg"].op(H)
    Sx = layer0.dense(r["X"]).detach()
    b = layer0.bias.detach()

    def fused():
        op.forward(Sx, bias=b, relu=True)

    def unfused():
        y = op.forward(Sx)
        torch.relu_(y.add_(b))

    ab = {"fused_ms": [], "unfused_ms": []}
    for _ in range(3):
        ab["fused_ms"].append(timed_ms(fused, a.steps, 1, world, dev))
        ab["unfused_ms"].append(timed_ms(unfused, a.steps, 1, world, dev))
    yf, yu = op.forward(Sx, bias=b, relu=True), op.forward(Sx)
    yu = torch.relu(yu + b)
    print(json.dumps({"mode": "epilogue_ab", "dtype": "fp32", "world": world,
                      "rank": dist.get_rank() if world > 1 else 0, "epilogue_ab_ms": ab, "fused_vs_unfused_max_abs_diff": float((yf - yu).abs().max().item())}),
          flush=True)


def main():
    ap = argparse.ArgumentParser()
    mode = ap.add_mutually_exclusive_group(required=True)
    mode.add_argument("--check", action="store_true")
    mode.add_argument("--time", action="store_true")
    ap.add_argument("--transports", nargs="+", default=["p2p", "ce", "nccl"])
    ap.add_argument("--configs", nargs="+", default=["1:auto", "4:2", "auto:auto"], help="waves:two_pass_chunks")
    ap.add_argument("--layers", nargs="+", type=int, default=[2])
    ap.add_argument("--transport", default="p2p")
    ap.add_argument("--nodes", type=int, default=20_000_000)
    ap.add_argument("--deg", type=float, default=13.55)
    ap.add_argument("--features", type=int, default=128)
    ap.add_argument("--hidden", type=int, default=64)
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
