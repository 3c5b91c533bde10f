#!/usr/bin/env python
"""Sparse GTN training across GPUs (torchrun, one rank per GPU): the drop-in `GTN_Model` on a
`partition.PartitionedRelationStack`, replicated weights, the global loss rule and one gradient all-reduce per step.
One JSON line per rank and configuration on stdout.

    torchrun --nproc-per-node N tools/gtn_dist_train.py --check
    torchrun --nproc-per-node N tools/gtn_dist_train.py --time [--out profiles/gtn_dist_train_time_Ngpu.jsonl]

--check (a DBLP-shaped stack from tools/gtn_sparse.py's `dblp_like` at 1/20 scale, C = 2, w_out 64, 1 to 3 layers):
  every rank also trains the same seeded model over the WHOLE RelationStack on its GPU and compares its rows of the
  logits (1e-5), every gradient at step 1 after the all-reduce (5e-5) and the weights after 3 Adam steps (1e-4), all
  max-normalised; the 3-step run is repeated and must be bit-identical.  One training step (forward, backward,
  gradient all-reduce) runs under torch.cuda.set_sync_debug_mode("error") once the stack is built: it reads nothing
  back to the host.
--time: DBLP x1 (the generator of tools/gtn_sparse.py), 2 and 3 layers, C = 2, 334 features: the stack build time,
  the per-rank nnz of every P_l, the training step (median of --reps host-clock windows around one step that ends in a
  device synchronise, after a warm-up), peak memory per rank and the device time of the reduce kernels in one
  profiled step (torch.profiler, a run of its own).  Then DBLP x10 at 1 and 2 layers: whether it fits at this world
  size (a `start` line precedes each attempt, so an attempt that kills the run is visible) and its step time.
  Device name and power limit are read in the same run."""
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
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from graphneuralnetwork_b200 import _lib  # noqa: E402
from graphneuralnetwork_b200.layers.gtn import RelationStack  # noqa: E402
from graphneuralnetwork_b200.partition import (PartitionedRelationStack, allreduce_gradients,  # noqa: E402
                                               broadcast_parameters, global_count, partitioned_cross_entropy)
from gcn_dist_train import device_info, rel  # noqa: E402
from gtn_sparse import DBLP, _inputs, _model, dblp_like  # noqa: E402

K, C, W_OUT = 5, 2, 64
BOUNDS = {"logits": 1e-5, "grad": 5e-5, "weights": 1e-4}


def _step(model, adj, X, target, labels, n_train, opt=None, world=1):
    """One training step; n_train None: the 1-GPU model over the whole stack (mean loss), else the partitioned one."""
    if opt is not None:
        opt.zero_grad(set_to_none=True)
    y, _ = model(adj, X, target)
    if n_train is None:
        loss = torch.nn.functional.cross_entropy(y, labels)
    else:
        loss = partitioned_cross_entropy(y, labels, n_train)
    loss.backward()
    if n_train is not None and world > 1:
        allreduce_gradients(model)
    return y


def train(model, adj, X, target, labels, n_train, steps, world):
    """`steps` Adam steps: (logits of step 1, gradients of step 1, final weights)."""
    opt = torch.optim.Adam(model.parameters(), lr=0.005, weight_decay=1e-3)
    logits1 = grads1 = None
    for s in range(steps):
        y = _step(model, adj, X, target, labels, n_train, opt, world)
        if s == 0:
            logits1 = y.detach().clone()
            grads1 = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
        opt.step()
    return logits1, grads1, {k: v.detach().clone() for k, v in model.state_dict().items()}


def run_check(rank, world, dev):
    rels, n = dblp_like(dev, scale=0.05, seed=3)
    stack = RelationStack.from_relations(rels)
    X, target, labels = _inputs(n, 16, dev)
    ok = True
    for L in (1, 2, 3):
        ref = _model(K, C, L, 16, L, dev)
        init = {k: v.clone() for k, v in ref.state_dict().items()}
        r_logits, r_grads, r_w = train(ref, stack, X, target, labels, None, 3, 1)
        ps = PartitionedRelationStack(stack, rank, world, L, C * W_OUT)
        lo, hi = ps.row_range
        mine = (target >= lo) & (target < hi)
        t_loc, y_loc = target[mine] - lo, labels[mine]
        n_train = global_count(int(t_loc.numel()), dev) if world > 1 else int(t_loc.numel())
        X_loc = X[lo:hi].contiguous()
        runs = []
        for _ in range(2):
            model = _model(K, C, L, 16, L, dev)
            model.load_state_dict(init)
            if world > 1:
                broadcast_parameters(model)
            runs.append(train(model, ps, X_loc, t_loc, y_loc, n_train, 3, world))
        # one more step with nothing read back to the host
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            _step(model, ps, X_loc, t_loc, y_loc, n_train, None, world)
            no_host_reads = True
        finally:
            torch.cuda.set_sync_debug_mode("default")
        torch.cuda.synchronize()
        ps.check_status()
        (logits, grads, w), (logits_b, grads_b, w_b) = runs
        line = {"mode": "check", "model": "GTN", "graph": "dblp_like x0.05", "n": n, "layers": L, "C": C,
                "world": world, "rank": rank, "bounds": ps.bounds, "nnz_P_local": ps.nnz_per_layer,
                "logits_rel_err": rel(logits, r_logits[mine]) if logits.numel() else 0.0,
                "grad_rel_err": max(rel(grads[k], r_grads[k]) for k in r_grads),
                "weights_rel_err": max(rel(w[k], r_w[k]) for k in r_w),
                "bitwise_repeat": bool(torch.equal(logits, logits_b) and all(torch.equal(grads[k], grads_b[k])
                                                                             for k in grads)
                                       and all(torch.equal(w[k], w_b[k]) for k in w)),
                "step_without_host_reads": no_host_reads}
        line["ok"] = (line["logits_rel_err"] <= BOUNDS["logits"] and line["grad_rel_err"] <= BOUNDS["grad"]
                      and line["weights_rel_err"] <= BOUNDS["weights"] and line["bitwise_repeat"])
        ok &= line["ok"]
        print(json.dumps(line), flush=True)
        ps.close()
    return ok


def _timed_ms(fn, reps, world):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return ts


def _reduce_kernel_ms(step, dev):
    """Device time of the reduce kernels (peer_reduce_rows_kernel) and of the flag waits in one profiled step."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    red = wait = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        t = e.cuda_time_total if t is None else t
        if "peer_reduce_rows_kernel" in e.key:
            red += t / 1e3
        elif "peer_wait_kernel" in e.key:
            wait += t / 1e3
    return round(red, 3), round(wait, 3)


def time_config(rels, n, L, rank, world, dev, reps, shape, info, out_rows, max_nnz_per_rank=None):
    X, target, labels = _inputs(n, DBLP["feats"], dev)
    stack = RelationStack.from_relations(rels)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    ps = PartitionedRelationStack(stack, rank, world, L, C * W_OUT, max_nnz_per_rank=max_nnz_per_rank)
    torch.cuda.synchronize()
    build_ms = (time.perf_counter() - t0) * 1e3
    lo, hi = ps.row_range
    mine = (target >= lo) & (target < hi)
    t_loc, y_loc = target[mine] - lo, labels[mine]
    n_train = global_count(int(t_loc.numel()), dev) if world > 1 else int(t_loc.numel())
    X_loc = X[lo:hi].contiguous()
    del X
    model = _model(K, C, L, DBLP["feats"], L, dev)
    if world > 1:
        broadcast_parameters(model)
    opt = torch.optim.Adam(model.parameters(), lr=0.005)

    def step():
        _step(model, ps, X_loc, t_loc, y_loc, n_train, opt, world)
        opt.step()

    step()  # warm-up
    step()
    torch.cuda.reset_peak_memory_stats(dev)
    ms = _timed_ms(step, reps, world)
    peak = torch.cuda.max_memory_allocated(dev) / 1e9
    red_ms, wait_ms = _reduce_kernel_ms(step, dev)
    ps.check_status()
    every = [None] * world
    nnz = ps.nnz_per_layer
    if world > 1:
        dist.all_gather_object(every, nnz)
    else:
        every = [nnz]
    r = {"mode": "time", "shape": shape, "n": n, "K": K, "C": C, "layers": L, "feats": DBLP["feats"], "world": world,
         "rank": rank, "bounds": ps.bounds, "nnz_P_local": nnz, "nnz_P_per_rank": every,
         "nnz_P_total": [sum(e[l] for e in every) for l in range(L)], "build_ms": round(build_ms, 1),
         "step_ms_median": round(statistics.median(ms), 2), "step_ms": [round(t, 2) for t in ms],
         "peak_mem_gb": round(peak, 2), "reduce_kernels_ms_per_step": red_ms, "flag_waits_ms_per_step": wait_ms,
         "reps": reps, **info}
    print(json.dumps(r), flush=True)
    out_rows.append(r)
    ps.close()
    del ps, model, opt, stack
    gc.collect()
    torch.cuda.empty_cache()


def run_time(rank, world, dev, reps, out):
    info = device_info(dev)
    rows = []

    def flush():
        if out and rank == 0:
            os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
            with open(out, "w") as f:
                for r in rows:
                    f.write(json.dumps(r) + "\n")

    rels, n = dblp_like(dev)
    for L in (2, 3):
        time_config(rels, n, L, rank, world, dev, reps, "dblp", info, rows)
        flush()
    del rels
    gc.collect()
    torch.cuda.empty_cache()
    rels, n = dblp_like(dev, scale=10.0, seed=1)
    for L in (1, 2):
        start = {"mode": "time", "shape": "dblp_x10", "n": n, "layers": L, "world": world, "rank": rank,
                 "start": True, **info}
        print(json.dumps(start), flush=True)
        rows.append(start)
        flush()
        try:
            time_config(rels, n, L, rank, world, dev, reps, "dblp_x10", info, rows)
            rows[-1]["fits"] = True
        except (_lib.GnnError, torch.OutOfMemoryError) as e:
            # an out-of-memory error on one rank leaves the others in a collective: torchrun then ends the run, and
            # the `start` line without a result shows it
            r = {"mode": "time", "shape": "dblp_x10", "n": n, "layers": L, "world": world, "rank": rank,
                 "fits": False, "refused": f"{type(e).__name__}: {str(e)[:300]}", **info}
            print(json.dumps(r), flush=True)
            rows.append(r)
        flush()
        gc.collect()
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    mode = ap.add_mutually_exclusive_group(required=True)
    mode.add_argument("--check", action="store_true")
    mode.add_argument("--time", action="store_true")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None, help="--time: rank 0 writes its lines here (JSON lines)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gtn_dist_train: needs CUDA devices (the sparse path has no CPU fallback)")
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ok = True
    try:
        if a.check:
            ok = run_check(rank, world, dev)
        else:
            run_time(rank, world, dev, a.reps, a.out)
    finally:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
