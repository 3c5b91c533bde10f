#!/usr/bin/env python
"""GraphSAGE over a feature table sharded across the GPUs of a node (torchrun, one rank per GPU): each rank holds one
row block of the table in a peer-mapped buffer (`partition.ShardedTable`), samples its own minibatches from the
replicated CSR (seed + rank), and the fused gather reads every sampled row from its owner.  Training: the loss
`partitioned_cross_entropy(logits, y, world * B)`, one gradient all-reduce, the optimizer step.  Features come from
`synthetic.hashed_feature_block`, so any rank recomputes any row in float64.  One JSON line per rank and measurement.

    torchrun --nproc-per-node N tools/sage_sharded.py --check
    torchrun --nproc-per-node N tools/sage_sharded.py --time [--out profiles/sage_sharded_time.jsonl]
    python tools/sage_sharded.py --time          (one GPU: the shard-lookup A/B only)

--check: every rank compares its sharded gather and one training step (loss and every gradient after the
  all-reduce) with the same computations over a replica of the table on the same rank, bit for bit; runs 3 Adam
  steps and checks that the weights are identical on every rank; and compares them with one process that runs the
  union of the ranks' minibatches with the same loss rule (max |diff| <= 1e-5).
--time: (1) the Reddit-shaped headline gather (B = 1024, fanout (25, 10), 232,965 x 602 fp32, L2 flushed between
  iterations as bench.py does) over a tensor table and over ShardedTable.local with 1, 2 and 8 shards on one GPU,
  the variants alternated in one run: the cost of the shard lookup.  With 2 or more ranks: (2) the gather and a
  training step, replicated table against sharded, and the bytes read from peers per step; (3) a float64 spot check
  of sampled gathered rows; (4) where memory allows, a 111 M x 602 fp32 table (267 GB) that no single GPU holds.
  Device name and power limit are read in the same run."""
import argparse
import copy
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from graphneuralnetwork_b200 import functional as Fn  # noqa: E402
from graphneuralnetwork_b200 import synthetic as S  # noqa: E402
from graphneuralnetwork_b200.layers import GraphSage  # noqa: E402
from graphneuralnetwork_b200.partition import (ShardedTable, allreduce_gradients, broadcast_parameters,  # noqa: E402
                                               locate_rows, partitioned_cross_entropy)
from gcn_dist_train import device_info  # noqa: E402

CLASSES = 41


def minibatch(g, n_nodes, B, fan, seed, dev):
    """Batch ids and sampled hops of one minibatch (device sampler on the replicated CSR), labels = id % CLASSES."""
    gen = torch.Generator(device="cpu").manual_seed(seed)
    src = torch.randint(0, n_nodes, (B,), generator=gen, dtype=torch.int32).to(dev)
    blocks = Fn.multihop_sampling(g, src, fan, seed)
    return blocks, (src.to(torch.int64) % CLASSES)


def flat_params(model):
    return torch.cat([p.detach().reshape(-1) for p in model.parameters()])


def bitwise(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def check(rank, world, dev):
    N, F, B, fan, steps = 20_000, 602, 256, [10, 5], 3
    g = S.powerlaw_csr(N, 12.0, seed=5, device=dev, with_values=False)
    bounds = [N * p // world for p in range(world + 1)]
    lo, hi = bounds[rank], bounds[rank + 1]
    st = ShardedTable(S.hashed_feature_block(lo, hi, F, dev), bounds, rank, world)
    replica = Fn.pad_table(S.hashed_feature_block(0, N, F, dev))
    seed = lambda r, s: 1000 + 100 * r + s  # noqa: E731  minibatch of rank r at step s
    res = {"rank": rank, "world": world}

    blocks, y = minibatch(g, N, B, fan, seed(rank, 0), dev)
    gb = [(blocks[2], B * fan[0], fan[1]), (blocks[1], B, fan[0]), (blocks[0], B, 1)]
    ok = True
    for reduce in ("mean", "sum", "max"):
        a = Fn.gather_reduce_multi_raw(replica, gb, reduce)
        b = Fn.gather_reduce_multi_raw(st, gb, reduce)
        ok &= all(bitwise(x, z) for x, z in zip(a, b))
    res["gather_bitwise"] = bool(ok)

    torch.manual_seed(0)
    base = GraphSage(F, [64, CLASSES], fan).to(dev)
    broadcast_parameters(base)

    def step(model, table, blocks, y):
        model.zero_grad(set_to_none=True)
        loss = partitioned_cross_entropy(model.forward_sampled(table, blocks), y, world * B)
        loss.backward()
        allreduce_gradients(model)
        return loss.detach()

    one = {}
    for name, table in (("replica", replica), ("sharded", st)):
        m = copy.deepcopy(base).train()
        loss = step(m, table, blocks, y)
        one[name] = (loss, [p.grad for p in m.parameters()])
    res["step_bitwise"] = bool(bitwise(one["replica"][0].reshape(1), one["sharded"][0].reshape(1)) and
                               all(bitwise(p, q) for p, q in zip(one["replica"][1], one["sharded"][1])))

    # 3 Adam steps over the sharded table, data parallel
    m = copy.deepcopy(base).train()
    opt = torch.optim.Adam(m.parameters(), lr=0.01)
    for s in range(steps):
        bl, yy = minibatch(g, N, B, fan, seed(rank, s), dev)
        step(m, st, bl, yy)
        opt.step()
    w = flat_params(m)
    every = [torch.empty_like(w) for _ in range(world)]
    dist.all_gather(every, w)
    res["weights_equal_across_ranks"] = all(torch.equal(every[0], e) for e in every)

    # one process, the union of the ranks' minibatches, same loss rule (Σ over all rows / world·B)
    u = copy.deepcopy(base).train()
    opt = torch.optim.Adam(u.parameters(), lr=0.01)
    for s in range(steps):
        u.zero_grad(set_to_none=True)
        total = 0.0
        for r in range(world):
            bl, yy = minibatch(g, N, B, fan, seed(r, s), dev)
            total = total + partitioned_cross_entropy(u.forward_sampled(replica, bl), yy, world * B)
        total.backward()
        opt.step()
    res["weights_vs_union_max_abs"] = float((flat_params(u) - w).abs().max())
    print(json.dumps(res), flush=True)
    st.close()


# ---- timing ---------------------------------------------------------------------------------
_flush = None


def flush_l2(dev):
    global _flush
    if _flush is None:
        _flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    _flush.zero_()


def time_variants(variants, steps, reps, dev, sync=None):
    """ms per call of each variant (median over `reps` rounds of `steps` calls, the L2 flushed before every call and
    outside the events), the variants alternated round by round."""
    per = {k: [] for k in variants}
    for k, fn in variants.items():  # warm-up
        fn(0)
    for r in range(reps):
        for k, fn in variants.items():
            tot = 0.0
            for i in range(steps):
                flush_l2(dev)
                if sync:
                    sync()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn(r * steps + i)
                b.record()
                b.synchronize()
                tot += a.elapsed_time(b)
            per[k].append(tot / steps)
    return {k: {"ms_median": sorted(v)[len(v) // 2], "ms_min": min(v), "ms_max": max(v)} for k, v in per.items()}


def headline_blocks(n_nodes, pool, seed, dev):
    B, (f1, f2) = 1024, (25, 10)
    gen = torch.Generator().manual_seed(seed)
    return [[torch.randint(0, n_nodes, (s,), generator=gen, dtype=torch.int32).to(dev) for s in (B, B * f1, B * f1 * f2)]
            for _ in range(pool)]


def time_lookup_ab(dev, info, out, steps, reps):
    """One GPU: the headline gather over a tensor table and over ShardedTable.local with 1, 2 and 8 shards."""
    N, F, B, (f1, f2) = 232_965, 602, 1024, (25, 10)
    X = S.hashed_feature_block(0, N, F, dev)
    tables = {"tensor": Fn.pad_table(X)}
    for k in (1, 2, 8):
        b = [N * p // k for p in range(k + 1)]
        tables[f"sharded_{k}"] = ShardedTable.local([X[b[s]:b[s + 1]] for s in range(k)])
    del X
    pool = headline_blocks(N, 8, 100, dev)
    outs = [Fn._padded_empty(B * f1, F, torch.float32, dev), Fn._padded_empty(B, F, torch.float32, dev)]

    def run(table):
        return lambda i: Fn.gather_reduce_multi_raw(table, [(pool[i % 8][2], B * f1, f2), (pool[i % 8][1], B, f1)],
                                                    "mean", outs=outs)
    res = time_variants({k: run(t) for k, t in tables.items()}, steps, reps, dev)
    ref = {}
    for k, t in tables.items():  # the same outputs from every variant
        Fn.gather_reduce_multi_raw(t, [(pool[0][2], B * f1, f2), (pool[0][1], B, f1)], "mean", outs=outs)
        ref[k] = [o.clone() for o in outs]
    same = all(bitwise(a, b) for k in ref for a, b in zip(ref["tensor"], ref[k]))
    line = dict(info, what="shard_lookup_ab_1gpu", workload="B=1024, fanout (25,10), 232,965 x 602 fp32, mean, "
                "hop-2 + hop-1 in one launch; L2 flushed (256 MB written) before every call, outside the events",
                steps=steps, reps=reps, outputs_bitwise_equal=bool(same), ms=res)
    print(json.dumps(line), flush=True)
    out.write(json.dumps(line) + "\n")
    for t in tables.values():
        if isinstance(t, ShardedTable):
            t.close()


def time_multi(rank, world, dev, info, out, steps, reps):
    """2 or more ranks: gather and training step, replicated against sharded; bytes read from peers; float64 check."""
    N, F, B, fan = 232_965, 602, 1024, [25, 10]
    bounds = [N * p // world for p in range(world + 1)]
    st = ShardedTable(S.hashed_feature_block(bounds[rank], bounds[rank + 1], F, dev), bounds, rank, world)
    replica = Fn.pad_table(S.hashed_feature_block(0, N, F, dev))
    g = S.powerlaw_csr(N, 492.0, seed=0, device=dev, with_values=False)
    pool = [minibatch(g, N, B, fan, 100 * rank + i, dev) for i in range(8)]
    outs = [Fn._padded_empty(B * fan[0], F, torch.float32, dev), Fn._padded_empty(B, F, torch.float32, dev)]

    def gather(table):
        return lambda i: Fn.gather_reduce_multi_raw(
            table, [(pool[i % 8][0][2], B * fan[0], fan[1]), (pool[i % 8][0][1], B, fan[0])], "mean", outs=outs)
    torch.manual_seed(0)
    base = GraphSage(F, [128, CLASSES], fan).to(dev).train()
    broadcast_parameters(base)
    models = {"replicated": copy.deepcopy(base), "sharded": copy.deepcopy(base)}
    opts = {k: torch.optim.Adam(m.parameters(), lr=0.01) for k, m in models.items()}

    def train(name, table):
        m, opt = models[name], opts[name]

        def fn(i):
            blocks, y = pool[i % 8]
            m.zero_grad(set_to_none=True)
            partitioned_cross_entropy(m.forward_sampled(table, blocks), y, world * B).backward()
            allreduce_gradients(m)
            opt.step()
        return fn
    sync = lambda: dist.barrier()  # noqa: E731  ranks enter every timed call together
    res = time_variants({"gather_replicated": gather(replica), "gather_sharded": gather(st),
                         "step_replicated": train("replicated", replica), "step_sharded": train("sharded", st)},
                        steps, reps, dev, sync=sync)
    # bytes read from peers per step: every sampled id another rank owns, times the row bytes (hop-2 and hop-1
    # neighbours and the batch's own rows)
    remote = 0
    for blocks, _ in pool:
        for ids in blocks:
            s, _ = locate_rows(ids, bounds)
            remote += int(((s >= 0) & (s != rank)).sum())
    remote_bytes = remote / len(pool) * st.ld * 4
    # float64 spot check: sampled output rows of the sharded gather against recomputed features
    blocks, _ = pool[0]
    o2, o1 = Fn.gather_reduce_multi_raw(st, [(blocks[2], B * fan[0], fan[1]), (blocks[1], B, fan[0])], "mean")
    rows = torch.randint(0, B, (64,), device=dev)
    ids = blocks[1].view(B, fan[0])[rows].reshape(-1)
    ref = S.hashed_features(ids, F, torch.float64).view(64, fan[0], F).mean(1)
    err = float((o1[rows].double() - ref).abs().max() / ref.abs().max())
    line = dict(info, what="sharded_vs_replicated", rank=rank, world=world, workload="232,965 x 602 fp32, B=1024 per "
                "rank, fanout (25,10), GraphSage 602->128->41 (training step: forward, backward, all-reduce, Adam)",
                steps=steps, reps=reps, ms=res, remote_bytes_per_step=remote_bytes, spot_check_rel_err_f64=err)
    print(json.dumps(line), flush=True)
    out.write(json.dumps(line) + "\n")
    st.close()
    del replica
    torch.cuda.empty_cache()

    # capacity: 111 M x 602 fp32 (papers100M-shaped node set), over the ranks
    N = 111_059_956
    per_rank = (N // world + 1) * 604 * 4
    free = torch.cuda.mem_get_info(dev)[0]
    # the generated block and the shard it is copied into are both resident while the table is built
    ok = torch.tensor([1 if free > 2 * per_rank + (8 << 30) else 0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if not ok.item():
        line = dict(info, what="capacity_111M", rank=rank, world=world, skipped=f"building a {per_rank / 1e9:.0f} GB "
                    f"shard needs twice that, with the generated block ({free / 1e9:.0f} GB free)")
    else:
        bounds = [N * p // world for p in range(world + 1)]
        X = torch.empty((bounds[rank + 1] - bounds[rank], F), device=dev)
        S.hashed_feature_block(bounds[rank], bounds[rank + 1], F, dev, out=X)
        st = ShardedTable(X, bounds, rank, world)
        del X
        torch.cuda.empty_cache()
        blk = headline_blocks(N, 8, 200 + rank, dev)

        def cap(i):
            Fn.gather_reduce_multi_raw(st, [(blk[i % 8][2], B * 25, 10), (blk[i % 8][1], B, 25)], "mean", outs=outs)
        r = time_variants({"gather_sharded": cap}, steps, reps, dev, sync=sync)
        Fn.gather_reduce_multi_raw(st, [(blk[0][2], B * 25, 10), (blk[0][1], B, 25)], "mean", outs=outs)
        rows = torch.randint(0, B, (64,), device=dev)
        ids = blk[0][1].view(B, 25)[rows].reshape(-1)
        ref = S.hashed_features(ids, F, torch.float64).view(64, 25, F).mean(1)
        err = float((outs[1][rows].double() - ref).abs().max() / ref.abs().max())
        line = dict(info, what="capacity_111M", rank=rank, world=world, table_gb=N * 604 * 4 / 1e9,
                    workload="111,059,956 x 602 fp32, uniform ids, B=1024, fanout (25,10)", ms=r,
                    spot_check_rel_err_f64=err)
        st.close()
    print(json.dumps(line), flush=True)
    out.write(json.dumps(line) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--time", action="store_true")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="jsonl file the --time lines are appended to")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sage_sharded.py needs CUDA devices (the gather has no CPU form)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    try:
        if args.check:
            if world < 2:
                raise SystemExit("--check needs 2 or more ranks (torchrun --nproc-per-node N)")
            check(rank, world, dev)
        if args.time:
            info = device_info(dev)
            out = open(args.out, "a") if args.out and rank == 0 else open(os.devnull, "w")
            with out:
                if rank == 0:
                    time_lookup_ab(dev, info, out, args.steps, args.reps)
                if world > 1:
                    dist.barrier()
                    time_multi(rank, world, dev, info, out, args.steps, args.reps)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
