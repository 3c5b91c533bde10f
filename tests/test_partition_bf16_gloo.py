"""partition.allreduce_gradients over gloo on CPU, world_size 2 and 3: bf16 gradients are summed in fp32 and each sum
is rounded once to bf16, identically on every rank; an all-fp32 model is reduced exactly as a plain fp32 all_reduce
of its gradients; plus the C ABI table lists the bf16 partitioned attention entries."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from graphneuralnetwork_b200 import _lib
from graphneuralnetwork_b200.partition import allreduce_gradients


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _model(dtype):
    torch.manual_seed(0)  # the same shapes and weights on every rank
    m = torch.nn.Sequential(torch.nn.Linear(37, 16), torch.nn.Linear(16, 41, bias=False), torch.nn.Linear(41, 3))
    return m.to(dtype)


def _grads(rank, dtype):
    """Rank-dependent gradients with a wide dynamic range (bf16 sums of them round differently per order)."""
    g = torch.Generator().manual_seed(100 + rank)
    out = []
    for p in _model(dtype).parameters():
        x = torch.randn(p.shape, generator=g, dtype=torch.float64) * torch.exp(
            torch.randn(p.shape, generator=g, dtype=torch.float64) * 3)
        out.append(x)
    return out


def _check(rank, world):
    # bf16: the fp32 sum of the ranks' bf16 gradients, rounded once
    m = _model(torch.bfloat16)
    params = list(m.parameters())
    mine = _grads(rank, torch.bfloat16)
    for p, x in zip(params, mine):
        p.grad = x.to(torch.bfloat16)
    params[1].grad = None  # a missing gradient counts as zeros
    allreduce_gradients(m)
    every = [_grads(r, torch.bfloat16) for r in range(world)]
    for k, p in enumerate(params):
        tot = torch.zeros(p.shape, dtype=torch.float32)
        if k != 1:
            for r in range(world):
                tot += every[r][k].to(torch.bfloat16).float()
        assert p.grad.dtype == torch.bfloat16
        assert torch.equal(p.grad, tot.to(torch.bfloat16)), k
    flat = torch.cat([p.grad.float().reshape(-1) for p in params])
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    assert all(torch.equal(x, gathered[0]) for x in gathered)  # identical on every rank
    # fp32: the same result as one plain all_reduce of the flattened gradients
    m = _model(torch.float32)
    params = list(m.parameters())
    for p, x in zip(params, _grads(rank, torch.float32)):
        p.grad = x.float()
    flat = torch.cat([p.grad.reshape(-1) for p in params]).clone()
    dist.all_reduce(flat)
    allreduce_gradients(m)
    off = 0
    for p in params:
        assert p.grad.dtype == torch.float32
        assert torch.equal(p.grad.reshape(-1), flat[off:off + p.numel()])
        off += p.numel()


def _worker(rank, world, port, out_q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        _check(rank, world)
        out_q.put((rank, "ok"))
    except Exception:  # reported to the parent, which fails the test with it
        import traceback
        out_q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_allreduce_gradients_bf16_sums_in_fp32_and_rounds_once(world):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for rank, status in results:
        assert status == "ok", f"rank {rank}:\n{status}"
    for p in procs:
        assert p.exitcode == 0


def test_bf16_partitioned_attention_entries_are_bound():
    for f in ("gnn_gat_fused_bwd_ex_bf16", "gnn_gat_fused_fwd_batch_bf16", "gnn_gat_fused_bwd_batch_bf16"):
        assert f in _lib.SIGNATURES
    # the bf16 twins take the fp32 entries' argument lists
    assert len(_lib.SIGNATURES["gnn_gat_fused_bwd_ex_bf16"][1]) == len(_lib.SIGNATURES["gnn_gat_fused_bwd_ex_f32"][1])
    assert (_lib.SIGNATURES["gnn_gat_fused_fwd_batch_bf16"][1] == _lib.SIGNATURES["gnn_gat_fused_fwd_batch_f32"][1])
    assert (_lib.SIGNATURES["gnn_gat_fused_bwd_batch_bf16"][1] == _lib.SIGNATURES["gnn_gat_fused_bwd_batch_f32"][1])
