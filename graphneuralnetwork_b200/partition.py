"""1-D row-partitioned SpMM with a wave-pipelined halo exchange over NVLink (SURVEY.md §8e).

The reference has no multi-GPU path for message passing (only single-process nn.DataParallel,
HAN/train_utils/train_eval.py:46); the seam this serves is `torch.spmm(adj, support)` and its autograd
(GCN/GCN.py:43) on a graph too large for one GPU.  One process per GPU.  Rank p owns the contiguous row
block [bounds[p], bounds[p+1]) of Â, X and Y (blocks balanced by nnz).

Plan (host logic on plain tensors, device-agnostic, gloo-testable — `build_halo_plan`):
  * the rank's CSR is split by column into local columns (re-based) and remote columns, the latter
    remapped into a compact, de-duplicated HALO whose slots are ordered by (owner peer, wave, id);
  * rows are cut into K nnz-balanced ROW CHUNKS; a halo row belongs to wave w if chunk w is the first
    chunk that needs it, so after waves 0..w have landed chunk w has everything it reads;
  * row classes: INTERIOR rows (no remote column) and MIXED rows.  Chunks [0, c0) are "two-pass": the
    local columns of their mixed rows are aggregated while the exchange is in flight and the remote
    columns are added after the wave lands (read-modify-write of those Y rows only); chunks [c0, K) are
    "single-pass": their mixed rows are aggregated once, from [X_local ; halo], after their wave lands —
    no read-modify-write at all.  c0 is chosen by a byte model of the overlap (or given).
Step (`PartitionedSpmm.forward`):
    comm stream:  for w in waves: push wave w to every peer (gnn_halo_push, TMA mover) ; signal flags
    main stream:  P1 = local columns of (interior rows ∪ mixed rows of two-pass chunks)
                  for w in waves: wait wave-w flags ; P2_w = the mixed rows of chunk w
There is no collective on the data path: arrival is announced per wave through monotonic flags in peer
memory (gnn_peer_signal / gnn_peer_wait), and a second flag set ("consumed") lets a single halo buffer
be reused safely.  Summation order is fixed (CSR order within each pass, local before remote), so the
result is deterministic; it differs from the single-GPU order only by fp32 re-association.

Backward (`PartitionedSpmm.backward`, dX = Âᵀ·dY for the own rows): the mirror image — the transposed
remote block turns dY into one partial row per halo slot, the (contiguous) per-owner segments travel
back over the copy engines, and the owner adds them to its local transposed product in fixed
(peer, slot) order through a pattern-only CSR over its send list: ordered summation, no atomics.

Transports: "p2p" (default: fused pack+push kernel, flags), "ce" (local pack, one copy-engine copy per
peer and wave, flags), "nccl" (all_to_all_single of packed rows — the library baseline and the path the
CPU/gloo tests replay).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from itertools import accumulate
from typing import Dict, List, Optional

import torch
import torch.distributed as dist

from . import _lib

# Byte model of the overlap (choose_two_pass_chunks / the automatic schedule), calibrated on r02 measurements
# (papers100M-shaped, F=128 fp32): the all-to-all rate the movers sustain per direction WHILE the SpMM runs
# (2 GPUs 640 GB/s, 8 GPUs 480 GB/s; the exchange alone reaches 575-610), the gather-model rate of the SpMM alone
# (0.87-1.0 of the measured HBM peak), and the cost of one more wave (a flag wait + a short consumer launch).
NVLINK_BPS_BY_WORLD = {2: 640e9, 3: 600e9, 4: 560e9}
NVLINK_BPS_LARGE = 480e9
HBM_BPS = 5.6e12
WAVE_OVERHEAD_S = 0.3e-3
SPMM_EDGES_PER_S = 11.9e9  # F=128 rows, one B200 (1.61 G edges in 135.3 ms)
AUTO_MAX_WAVES = 8
# modelled exchange time / modelled SpMM time above which the step is exchange-bound: the mover then runs on 32 CTAs
# (8 GPUs, random graph, 31.9 GB received per rank: 59.0 ms with 32 mover CTAs, 73.0 with 64, 81.0 with 148 — more
# writers only congest the receivers' ingress; profiles/r02_dist_8gpu.jsonl)
EXCHANGE_BOUND_RATIO = 2.5


def nvlink_bps(world: int) -> float:
    return NVLINK_BPS_BY_WORLD.get(int(world), NVLINK_BPS_LARGE)


def balanced_bounds(rowptr_or_deg_prefix: torch.Tensor, world: int) -> List[int]:
    """Row-block boundaries with (nearly) equal nnz per block.  Input: the global int64 rowptr
    (exclusive prefix sum of degrees, length N+1)."""
    rp = rowptr_or_deg_prefix
    n = rp.numel() - 1
    total = int(rp[-1].item())
    targets = torch.tensor([total * p // world for p in range(1, world)], dtype=rp.dtype, device=rp.device)
    cuts = torch.searchsorted(rp, targets).clamp_(0, n).tolist() if world > 1 else []
    bounds = [0] + [int(c) for c in cuts] + [n]
    for i in range(1, len(bounds)):
        bounds[i] = max(bounds[i], bounds[i - 1])
    return bounds


def split_columns(rowptr, col, val, lo: int, hi: int):
    """Split one row block's CSR by column ownership.  Order within a row is preserved."""
    is_loc = (col >= lo) & (col < hi)
    csum = torch.zeros(col.numel() + 1, dtype=torch.int64, device=col.device)
    torch.cumsum(is_loc.to(torch.int64), 0, out=csum[1:])
    rowptr_loc = csum[rowptr]
    rowptr_rem = rowptr - rowptr_loc
    col_loc = (col[is_loc] - lo).to(torch.int32)
    rem = ~is_loc
    col_rem_global = col[rem]
    val_loc = None if val is None else val[is_loc]
    val_rem = None if val is None else val[rem]
    return rowptr_loc, col_loc, val_loc, rowptr_rem, col_rem_global, val_rem


def _offsets(counts) -> List[int]:
    """Exclusive prefix sum of `counts`, with the total appended."""
    return list(accumulate(counts, initial=0))


def _local_index(idx: torch.Tensor, lo: int, hi: int) -> torch.Tensor:
    """The ids of `idx` in [lo, hi) as row indices local to that block (ascending where idx is)."""
    idx = idx.to(torch.int64)
    return idx[(idx >= lo) & (idx < hi)] - lo


def select_rows(rowptr: torch.Tensor, col: torch.Tensor, val: Optional[torch.Tensor], rows: torch.Tensor):
    """Compact CSR over the (ascending) row subset `rows`: (rowptr', col', val')."""
    deg = rowptr[rows + 1] - rowptr[rows]
    new_rowptr = torch.zeros(rows.numel() + 1, dtype=torch.int64, device=rowptr.device)
    torch.cumsum(deg, 0, out=new_rowptr[1:])
    total = int(new_rowptr[-1].item()) if rows.numel() else 0
    shift = torch.repeat_interleave(rowptr[rows] - new_rowptr[:-1], deg, output_size=total)
    idx = torch.arange(total, dtype=torch.int64, device=rowptr.device) + shift
    return new_rowptr, col[idx], None if val is None else val[idx]


@dataclass
class Consumer:
    """One SpMM launch of the step: a compact CSR over a row subset of the rank's block.
    mode "local": columns index X_local.  "remote": columns index the halo, accumulate into Y.
    "combined": columns < n_local index X_local, the others (col - n_local) the halo; overwrite.
    With a bias/ReLU epilogue every row gets it in the launch that adds its last contribution: compact rows
    [0, epilogue_skip) of P1 are the first pass of two-pass rows and get it later, in their "remote" pass."""
    mode: str
    rowptr: torch.Tensor
    col: torch.Tensor
    val: Optional[torch.Tensor]
    row_map: Optional[torch.Tensor]   # int32 compact row -> local row; None = every local row in order
    n_cols: int
    epilogue_skip: int = 0

    @property
    def n_rows(self) -> int:
        return int(self.rowptr.numel()) - 1

    @property
    def nnz(self) -> int:
        return int(self.col.numel())


@dataclass
class HaloPlan:
    rank: int
    world: int
    bounds: List[int]
    waves: int
    two_pass_chunks: int
    chunk_bounds: List[int]       # local row boundaries of the K row chunks
    # base local / remote split over ALL rows (the backward and the world == 1 path use it)
    rowptr_loc: torch.Tensor
    col_loc: torch.Tensor
    val_loc: Optional[torch.Tensor]
    rowptr_rem: torch.Tensor
    col_rem: torch.Tensor
    val_rem: Optional[torch.Tensor]
    halo_ids: torch.Tensor        # global column id of every halo slot, ordered by (owner, wave, id)
    recv_counts: List[int]        # halo rows per owner q
    recv_wave_counts: List[List[int]]   # [q][w]
    send_rows: torch.Tensor       # int32 local row indices this rank must send, grouped by requester, in the
    send_counts: List[int]        # requester's slot order (wave, id)
    send_wave_counts: List[List[int]]   # [p][w]
    dst_off: List[int]            # where, in requester p's halo, this rank's segment starts
    back_off: List[int]           # where, in owner q's send list, the segment requested by this rank starts
    p1: Optional[Consumer] = None
    p2: List[Optional[Consumer]] = field(default_factory=list)
    model: Dict[str, float] = field(default_factory=dict)

    @property
    def n_local(self) -> int:
        return self.bounds[self.rank + 1] - self.bounds[self.rank]

    @property
    def n_halo(self) -> int:
        return int(self.halo_ids.numel())

    def send_off(self) -> List[int]:
        return _offsets(self.send_counts)

    def recv_off(self) -> List[int]:
        return _offsets(self.recv_counts)


def choose_two_pass_chunks(K: int, F: int, elem: int, nnz_p1_base: int, rows_interior: int, m_rows, m_nnz_loc, m_nnz_rem,
                           wave_bytes, world: int = 2) -> (int, Dict[str, float]):
    """Byte model of the overlap: for every c0 in [0, K] simulate the main stream (P1, then the wave
    consumers, each gated by its wave's arrival; the SpMM runs slower while the exchange shares the HBM)
    and return the c0 with the earliest finish.  All quantities are this rank's own."""
    row_b, edge_b = F * elem, 8 + F * elem
    arrival, t = [], 0.0
    link = nvlink_bps(world)
    for w in range(K):
        t += wave_bytes[w] / link
        arrival.append(t)
    t_x = arrival[-1] if K else 0.0
    slow = max(HBM_BPS - 2 * link, 0.3 * HBM_BPS)  # exchange reads X here and lands the peers' rows here

    def run(t0, nbytes):
        if t0 >= t_x:
            return t0 + nbytes / HBM_BPS
        dt = nbytes / slow
        if t0 + dt <= t_x:
            return t0 + dt
        done = (t_x - t0) * slow
        return t_x + (nbytes - done) / HBM_BPS

    best, report = None, {}
    for c0 in range(K + 1):
        p1_rows = rows_interior + sum(m_rows[:c0])
        p1_nnz = nnz_p1_base + sum(m_nnz_loc[:c0])
        t = run(0.0, p1_nnz * edge_b + p1_rows * row_b)
        for w in range(K):
            t = max(t, arrival[w]) + WAVE_OVERHEAD_S
            if w < c0:
                t = run(t, m_nnz_rem[w] * edge_b + m_rows[w] * 2 * row_b)
            else:
                t = run(t, (m_nnz_loc[w] + m_nnz_rem[w]) * edge_b + m_rows[w] * row_b)
        report[f"c0={c0}"] = t * 1e3
        if best is None or t < best[1] - 1e-9:
            best = (c0, t)
    report["exchange_ms"] = t_x * 1e3
    nnz_all = nnz_p1_base + sum(m_nnz_loc) + sum(m_nnz_rem)
    # the whole block as one single-pass SpMM: gather-model bytes at the HBM rate, never faster than the kernel's
    # edge rate (bf16 rows halve the bytes, not the time: 137.9 ms vs 135.3 ms on one GPU)
    report["compute_ms"] = max((nnz_all * edge_b + (rows_interior + sum(m_rows)) * row_b) / HBM_BPS,
                               nnz_all / SPMM_EDGES_PER_S) * 1e3
    return best[0], report


def _chunk_stats(chunk_bounds: List[int], rowptr_loc: torch.Tensor, rem_deg: torch.Tensor):
    """The MIXED rows (rows with a remote column) of every row chunk: ([row count], [their local nnz], [their remote
    nnz]), lists over the chunks; and the INTERIOR rows of the whole block: (row count, nnz)."""
    loc_deg = rowptr_loc[1:] - rowptr_loc[:-1]
    mixed = rem_deg > 0
    m_rows, m_loc, m_rem = [], [], []
    for a, b in zip(chunk_bounds[:-1], chunk_bounds[1:]):
        mw = mixed[a:b]
        m_rows.append(int(mw.sum().item()))
        m_loc.append(int(loc_deg[a:b][mw].sum().item()))
        m_rem.append(int(rem_deg[a:b].sum().item()))
    return (m_rows, m_loc, m_rem), (rem_deg.numel() - sum(m_rows), int(loc_deg.sum().item()) - sum(m_loc))


def _coarsen(per_chunk: List[int], K: int) -> List[int]:
    """Per-chunk sums at K chunks from the sums at a multiple of K chunks cut by `balanced_bounds` (the cuts for K
    are every (len/K)-th cut of the finer ones: total*k//K == total*(k*g)//(K*g))."""
    g = len(per_chunk) // K
    return [sum(per_chunk[w * g:(w + 1) * g]) for w in range(K)]


def _first_chunk(chunk_bounds: List[int], rem_deg: torch.Tensor, inverse: torch.Tensor, n_uniq: int) -> torch.Tensor:
    """For every distinct remote column (`inverse` maps each remote entry, in CSR order, to its index among the
    n_uniq), the first row chunk that reads it."""
    K, dev = len(chunk_bounds) - 1, rem_deg.device
    if K == 1 or n_uniq == 0:
        return torch.zeros(n_uniq, dtype=torch.int64, device=dev)
    row_of_rem = torch.repeat_interleave(torch.arange(rem_deg.numel(), dtype=torch.int64, device=dev), rem_deg,
                                         output_size=int(inverse.numel()))
    chunk_of_rem = torch.bucketize(row_of_rem, torch.tensor(chunk_bounds[1:-1], dtype=torch.int64, device=dev),
                                   right=True)
    del row_of_rem
    first = torch.full((n_uniq,), K, dtype=torch.int64, device=dev)
    first.scatter_reduce_(0, inverse, chunk_of_rem, reduce="amin", include_self=True)
    return first


def _combined_columns(plan: "HaloPlan", col: torch.Tensor) -> torch.Tensor:
    """The int32 column ids of the block `plan` was built from (GLOBAL ids `col`) in the COMBINED column space:
    local column c -> c - lo, remote column -> n_local + its halo slot."""
    lo, hi = plan.bounds[plan.rank], plan.bounds[plan.rank + 1]
    col64 = col.to(torch.int64)
    is_loc = (col64 >= lo) & (col64 < hi)
    del col64
    comb = torch.empty(col.numel(), dtype=torch.int32, device=col.device)
    comb[is_loc] = plan.col_loc.to(col.device)
    comb[~is_loc] = plan.col_rem.to(col.device) + (hi - lo)
    return comb


def _auto_schedule(per_chunk, interior, first_chunk, world, group, F, elem_size):
    """(K, c0) for all ranks from this rank's statistics at the finest wave count (`_chunk_stats` and `_first_chunk`
    at AUTO_MAX_WAVES chunks), coarsened for the smaller K, and one all_reduce of the modelled step times."""
    KM = AUTO_MAX_WAVES
    rows_interior, nnz_interior = interior
    wave_rows = torch.bincount(first_chunk, minlength=KM).tolist()[:KM]  # halo rows per finest wave
    ks = [k for k in (1, 2, 4, 8) if k <= KM]
    times = torch.full((len(ks), KM + 1), 1e9, dtype=torch.float64, device=first_chunk.device)
    for ki, K in enumerate(ks):
        m_rows, m_loc, m_rem = (_coarsen(v, K) for v in per_chunk)
        _, rep_k = choose_two_pass_chunks(K, F, elem_size, nnz_interior, rows_interior, m_rows, m_loc, m_rem,
                                          [r * F * elem_size for r in _coarsen(wave_rows, K)], world)
        for c0 in range(K + 1):
            times[ki, c0] = rep_k[f"c0={c0}"]
    dist.all_reduce(times, group=group)
    best = int(torch.argmin(times).item())
    K, c0 = ks[best // (KM + 1)], best % (KM + 1)
    report = {f"K={ks[i]}": [round(float(x), 2) for x in times[i, :ks[i] + 1].tolist()] for i in range(len(ks))}
    return K, c0, report


def build_halo_plan(rowptr: torch.Tensor, col: torch.Tensor, val: Optional[torch.Tensor], bounds: List[int],
                    rank: int, world: int, group=None, waves: Optional[int] = 1,
                    two_pass_chunks: Optional[int] = None, F: int = 128, elem_size: int = 4,
                    consumers: bool = True) -> HaloPlan:
    """Plan for this rank's row block (rowptr over its own rows, GLOBAL column ids).
    Collective: every rank of `group` must call it with the same `waves` (exchanges the request lists).
    waves: number of row chunks / exchange waves K; None = AUTOMATIC: the byte model is evaluated for
      K in {1, 2, 4, 8} and every two-pass count on every rank, the modelled times are summed over the ranks
      and the (K, c0) with the smallest sum is used by all of them.
    two_pass_chunks: c0 in [0, waves] (None: chosen by `choose_two_pass_chunks` for feature width F)."""
    dev = col.device
    lo, hi = bounds[rank], bounds[rank + 1]
    n_loc = hi - lo
    col = col.to(torch.int64)
    rowptr_loc, col_loc, val_loc, rowptr_rem, col_rem_g, val_rem = split_columns(rowptr, col, val, lo, hi)
    rem_deg = rowptr_rem[1:] - rowptr_rem[:-1]
    uniq, inverse = torch.unique(col_rem_g, sorted=True, return_inverse=True)  # de-duplicated halo
    stats = None  # _chunk_stats at the plan's K, once known
    if waves is None and world > 1:
        cuts = balanced_bounds(rowptr, AUTO_MAX_WAVES)
        per_chunk, interior = _chunk_stats(cuts, rowptr_loc, rem_deg)
        first = _first_chunk(cuts, rem_deg, inverse, uniq.numel())
        K, two_pass_chunks, auto_report = _auto_schedule(per_chunk, interior, first, world, group, F, elem_size)
        g = AUTO_MAX_WAVES // K
        chunk_bounds, first_wave = cuts[::g], first // g
        stats = [_coarsen(v, K) for v in per_chunk], interior
        del first
    else:
        auto_report = None
        K = max(int(waves or 1), 1) if world > 1 else 1
        chunk_bounds = balanced_bounds(rowptr, K)  # K row chunks of (nearly) equal nnz
        first_wave = _first_chunk(chunk_bounds, rem_deg, inverse, uniq.numel())
    edges = torch.tensor(bounds[1:-1], dtype=torch.int64, device=dev)
    owner = torch.bucketize(uniq, edges, right=True) if world > 1 else torch.zeros_like(uniq)
    key = owner * K + first_wave
    order = torch.argsort(key, stable=True)  # uniq is ascending: ties keep id order
    slot_of_uniq = torch.empty_like(order)
    slot_of_uniq[order] = torch.arange(order.numel(), dtype=torch.int64, device=dev)
    halo_ids = uniq[order]
    col_rem = slot_of_uniq[inverse].to(torch.int32)
    counts2d = (torch.bincount(key, minlength=world * K) if uniq.numel() else
                torch.zeros(world * K, dtype=torch.int64, device=dev)).view(world, K)
    recv_wave_counts = [[int(x) for x in r] for r in counts2d.tolist()]
    recv_counts = [sum(r) for r in recv_wave_counts]
    recv_off = _offsets(recv_counts)
    plan_kw = dict(rank=rank, world=world, bounds=bounds, waves=K, chunk_bounds=chunk_bounds, rowptr_loc=rowptr_loc,
                   col_loc=col_loc, val_loc=val_loc, rowptr_rem=rowptr_rem, col_rem=col_rem, val_rem=val_rem,
                   halo_ids=halo_ids, recv_counts=recv_counts, recv_wave_counts=recv_wave_counts)
    if world == 1:
        return HaloPlan(two_pass_chunks=1, send_rows=torch.zeros(0, dtype=torch.int32, device=dev), send_counts=[0],
                        send_wave_counts=[[0]], dst_off=[0], back_off=[0], **plan_kw)
    # tell every owner where its segment starts in our halo and how many rows of each wave we want
    meta_out = torch.tensor([[recv_off[q]] + recv_wave_counts[q] for q in range(world)], dtype=torch.int64, device=dev)
    meta_in = torch.empty_like(meta_out)
    dist.all_to_all_single(meta_in, meta_out, group=group)
    dst_off = [int(x) for x in meta_in[:, 0].tolist()]
    send_wave_counts = [[int(x) for x in r] for r in meta_in[:, 1:].tolist()]
    send_counts = [sum(r) for r in send_wave_counts]
    # the requested ids, as row indices local to their owner, in our slot order
    bounds_t = torch.tensor(bounds, dtype=torch.int64, device=dev)
    req_out = (halo_ids - bounds_t[owner[order]]).contiguous()
    req_in = torch.empty(int(sum(send_counts)), dtype=torch.int64, device=dev)
    dist.all_to_all_single(req_in, req_out, output_split_sizes=send_counts, input_split_sizes=recv_counts, group=group)
    # backward: owner q tells requester p where p's segment starts in q's send list
    so_out = torch.tensor(_offsets(send_counts)[:world], dtype=torch.int64, device=dev)
    so_in = torch.empty_like(so_out)
    dist.all_to_all_single(so_in, so_out, group=group)
    plan = HaloPlan(two_pass_chunks=K, send_rows=req_in.to(torch.int32), send_counts=send_counts,
                    send_wave_counts=send_wave_counts, dst_off=dst_off, back_off=[int(x) for x in so_in.tolist()],
                    **plan_kw)
    if not consumers:
        return plan
    # ---- row classes and the consumers of the step --------------------------------------------
    if stats is None:
        stats = _chunk_stats(chunk_bounds, rowptr_loc, rem_deg)
    (m_rows, m_nnz_loc, m_nnz_rem), (rows_interior, nnz_interior) = stats
    row_b = F * elem_size
    wave_bytes = [max(sum(recv_wave_counts[q][w] for q in range(world)), sum(send_wave_counts[p][w] for p in range(world)))
                  * row_b for w in range(K)]
    c0_model, report = choose_two_pass_chunks(K, F, elem_size, nnz_interior, rows_interior, m_rows, m_nnz_loc,
                                              m_nnz_rem, wave_bytes, world)
    if auto_report is not None:
        report["auto_schedule_ms_sum_over_ranks"] = auto_report
    c0 = c0_model if two_pass_chunks is None else max(0, min(int(two_pass_chunks), K))
    # exchange-bound steps (the modelled exchange outlasts the whole SpMM several times over): nothing is left to hide
    # behind the exchange, so every chunk is single-pass — the consumers park on their wave's flag and Y is written
    # once.  8 GPUs, random graph: c0 = 0 / 4 / 8 -> 60.2 / 71.4 / 65.6 ms at 32 mover CTAs (r02, r2i_rand).
    exchange_bound = world > 1 and report["exchange_ms"] >= EXCHANGE_BOUND_RATIO * max(report["compute_ms"], 1e-9)
    report["exchange_bound"] = bool(exchange_bound)
    if exchange_bound and (two_pass_chunks is None or auto_report is not None):
        c0 = 0
    plan.two_pass_chunks = c0
    plan.model = dict(report, chosen=c0, model_choice=c0_model, rows_interior=rows_interior,
                      rows_mixed=sum(m_rows), nnz_interior=nnz_interior)
    cut_row = chunk_bounds[c0]  # mixed rows at or beyond this row are single-pass
    mixed = rem_deg > 0
    all_rows = torch.arange(n_loc, dtype=torch.int64, device=dev)
    # P1: local columns of every row except the single-pass mixed rows.  The two-pass mixed rows come first (their
    # remote pass adds the rest, so a fused epilogue skips them: Consumer.epilogue_skip), then the interior rows.
    # Every row is its own ordered reduction, so the order of the rows changes no result.
    first = all_rows[mixed & (all_rows < cut_row)]
    interior = all_rows[~mixed]
    n_first = int(first.numel())
    if n_first + int(interior.numel()) == n_loc and (n_first == 0 or n_first == n_loc):
        plan.p1 = Consumer("local", rowptr_loc, col_loc, val_loc, None, n_loc, epilogue_skip=n_first)
    else:
        rows = torch.cat([first, interior])
        rp, cc, vv = select_rows(rowptr_loc, col_loc, val_loc, rows)
        plan.p1 = (Consumer("local", rp, cc, vv, rows.to(torch.int32), n_loc, epilogue_skip=n_first)
                   if rows.numel() else None)
    col_comb = _combined_columns(plan, col) if c0 < K else None  # the column space of the single-pass rows
    plan.p2 = []
    for w in range(K):
        a, b = chunk_bounds[w], chunk_bounds[w + 1]
        rows = all_rows[a:b][mixed[a:b]]
        if rows.numel() == 0:
            plan.p2.append(None)
        elif w < c0:
            rp, cc, vv = select_rows(rowptr_rem, col_rem, val_rem, rows)
            plan.p2.append(Consumer("remote", rp, cc, vv, rows.to(torch.int32), max(plan.n_halo, 1)))
        else:
            rp, cc, vv = select_rows(rowptr, col_comb, val, rows)
            plan.p2.append(Consumer("combined", rp, cc, vv, rows.to(torch.int32), n_loc + max(plan.n_halo, 1)))
    return plan


@dataclass
class AttentionView:
    """This rank's row block in the COMBINED column space of `build_halo_plan`: local column c -> c - lo, remote
    column -> n_local + its halo slot.  The columns address Wh_comb = [Wh_local ; Wh_halo] (functional.halo_exchange),
    and every row keeps the edge order of the global CSR, so a fused attention row over it is the same ordered
    reduction as over the whole graph.  edge_slot_base = the block's first global edge slot (global rowptr[lo]): the
    seeded attention dropout of local slot e is the one of global slot e + edge_slot_base."""
    rowptr: torch.Tensor
    col: torch.Tensor             # int32 combined column ids
    n_rows: int
    n_cols: int                   # n_local + n_halo
    edge_slot_base: int
    any_empty_row: bool           # some row of the GLOBAL graph (any rank's block) has no edge

    def require_edges(self):
        """GAT's rule for a row without edges is the mean of ALL N rows of Wh (GAT/models/layers.py:28-30), which the
        partitioned layer does not compute.  The flag is global, so every rank raises together."""
        if self.any_empty_row:
            raise _lib.GnnError("GAT on a PartitionedGraph: the graph has rows without edges (their output is the mean "
                                "over all nodes, not supported across ranks); add self-loops")


def build_attention_view(plan: HaloPlan, rowptr: torch.Tensor, col: torch.Tensor, group=None) -> AttentionView:
    """The attention view of the block `plan` was built from (rowptr over the rank's rows, GLOBAL column ids).
    Collective when world > 1: one all_gather of (nnz, has-empty-row) per rank gives the exclusive scan of the
    ranks' nnz and the global empty-row flag."""
    n_loc = plan.n_local
    col_comb = _combined_columns(plan, col)
    empty = bool((rowptr[1:] == rowptr[:-1]).any().item()) if n_loc > 0 else False
    base, any_empty = 0, empty
    if plan.world > 1:
        mine = torch.tensor([col.numel(), int(empty)], dtype=torch.int64, device=col.device)
        parts = [torch.empty_like(mine) for _ in range(plan.world)]
        dist.all_gather(parts, mine, group=group)
        base = sum(int(p[0].item()) for p in parts[:plan.rank])
        any_empty = any(int(p[1].item()) for p in parts)
    return AttentionView(rowptr, col_comb, n_loc, n_loc + plan.n_halo, base, any_empty)


def reference_step_cpu(plan: HaloPlan, X_local: torch.Tensor, halo: torch.Tensor, bias: Optional[torch.Tensor] = None,
                       relu: bool = False) -> torch.Tensor:
    """The step's arithmetic with torch ops in float64 (test-side: replays P1 and the wave consumers of a
    plan exactly as `PartitionedSpmm.forward` schedules them).  `halo` = the received rows in slot order.
    bias / relu: the fused epilogue, applied where the schedule applies it (P1 rows past its epilogue_skip,
    after the add of a "remote" pass, on every "combined" row)."""
    n_loc, F = plan.n_local, X_local.shape[1]
    Y = torch.zeros((n_loc, F), dtype=torch.float64)
    Xl, Hl = X_local.double(), halo.double()
    table = torch.cat([Xl, Hl], 0)
    b = None if bias is None else bias.double().view(1, -1)

    def epilogue(y):
        y = y if b is None else y + b
        return y.clamp_min(0.0) if relu else y

    def product(c: Consumer, src):
        rows = torch.repeat_interleave(torch.arange(c.n_rows), c.rowptr[1:] - c.rowptr[:-1])
        v = torch.ones(c.nnz, dtype=torch.float64) if c.val is None else c.val.double()
        out = torch.zeros((c.n_rows, F), dtype=torch.float64)
        out.index_add_(0, rows, src[c.col.long()] * v[:, None])
        return out

    def target(c: Consumer):
        return torch.arange(n_loc) if c.row_map is None else c.row_map.long()

    if plan.p1 is not None:
        y, k = product(plan.p1, Xl), plan.p1.epilogue_skip
        y[k:] = epilogue(y[k:])
        Y[target(plan.p1)] = y
    for c in plan.p2:
        if c is None:
            continue
        if c.mode == "remote":
            t = target(c)
            Y[t] = epilogue(Y[t] + product(c, Hl))
        else:
            Y[target(c)] = epilogue(product(c, table))
    return Y


class _RawCudaBuffer:
    """Expose a raw device pointer to torch (zero-copy) through __cuda_array_interface__."""

    def __init__(self, ptr: int, shape, typestr="<f4"):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 3, "strides": None}


class _PeerBuffer:
    """One cudaMalloc allocation of this rank, exported with CUDA IPC and mapped by every peer."""

    def __init__(self, nbytes: int, rank: int, world: int, group):
        lib = _lib.load()
        self.rank, self.world, self.group = rank, world, group
        p = C.c_void_p()
        h = (C.c_ubyte * 64)()
        _lib.check(lib.gnn_peer_alloc(max(int(nbytes), 256), C.byref(p), h), "gnn_peer_alloc")
        self.own = p.value
        gathered = [None] * world
        dist.all_gather_object(gathered, bytes(h), group=group)
        self.ptrs = []
        for q in range(world):
            if q == rank:
                self.ptrs.append(self.own)
            else:
                pq = C.c_void_p()
                hb = (C.c_ubyte * 64).from_buffer_copy(gathered[q])
                _lib.check(lib.gnn_peer_open(hb, C.byref(pq)), "gnn_peer_open")
                self.ptrs.append(pq.value)

    def close(self):
        lib = _lib.load()
        if self.ptrs is None:
            return
        for q, p in enumerate(self.ptrs):
            if q != self.rank:
                lib.gnn_peer_close(p)
        if dist.is_initialized():
            dist.barrier(group=self.group)
        lib.gnn_peer_free(self.own)
        self.ptrs = None


_TORCH_TYPESTR = {torch.float32: "<f4", torch.bfloat16: "<u2"}


def _raw_view(ptr: int, rows: int, ld: int, dtype: torch.dtype, device) -> torch.Tensor:
    """[rows, ld] tensor of `dtype` over the device memory at `ptr` (zero-copy)."""
    t = torch.as_tensor(_RawCudaBuffer(ptr, (rows, ld), _TORCH_TYPESTR[dtype]), device=device)
    return t.view(dtype) if dtype != torch.float32 else t


def _close_peer_buffers(bufs: List[_PeerBuffer], device, group):
    """Free peer buffers (collective): every rank finishes its queued work, which may read a peer's buffer or be read
    from, before any mapping is closed."""
    if bufs:
        torch.cuda.synchronize(device)
        if dist.is_initialized():
            dist.barrier(group=group)
        for b in bufs:
            b.close()


class _PeerFlags:
    """Monotonic flags in peer memory: `n_arrays` arrays of 32 uint32 slots (128 bytes) in one peer buffer per rank,
    slot q of an array written by rank q only.  `signal(a, v)` sets this rank's slot of array a to v on every rank;
    `wait(a, v)` holds `stream` until every peer's slot of this rank's array a has reached v.  Values wrap at 2^32.
    Every wait is bounded by timeout_ms: a lost peer sets the status word (`check_status`) instead of hanging the
    GPU.  Construction is collective."""

    def __init__(self, n_arrays: int, rank: int, world: int, group, device, timeout_ms: int):
        self.rank, self.world, self.timeout_ms = rank, world, int(timeout_ms)
        self.status = torch.zeros(1, dtype=torch.int32, device=device)
        self.buf = _PeerBuffer(n_arrays * 128, rank, world, group)

    def ptrs(self, array: int):
        """Device pointers of flag array `array` on every rank."""
        return (C.c_void_p * self.world)(*[p + array * 128 for p in self.buf.ptrs])

    def signal(self, array: int, value: int, stream):
        _lib.check(_lib.load().gnn_peer_signal(self.ptrs(array), self.world, self.rank, self.rank,
                                               value & 0xFFFFFFFF, stream.cuda_stream), "gnn_peer_signal")

    def wait(self, array: int, value: int, stream):
        _lib.check(_lib.load().gnn_peer_wait(self.buf.own + array * 128, self.world, self.rank, value & 0xFFFFFFFF,
                                             self.status.data_ptr(), self.timeout_ms, stream.cuda_stream),
                   "gnn_peer_wait")

    def check_status(self, what: str):
        """Raise if a wait timed out (synchronises)."""
        s = int(self.status.item())
        if s:
            raise _lib.GnnError(f"rank {self.rank}: timed out waiting for the {what} flag of peer {s - 1}")


class PartitionedSpmm:
    """Executes Y_local = (Â·X)[own rows] (and dX_local = (Âᵀ·dY)[own rows]) for one rank.

    Every scheduling choice is a constructor argument and is passed to the C ABI per call
    (gnn_halo_opts / gnn_spmm_opts): nothing is routed through process-global knobs.
      transport      "p2p" | "ce" | "nccl"
      mover          "tma" | "vector" | "auto"  (p2p only)
      mover_ctas     CTAs of the push kernel (0 = one per SM; -1 = measured default: 4-warp movers on 32 SMs when
                     the step is single-pass / exchange-dominated, on 48 SMs otherwise — r02 sweeps at 2 and 8 GPUs:
                     more mover CTAs take SpMM occupancy without raising the all-to-all rate, fewer starve it)
      mover_warps    warps per push CTA (0 = default: TMA 1, vector 8; -1 = measured default 4)
      dedicated_sms  > 0: vector mover on that many SMs of its own (each CTA claims 200 KB of shared memory
                     and the concurrent P1 asks for 28 KB so that the block scheduler keeps them apart)
      timeout_ms     bound of every flag wait (a lost peer must not hang the GPU)
      interleave     fused-signal mover: > 0 cuts every peer segment of a wave into pieces of that many ring stages
                     and deals the pieces round-robin over the peers, so a sender feeds all its peers at once
                     (uniform ingress load on every receiver); 0 = one peer after the other, rotated by rank
      fused_signal   p2p + TMA mover: all waves of a step in ONE launch, the arrival flags raised from inside
                     the kernel by the last warp that finishes a wave (gnn_halo_push_waves); False = one
                     mover launch + one signal launch per wave
    """

    def __init__(self, plan: HaloPlan, F: int, device, group=None, transport: str = "p2p",
                 dtype: torch.dtype = torch.float32, mover: str = "auto", mover_ctas: int = -1, mover_warps: int = -1,
                 dedicated_sms: int = 0, timeout_ms: int = 20000, fused_signal: bool = True, interleave: int = 0):
        from .graph import CSRGraph
        if dtype not in _TORCH_TYPESTR:
            raise _lib.GnnError(f"PartitionedSpmm: unsupported dtype {dtype}")
        self.plan, self.F, self.dev, self.group, self.dtype = plan, int(F), torch.device(device), group, dtype
        self.elem = 4 if dtype == torch.float32 else 2
        self.transport = transport if plan.world > 1 else "none"
        if self.transport not in ("p2p", "ce", "nccl", "none"):
            raise ValueError(f"unknown transport {transport!r}")
        self.mover = {"auto": 0, "vector": 1, "tma": 2}[mover]
        if int(mover_ctas) < 0:
            mover_ctas = 32 if (plan.two_pass_chunks == 0 or plan.model.get("exchange_bound", False)) else 48
        if int(mover_warps) < 0:
            mover_warps = 4
        self.mover_ctas, self.mover_warps, self.dedicated = int(mover_ctas), int(mover_warps), int(dedicated_sms)
        self.timeout_ms = int(timeout_ms)
        self.interleave = int(interleave)
        n_loc, n_halo = plan.n_local, max(plan.n_halo, 1)
        per16 = 16 // self.elem
        # halo rows are contiguous (ld == F) when a row is a 16-byte multiple: one bulk store per ring stage
        self.ld = self.F if self.F % per16 == 0 else (self.F + per16 - 1) // per16 * per16
        self.A_loc = CSRGraph(plan.rowptr_loc, plan.col_loc, plan.val_loc, n_loc, n_loc)
        self._cons = {}
        self._wave_table = None
        self._t_loc = self._t_rem = self._R = None
        self._fstep = self._bstep = 0
        self._bufs: List[_PeerBuffer] = []
        self._flags: Optional[_PeerFlags] = None
        if plan.world == 1:
            return
        self.comm = torch.cuda.Stream(device=self.dev, priority=-1)  # halo traffic is scheduled first
        self._ev_x = torch.cuda.Event()
        self._ev_halo = torch.cuda.Event()
        self._send_off = plan.send_off()
        self._recv_off = plan.recv_off()
        self._wave_cum_send = [[sum(r[:w]) for w in range(plan.waves + 1)] for r in plan.send_wave_counts]
        if self.transport in ("p2p", "ce"):
            self._halo_buf = _PeerBuffer(n_halo * self.ld * self.elem, plan.rank, plan.world, group)
            # flag arrays 0 arrive_fwd, 1 consumed_fwd, 2 arrive_bwd, 3 consumed_bwd
            self._flags = _PeerFlags(4, plan.rank, plan.world, group, self.dev, self.timeout_ms)
            self._bufs += [self._halo_buf, self._flags.buf]
            self.halo = _raw_view(self._halo_buf.own, n_halo, self.ld, dtype, self.dev)[:, :self.F]
            R = _lib.load().gnn_halo_rows_per_stage(self.F * self.elem)
            if (self.transport == "p2p" and fused_signal and self.mover != 1 and self.dedicated == 0 and R > 0
                    and self.ld == self.F):
                self._wave_table = self._build_wave_table(R)
            if self.transport == "ce":
                self._sendbuf = torch.empty((max(self._send_off[-1], 1), self.ld), dtype=dtype, device=self.dev)
                self._copy_streams = [torch.cuda.Stream(device=self.dev, priority=-1) for _ in range(4)]
                self._ev_packed = torch.cuda.Event()
                self._ev_copied = [torch.cuda.Event() for _ in range(4)]
        else:
            self.halo = torch.empty((n_halo, self.F), dtype=dtype, device=self.dev)
            self._sendbuf = torch.empty((max(int(plan.send_rows.numel()), 1), self.F), dtype=dtype, device=self.dev)
        self.halo_bytes_received = plan.n_halo * self.F * self.elem

    def _build_wave_table(self, R: int):
        """Device segment table of gnn_halo_push_waves: segments sorted by wave, peers in rotated order."""
        plan, W = self.plan, self.plan.world
        row_bytes = self.ld * self.elem
        rows, chunk = [], 0
        piece = self.interleave * R  # rows per interleaved piece (0: whole segments, one peer after the other)
        for w in range(plan.waves):
            segs = []
            for s_i in range(1, W):
                q = (plan.rank + s_i) % W
                n = plan.send_wave_counts[q][w]
                if n:
                    b = self._wave_cum_send[q][w]
                    segs.append((self._send_off[q] + b, n, self._halo_buf.ptrs[q] + (plan.dst_off[q] + b) * row_bytes))
            if piece > 0:
                pieces, k = [], 0
                while any(k * piece < n for _, n, _ in segs):
                    for src, n, dst in segs:  # round-robin over the peers, rotated order kept within a round
                        if k * piece < n:
                            m = min(piece, n - k * piece)
                            pieces.append((src + k * piece, m, dst + k * piece * row_bytes))
                    k += 1
                segs = pieces
            for src, n, dst in segs:
                rows.append([src, n, dst, chunk, w])
                chunk += (n + R - 1) // R
        table = torch.tensor(rows if rows else [[0, 0, 0, 0, 0]], dtype=torch.int64, device=self.dev)
        done = torch.zeros(max(plan.waves, 1), dtype=torch.int32, device=self.dev)
        return table, len(rows), chunk, done

    # -- helpers ---------------------------------------------------------------------------
    def check_status(self):
        """Raise if a flag wait of an earlier step timed out (synchronises)."""
        if self._flags is not None:
            self._flags.check_status("halo")

    def _graph(self, c: Consumer):
        from .graph import CSRGraph
        g = self._cons.get(id(c))
        if g is None:
            g = CSRGraph(c.rowptr.to(self.dev), c.col.to(self.dev), None if c.val is None else c.val.to(self.dev),
                         c.n_rows, c.n_cols)
            g._row_map = None if c.row_map is None else c.row_map.to(self.dev).contiguous()
            self._cons[id(c)] = g
        return g

    def _push(self, X: torch.Tensor, peer_ptrs, seg_begin, seg_rows, dst_row, ld_dst, send_rows, stream,
              force_vector_shared: bool = False):
        plan, lib = self.plan, _lib.load()
        W = plan.world
        o = _lib.HaloOpts()
        o.struct_size = C.sizeof(_lib.HaloOpts)
        o.first_peer = (plan.rank + 1) % W
        if force_vector_shared:
            o.mover, o.ctas, o.warps_per_cta = 1, 0, 8
        elif self.dedicated > 0:
            o.mover, o.ctas, o.warps_per_cta, o.claim_smem_bytes = 1, self.dedicated, 32, 200 * 1024
        else:
            o.mover, o.ctas, o.warps_per_cta = self.mover, self.mover_ctas, self.mover_warps
        _lib.check(lib.gnn_halo_push(X.data_ptr(), X.stride(0), self.F, self.elem,
                                     None if send_rows is None else send_rows.data_ptr(),
                                     (C.c_int64 * W)(*seg_begin), (C.c_int64 * W)(*seg_rows),
                                     (C.c_void_p * W)(*peer_ptrs), (C.c_int64 * W)(*dst_row), ld_dst, W, C.byref(o),
                                     stream.cuda_stream), "gnn_halo_push")

    # -- forward ---------------------------------------------------------------------------
    def _exchange_wave(self, X: torch.Tensor, w: int, stream):
        """Push wave w of every peer's segment (p2p) / copy it (ce) on `stream`."""
        plan = self.plan
        W = plan.world
        seg_begin = [self._send_off[p] + self._wave_cum_send[p][w] for p in range(W)]
        seg_rows = [plan.send_wave_counts[p][w] for p in range(W)]
        dst_row = [plan.dst_off[p] + self._wave_cum_send[p][w] for p in range(W)]
        if self.transport == "p2p":
            self._push(X, self._halo_buf.ptrs, seg_begin, seg_rows, dst_row, self.ld, plan.send_rows, stream)
            return
        self._ev_packed.record(stream)
        self._copy_to_peers(self._copy_streams, self._ev_copied, self._ev_packed, stream, self._halo_buf.ptrs, dst_row,
                            self._sendbuf.data_ptr(), seg_begin, seg_rows)

    def _copy_to_peers(self, streams, done, ready, join, dst_ptrs, dst_row, src, src_row, rows, wait_join=False):
        """One gnn_peer_copy_async of rows[q] rows (src row src_row[q] -> row dst_row[q] of dst_ptrs[q]) per peer q
        with rows to send, in rotated order (rank r copies to r+1 first), dealt over the copy `streams`; each stream
        first waits on the event `ready` (and on the stream `join` too with wait_join).  Then `join` waits on every
        stream through the events `done`."""
        plan, lib = self.plan, _lib.load()
        W, row_bytes = plan.world, self.ld * self.elem
        for s_i in range(1, W):
            q = (plan.rank + s_i) % W
            if rows[q] == 0:
                continue
            st = streams[s_i % len(streams)]
            st.wait_event(ready)
            if wait_join:
                st.wait_stream(join)
            _lib.check(lib.gnn_peer_copy_async(dst_ptrs[q] + dst_row[q] * row_bytes, src + src_row[q] * row_bytes,
                                               rows[q] * row_bytes, st.cuda_stream), "gnn_peer_copy_async")
        for ev, st in zip(done, streams):
            ev.record(st)
            join.wait_event(ev)

    def _exchange(self, X: torch.Tensor, stream):
        """Whole exchange of one step on `stream` (waves in order, flags after every wave)."""
        plan = self.plan
        K, s = plan.waves, self._fstep
        if self.transport == "nccl":
            n_send = int(plan.send_rows.numel())
            torch.index_select(X, 0, plan.send_rows.to(torch.int64), out=self._sendbuf[:n_send])
            dist.all_to_all_single(self.halo[:plan.n_halo], self._sendbuf[:n_send],
                                   output_split_sizes=plan.recv_counts, input_split_sizes=plan.send_counts,
                                   group=self.group)
            return
        if s > 0:
            self._flags.wait(1, s, stream)  # every peer has consumed the halo of the previous step: safe to overwrite
        if self.transport == "ce":
            # pack: the push kernel with this rank's own send buffer as every "peer" (rows land in send order)
            W = plan.world
            self._push(X, [self._sendbuf.data_ptr()] * W, self._send_off[:W], plan.send_counts, self._send_off[:W],
                       self.ld, plan.send_rows, stream, force_vector_shared=True)
        if self._wave_table is not None:
            table, n_segs, n_chunks, done = self._wave_table
            o = _lib.HaloOpts()
            o.struct_size = C.sizeof(_lib.HaloOpts)
            o.ctas, o.warps_per_cta = self.mover_ctas, self.mover_warps
            _lib.check(_lib.load().gnn_halo_push_waves(
                X.data_ptr(), X.stride(0), self.F, self.elem, plan.send_rows.data_ptr(), table.data_ptr(), n_segs, K,
                n_chunks, done.data_ptr(), self._flags.ptrs(0), plan.world, plan.rank, (s * K) & 0xFFFFFFFF,
                C.byref(o), stream.cuda_stream), "gnn_halo_push_waves")
            return
        for w in range(K):
            self._exchange_wave(X, w, stream)
            self._flags.signal(0, s * K + w + 1, stream)

    def _run(self, c: Consumer, X, halo, out, excl: int = 0, bias: Optional[torch.Tensor] = None, relu: bool = False):
        from .functional import spmm_ex
        g = self._graph(c)
        if c.mode == "local":
            spmm_ex(g, X, out, row_map=g._row_map, exclusion_smem=excl, bias=bias, relu=relu,
                    epilogue_skip_prefix=c.epilogue_skip if (bias is not None or relu) else 0)
        elif c.mode == "remote":
            spmm_ex(g, halo, out, row_map=g._row_map, accumulate=True, bias=bias, relu=relu)
        else:
            spmm_ex(g, X, out, row_map=g._row_map, X2=halo, split=self.plan.n_local, bias=bias, relu=relu)

    def _exchange_begin(self, X: torch.Tensor, overlap: bool):
        """Start the exchange of this step: on the comm stream once X is ready (overlap) or on the main stream."""
        main = torch.cuda.current_stream()
        comm = self.comm if overlap else main
        if overlap:
            self._ev_x.record(main)
            self.comm.wait_event(self._ev_x)  # X is ready (and everything earlier on the main stream is done)
            X.record_stream(self.comm)  # the movers read X after the main stream is done with it
        with torch.cuda.stream(comm):
            self._exchange(X, comm)
            if self.transport not in ("p2p", "ce"):
                self._ev_halo.record(comm)

    def _exchange_wait(self, w: int, stream):
        """The halo rows of wave w are readable on `stream` (flags: per wave; nccl: the whole halo, at wave 0)."""
        if self.transport in ("p2p", "ce"):
            self._flags.wait(0, self._fstep * self.plan.waves + w + 1, stream)
        elif w == 0:
            stream.wait_event(self._ev_halo)

    def _exchange_end(self, stream):
        """This rank is done reading its halo: the peers may overwrite it in the next step."""
        if self.transport in ("p2p", "ce"):
            self._flags.signal(1, self._fstep + 1, stream)
        self._fstep += 1

    def forward(self, X: torch.Tensor, out: Optional[torch.Tensor] = None, overlap: bool = True,
                bias: Optional[torch.Tensor] = None, relu: bool = False) -> torch.Tensor:
        """Y_local = relu?((Â·X)[own rows] + bias).  bias (fp32 [F], nullable) / relu: the GCN epilogue, fused into
        the launch that writes each row's last contribution (no extra pass over Y).  Collective: every rank of the
        group runs the same sequence of forward / backward calls (the arrival flags count steps)."""
        from .functional import spmm_raw
        plan = self.plan
        assert X.shape == (plan.n_local, self.F) and X.dtype == self.dtype and X.is_cuda
        main = torch.cuda.current_stream()
        if out is None:
            out = torch.empty((plan.n_local, self.F), dtype=self.dtype, device=self.dev)
        if plan.world == 1:
            return spmm_raw(self.A_loc, X, out=out, bias=bias, relu=relu)
        self._exchange_begin(X, overlap)
        excl = 28 * 1024 if (self.transport == "p2p" and self.dedicated > 0 and overlap) else 0
        if plan.p1 is not None:
            self._run(plan.p1, X, self.halo, out, excl, bias, relu)
        for w in range(plan.waves):
            self._exchange_wait(w, main)
            if plan.p2[w] is not None:
                self._run(plan.p2[w], X, self.halo, out, 0, bias, relu)
        self._exchange_end(main)
        return out

    def gather_halo(self, X: torch.Tensor) -> torch.Tensor:
        """X_comb = [X ; halo] ([n_local + n_halo, F]): the exchange of one step (waves, flags, transport as in
        `forward`), then a private copy of the received rows in slot order.  Collective, like `forward`."""
        plan = self.plan
        assert X.shape == (plan.n_local, self.F) and X.dtype == self.dtype and X.is_cuda
        out = torch.empty((plan.n_local + plan.n_halo, self.F), dtype=self.dtype, device=self.dev)
        if plan.world > 1:
            main = torch.cuda.current_stream()
            self._exchange_begin(X, True)
        out[:plan.n_local].copy_(X)
        if plan.world == 1:
            return out
        for w in range(plan.waves):
            self._exchange_wait(w, main)
        out[plan.n_local:].copy_(self.halo[:plan.n_halo])
        self._exchange_end(main)
        return out

    def exchange_only(self, X: torch.Tensor):
        """One halo exchange with no aggregation (measurement: the transport alone), flag protocol kept."""
        plan = self.plan
        if plan.world == 1:
            return
        main = torch.cuda.current_stream()
        K, s = plan.waves, self._fstep
        self._exchange(X, main)
        if self.transport in ("p2p", "ce"):
            self._flags.wait(0, s * K + K, main)
            self._flags.signal(1, s + 1, main)
        self._fstep += 1

    # -- backward --------------------------------------------------------------------------
    def _backward_setup(self):
        from .graph import CSRGraph
        plan = self.plan
        n_loc, n_halo = plan.n_local, max(plan.n_halo, 1)
        self._t_loc = self.A_loc.transpose()
        if plan.world == 1:
            return
        A_rem = CSRGraph(plan.rowptr_rem, plan.col_rem, plan.val_rem, n_loc, n_halo)
        self._t_rem = A_rem.transpose()          # [n_halo, n_loc]: one partial row per halo slot
        self._t_rem._t = None
        del A_rem
        if self._R is None:
            self._return_setup()

    def _return_setup(self):
        """Buffers of the gradient return: the partial rows (one per halo slot), the receive buffer of the rows the
        peers send back, and R, the pattern-only CSR that adds them to their local rows in (peer, slot) order."""
        from .graph import CSRGraph, index_block_transpose
        plan = self.plan
        n_loc, n_halo = plan.n_local, max(plan.n_halo, 1)
        n_send = int(plan.send_rows.numel())
        # R: local row r <- the positions k of the send list with send_rows[k] == r, ascending k
        rowptr_t, pos_t = index_block_transpose(plan.send_rows, n_loc)
        deg = rowptr_t[1:] - rowptr_t[:-1]
        rows = torch.nonzero(deg > 0).flatten()
        rp, cc, _ = select_rows(rowptr_t, pos_t[:max(n_send, 0)], None, rows)
        self._R = CSRGraph(rp, cc.to(torch.int32), None, int(rows.numel()), max(n_send, 1))
        self._R._row_map = rows.to(torch.int32).contiguous()
        self._partial = torch.empty((n_halo, self.ld), dtype=self.dtype, device=self.dev)[:, :self.F]
        if self.transport in ("p2p", "ce"):
            self._back_buf = _PeerBuffer(max(n_send, 1) * self.ld * self.elem, plan.rank, plan.world, self.group)
            self._bufs.append(self._back_buf)
            self.back = _raw_view(self._back_buf.own, max(n_send, 1), self.ld, self.dtype, self.dev)[:, :self.F]
            self._bcopy_streams = [torch.cuda.Stream(device=self.dev, priority=-1) for _ in range(4)]
            self._ev_partial = torch.cuda.Event()
            self._ev_bcopied = [torch.cuda.Event() for _ in range(4)]
        else:
            self.back = torch.empty((max(n_send, 1), self.F), dtype=self.dtype, device=self.dev)

    def backward(self, dY: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """dX_local = (Âᵀ·dY)[own rows]: the autograd of GCN/GCN.py:43 on the partitioned graph.
        Remote partials first (they must travel), the local transposed product while they do, then the
        partials this rank's rows received are added in fixed (peer, slot) order."""
        from .functional import spmm_raw
        plan = self.plan
        assert dY.shape == (plan.n_local, self.F) and dY.dtype == self.dtype and dY.is_cuda
        if self._t_loc is None:
            self._backward_setup()
        if out is None:
            out = torch.empty((plan.n_local, self.F), dtype=self.dtype, device=self.dev)
        if plan.world == 1:
            return spmm_raw(self._t_loc, dY, out=out)
        spmm_raw(self._t_rem, dY, out=self._partial)           # partial[h] = Σ_i Â[i, halo h] dY[i]
        self._return_send(lambda: spmm_raw(self._t_loc, dY, out=out))  # local transposed product, under the copies
        self._return_add(out)
        return out

    def return_halo_grad(self, dX_comb: torch.Tensor) -> torch.Tensor:
        """Backward of `gather_halo`: dX_local = dX_comb[:n_local] + the gradients of this rank's rows that the peers
        return (rows dX_comb[n_local:] travel to their owners), added in fixed (peer, slot) order."""
        plan = self.plan
        assert dX_comb.shape == (plan.n_local + plan.n_halo, self.F) and dX_comb.dtype == self.dtype
        out = dX_comb[:plan.n_local].clone()
        if plan.world == 1:
            return out
        if self._R is None:
            self._return_setup()
        self._partial[:plan.n_halo].copy_(dX_comb[plan.n_local:])
        self._return_send()
        self._return_add(out)
        return out

    def _return_send(self, local=None):
        """Send the partial rows to their owners (copy engines + flags, or all_to_all); `local()` runs on the main
        stream while they travel.  On return the rows this rank receives are in `self.back`, visible to the main
        stream."""
        plan = self.plan
        main = torch.cuda.current_stream()
        s = self._bstep
        if self.transport == "nccl":
            dist.all_to_all_single(self.back[:int(plan.send_rows.numel())], self._partial[:plan.n_halo].contiguous(),
                                   output_split_sizes=plan.send_counts, input_split_sizes=plan.recv_counts,
                                   group=self.group)
            if local is not None:
                local()
        else:
            self._ev_partial.record(main)
            comm = self.comm
            comm.wait_event(self._ev_partial)
            with torch.cuda.stream(comm):
                if s > 0:
                    self._flags.wait(3, s, comm)  # every owner has consumed the partials of the previous step
                self._copy_to_peers(self._bcopy_streams, self._ev_bcopied, self._ev_partial, comm, self._back_buf.ptrs,
                                    plan.back_off, self._partial.data_ptr(), self._recv_off, plan.recv_counts,
                                    wait_join=s > 0)
                self._flags.signal(2, s + 1, comm)
            if local is not None:
                local()
            self._flags.wait(2, s + 1, main)

    def _return_add(self, out: torch.Tensor):
        """out[r] += the received rows of local row r, in (peer, slot) order; frees the receive buffer for the
        peers' next step.  bf16: the partial rows travel as bf16, and out[r] plus its received rows is summed in fp32
        and rounded once per row (the accumulating SpMM row flush) — the 1-GPU bf16 rule of fp32 accumulation with
        one rounding at the end, applied to the owner's add."""
        from .functional import spmm_ex
        if self._R.n_rows > 0:
            spmm_ex(self._R, self.back, out, row_map=self._R._row_map, accumulate=True)
        if self.transport != "nccl":
            self._flags.signal(3, self._bstep + 1, torch.cuda.current_stream())
        self._bstep += 1

    def close(self):
        _close_peer_buffers(self._bufs, self.dev, self.group)
        self._bufs = []


class PartitionedGraph:
    """This rank's share of a row-partitioned graph, in the form a GCN layer takes as `adj`
    (`Graph_conv_layer.forward(X_local, pg)`, `GCN_Model.forward(X_local, pg)`; X_local = the rank's own rows).

    Holds the row-block `bounds`, the `HaloPlan` (built once, at the widest width: only the schedule choice
    depends on F) and one `PartitionedSpmm` per feature width in `widths`.  The operators are built here, not on
    first use: creating one maps peer buffers and is a collective.

    Lock-step: the halo exchange counts steps with flags in peer memory, so every rank of `group` must run the
    same sequence of forward and backward calls (same layers, same order) — a model's forward / backward on every
    rank, every step.  Ranks that own no training row still run both.

    GAT layers take it as well (`GAT.forward(X_local, pg)`): `attention()` is the block in the combined column space
    (AttentionView, built here: one more collective), and `widths` must then list every layer's H*F'.

    Constructors: `PartitionedGraph(rowptr, col, val, bounds, rank, world, widths, ...)` from the rank's own row
    block (rowptr over its rows, GLOBAL column ids — what `build_halo_plan` takes), or `from_global(g, ...)` for a
    graph every rank holds.  Keyword arguments other than the plan's go to every `PartitionedSpmm`."""

    def __init__(self, rowptr: torch.Tensor, col: torch.Tensor, val: Optional[torch.Tensor], bounds: List[int],
                 rank: int, world: int, widths, device=None, group=None, waves: Optional[int] = 1,
                 two_pass_chunks: Optional[int] = None, transport: str = "p2p", dtype: torch.dtype = torch.float32,
                 **op_kw):
        self.bounds, self.rank, self.world, self.group = [int(b) for b in bounds], int(rank), int(world), group
        self.dev = torch.device(device) if device is not None else col.device
        self.dtype = dtype  # the feature dtype of every operator and exchange (fp32 or bf16)
        widths = sorted({int(w) for w in widths})
        if not widths or widths[0] <= 0:
            raise ValueError("PartitionedGraph: at least one positive feature width is needed")
        elem = 4 if dtype == torch.float32 else 2
        rowptr, col = rowptr.to(self.dev), col.to(self.dev)
        self.plan = build_halo_plan(rowptr, col, None if val is None else val.to(self.dev),
                                    self.bounds, self.rank, self.world, group=group, waves=waves,
                                    two_pass_chunks=two_pass_chunks, F=widths[-1], elem_size=elem)
        self._att = build_attention_view(self.plan, rowptr, col, group)
        self._att_graph = None
        self.ops: Dict[int, PartitionedSpmm] = {}
        try:
            for F in widths:
                self.ops[F] = PartitionedSpmm(self.plan, F, self.dev, group=group, transport=transport, dtype=dtype,
                                              **op_kw)
        except Exception:
            self.close()
            raise

    @classmethod
    def from_global(cls, g, rank: int, world: int, widths, group=None, **kw) -> "PartitionedGraph":
        """From a whole `CSRGraph` every rank holds: row blocks balanced by nnz (`balanced_bounds`), this rank's
        block cut out of it."""
        bounds = balanced_bounds(g.rowptr, world)
        lo, hi = bounds[rank], bounds[rank + 1]
        rows = torch.arange(lo, hi, dtype=torch.int64, device=g.rowptr.device)
        rp, cc, vv = select_rows(g.rowptr, g.col, g.val, rows)
        return cls(rp, cc, vv, bounds, rank, world, widths, device=kw.pop("device", g.rowptr.device), group=group, **kw)

    @property
    def n_local(self) -> int:
        return self.plan.n_local

    @property
    def row_range(self):
        return self.bounds[self.rank], self.bounds[self.rank + 1]

    def op(self, F: int) -> PartitionedSpmm:
        op = self.ops.get(int(F))
        if op is None:
            raise _lib.GnnError(f"PartitionedGraph: no operator for feature width {F} (built for {sorted(self.ops)}); "
                                "list every layer's output width in `widths`")
        return op

    @property
    def edge_slot_base(self) -> int:
        return self._att.edge_slot_base

    def attention(self):
        """(CSRGraph of the block in the combined column space [n_local, n_local + n_halo], edge_slot_base) for the
        fused attention kernels.  Raises on every rank when the graph has a row without edges."""
        from .graph import CSRGraph
        self._att.require_edges()
        if self._att_graph is None:
            a = self._att
            self._att_graph = CSRGraph(a.rowptr, a.col, None, a.n_rows, a.n_cols)
        return self._att_graph, self._att.edge_slot_base

    def local_index(self, idx_global: torch.Tensor) -> torch.Tensor:
        """The global node ids of `idx_global` (train / val / test ids) that this rank owns, as local row indices
        (ascending where idx_global is)."""
        return _local_index(idx_global, *self.row_range)

    def close(self):
        """Free the peer buffers (collective: every rank calls it)."""
        for op in self.ops.values():
            op.close()
        self.ops = {}


# ---- HAN's metapath graphs over one row partition ---------------------------------------------

def union_block(rowptrs, cols, n_global: int):
    """Per-row union of the columns of M row blocks over the same rows (GLOBAL column ids): the block whose halo
    plan serves all M metapaths with one exchange.  Returns (rowptr, col int64), columns ascending per row."""
    n_loc = int(rowptrs[0].numel()) - 1
    dev = cols[0].device
    keys = []
    for rp, c in zip(rowptrs, cols):
        rows = torch.repeat_interleave(torch.arange(n_loc, dtype=torch.int64, device=dev), rp[1:] - rp[:-1],
                                       output_size=int(c.numel()))
        keys.append(rows * n_global + c.to(torch.int64))
    key = torch.unique(torch.cat(keys), sorted=True)
    rowptr = torch.zeros(n_loc + 1, dtype=torch.int64, device=dev)
    torch.cumsum(torch.bincount(key // n_global, minlength=n_loc), 0, out=rowptr[1:])
    return rowptr, key % n_global


@dataclass
class MetapathView:
    """This rank's row block of M metapath graphs in ONE combined column space, that of the union block's halo plan:
    local column c -> c - lo, remote column -> n_local + its slot in the union halo.  The M renamed blocks are stacked
    as a block diagonal (graph m's rows at m * n_local, its column ids at m * n_comb), which the batched-rectangular
    attention kernels walk in one launch; every row keeps its metapath's global edge order.
    slot_shift[m]: global batched edge slot (the block diagonal of the M whole graphs, as one GPU numbers them) minus
    local batched slot, for graph m's edges — the seeded attention dropout of the block is then the whole set's."""
    rowptr: torch.Tensor          # [M * n_local + 1]
    col: torch.Tensor             # int32 batched combined column ids
    n_graphs: int
    n_local: int
    n_comb: int                   # n_local + n_halo of the union plan
    slot_shift: List[int]
    any_empty_row: bool           # some row of some metapath, on any rank, has no edge
    halo_rows_per_graph: List[int]  # distinct remote columns of each metapath's block (what it alone would fetch)

    def require_edges(self):
        """GAT's rule for a row without edges is the mean over ALL N nodes; the flag is global, so every rank raises
        together."""
        if self.any_empty_row:
            raise _lib.GnnError("HAN on PartitionedMetapaths: a metapath graph has rows without edges (their output "
                                "is the mean over all nodes, not supported across ranks); add self-loops")


def build_metapath_view(plan: HaloPlan, rowptrs, cols, group=None) -> MetapathView:
    """The view of M row blocks (rowptr over the rank's rows, GLOBAL column ids) in the combined column space of
    `plan`, the union block's plan (its halo must hold every remote column of every block).  Collective when
    world > 1: one all_gather of (per-metapath nnz, has-empty-row) per rank."""
    lo, hi = plan.bounds[plan.rank], plan.bounds[plan.rank + 1]
    n_loc, M = hi - lo, len(rowptrs)
    n_comb = n_loc + plan.n_halo
    dev = cols[0].device
    halo_ids = plan.halo_ids.to(dev)
    order = torch.argsort(halo_ids)
    sorted_ids = halo_ids[order]
    parts_rp, parts_col, halo_m, nnz_loc, off = [], [], [], [], 0
    empty = False
    for m, (rp, c) in enumerate(zip(rowptrs, cols)):
        c64 = c.to(dev).to(torch.int64)
        is_loc = (c64 >= lo) & (c64 < hi)
        rem = c64[~is_loc]
        pos = torch.searchsorted(sorted_ids, rem)
        if rem.numel() and (sorted_ids.numel() == 0 or
                            not torch.equal(sorted_ids[pos.clamp_max(sorted_ids.numel() - 1)], rem)):
            raise ValueError("build_metapath_view: a remote column is missing from the plan's halo")
        comb = torch.empty_like(c64)
        comb[is_loc] = c64[is_loc] - lo
        comb[~is_loc] = order[pos] + n_loc
        parts_rp.append(rp.to(dev)[:-1] + off)
        parts_col.append(comb + m * n_comb)
        halo_m.append(int(torch.unique(rem).numel()))
        nnz_loc.append(int(c.numel()))
        off += int(c.numel())
        empty = empty or (n_loc > 0 and bool((rp[1:] == rp[:-1]).any().item()))
    parts_rp.append(torch.tensor([off], dtype=torch.int64, device=dev))
    rowptr = torch.cat(parts_rp)
    col = torch.cat(parts_col).to(torch.int32)
    if plan.world > 1:
        mine = torch.tensor(nnz_loc + [int(empty)], dtype=torch.int64, device=dev)
        every = [torch.empty_like(mine) for _ in range(plan.world)]
        dist.all_gather(every, mine, group=group)
        every = [[int(x) for x in e.tolist()] for e in every]
    else:
        every = [nnz_loc + [int(empty)]]
    nnz_glob = [sum(e[m] for e in every) for m in range(M)]
    shift = []
    for m in range(M):
        before = sum(e[m] for e in every[:plan.rank])  # the whole graph m's rowptr[lo]
        shift.append(sum(nnz_glob[k] - nnz_loc[k] for k in range(m)) + before)
    return MetapathView(rowptr, col, M, n_loc, n_comb, shift, any(e[M] for e in every), halo_m)


def metapath_row_plan(count, n: int, M: int, rank: int, world: int, max_nnz_per_rank: Optional[int] = None,
                      group=None, what: str = "PartitionedMetapaths.from_relations", items: str = "metapaths"):
    """Row bounds of M metapath graphs over n nodes that no rank holds whole, and this rank's block rowptrs.

    `count(m, lo, hi)` returns the int64 rowptr [hi - lo + 1] of rows [lo, hi) of metapath m.  Each rank counts its
    rows of an even split (`shard_bounds`) for every metapath; one all_gather in rank order gives every rank all
    M·N per-row counts (8·M·N bytes), hence the global rowptr_m and bounds = balanced_bounds(Σ_m rowptr_m, world),
    the bounds `PartitionedMetapaths.from_global` would choose.  If some rank's block holds more than
    `max_nnz_per_rank` entries, every rank raises the same GnnError (they all see every count); `what` and `items`
    name the caller and what its M graphs are in that message.
    Returns (bounds, [rowptr_m of this rank's block, starting at 0])."""
    even = shard_bounds(n, world)
    lo, hi = even[rank], even[rank + 1]
    mine = [count(m, lo, hi) for m in range(M)]
    deg = torch.stack([rp[1:] - rp[:-1] for rp in mine]) if hi > lo else None
    dev = mine[0].device
    width = max(even[p + 1] - even[p] for p in range(world))
    if world > 1:
        send = torch.zeros(M, width, dtype=torch.int64, device=dev)
        if deg is not None:
            send[:, :hi - lo] = deg
        every = [torch.empty_like(send) for _ in range(world)]
        dist.all_gather(every, send, group=group)
        deg_all = torch.cat([e[:, :even[p + 1] - even[p]] for p, e in enumerate(every)], dim=1)
    else:
        deg_all = deg if deg is not None else torch.zeros(M, 0, dtype=torch.int64, device=dev)
    rowptr = torch.zeros(M, n + 1, dtype=torch.int64, device=dev)
    torch.cumsum(deg_all, 1, out=rowptr[:, 1:])
    bounds = balanced_bounds(rowptr.sum(0), world)
    block_nnz = [int(x) for x in (rowptr[:, bounds[1:]] - rowptr[:, bounds[:-1]]).sum(0).tolist()]
    if max_nnz_per_rank is not None and max(block_nnz) > max_nnz_per_rank:
        over = ", ".join(f"rank {p}: {v}" for p, v in enumerate(block_nnz) if v > max_nnz_per_rank)
        raise _lib.GnnError(f"{what}: a rank's block has more than max_nnz_per_rank = "
                            f"{max_nnz_per_rank} entries over the {M} {items} ({over}; "
                            f"{4 * max(block_nnz)} bytes of column ids)")
    b_lo, b_hi = bounds[rank], bounds[rank + 1]
    return bounds, [(rowptr[m, b_lo:b_hi + 1] - rowptr[m, b_lo]).contiguous() for m in range(M)]


class PartitionedMetapaths:
    """This rank's share of HAN's M metapath graphs over the same N nodes, row-partitioned, in the form
    `HANModel.forward(pm, X_local)` takes (X_local = the rank's own rows).  A sequence of length M, as the list of
    graphs it replaces.

    The row bounds are common to all metapaths, balanced on Σ_m rowptr_m (every rank's attention work is the sum over
    the metapaths).  ONE halo serves them all: `union`, a `PartitionedGraph` over the per-row union of the M blocks'
    columns, whose operators exchange the stacked Wh_local [n_local, M*H*F'] once per layer (`widths` lists every
    layer's M*H*F').  The union moves some rows for metapaths that do not read them: `halo_rows` against
    `halo_rows_per_graph` (Σ over the metapaths) shows that cost.  `attention()` is the batched block in the union's
    combined column space (MetapathView) and the per-graph dropout slot shifts.

    Collective construction; the lock-step rule of PartitionedGraph holds.  Constructors: from the rank's own row
    blocks (rowptr over its rows, GLOBAL column ids) or `from_global(graphs, ...)` for graphs every rank holds."""

    def __init__(self, rowptrs, cols, bounds: List[int], rank: int, world: int, widths, device=None, group=None,
                 **kw):
        if not 1 <= len(rowptrs) == len(cols):
            raise ValueError("PartitionedMetapaths: one (rowptr, col) block per metapath")
        dev = torch.device(device) if device is not None else cols[0].device
        rowptrs = [r.to(dev) for r in rowptrs]
        cols = [c.to(dev) for c in cols]
        self.n_total = int(bounds[-1])
        rp_u, col_u = union_block(rowptrs, cols, max(self.n_total, 1))
        self.union = PartitionedGraph(rp_u, col_u, None, bounds, rank, world, widths, device=dev, group=group, **kw)
        try:
            self._view = build_metapath_view(self.union.plan, rowptrs, cols, group)
        except Exception:
            self.union.close()
            raise
        self.rank, self.world, self.group, self.bounds = self.union.rank, self.union.world, group, self.union.bounds
        self._graph = None
        self._shift = None

    @classmethod
    def from_global(cls, graphs, rank: int, world: int, widths, group=None, **kw) -> "PartitionedMetapaths":
        """From M whole `CSRGraph`s over the same N nodes that every rank holds: bounds balanced on Σ_m rowptr_m."""
        graphs = list(graphs)
        n = graphs[0].n_rows
        if any(g.n_rows != n or g.n_cols != n for g in graphs):
            raise ValueError("PartitionedMetapaths: square metapath graphs over the same nodes")
        bounds = balanced_bounds(sum(g.rowptr for g in graphs), world)
        lo, hi = bounds[rank], bounds[rank + 1]
        rows = torch.arange(lo, hi, dtype=torch.int64, device=graphs[0].rowptr.device)
        blocks = [select_rows(g.rowptr, g.col, None, rows)[:2] for g in graphs]
        return cls([b[0] for b in blocks], [b[1] for b in blocks], bounds, rank, world, widths,
                   device=kw.pop("device", graphs[0].rowptr.device), group=group, **kw)

    @classmethod
    def from_relations(cls, relations, rank: int, world: int, widths, self_loops: bool = True,
                       max_nnz_per_rank: Optional[int] = None, group=None, **kw) -> "PartitionedMetapaths":
        """From M relation CSRs R_m [N x X_m] (paper x author, paper x subject) that every rank holds: metapath m is
        pattern(R_m·R_mᵀ) (+ I with self_loops), composed on the device (`CSRGraph.metapath`), but each rank fills
        only its own row block.  Collective: the ranks count the rows of an even split and exchange the per-row
        counts (`metapath_row_plan`: M·N int64 on every rank), which gives exactly the bounds `from_global` chooses
        for the composed graphs; a block of more than `max_nnz_per_rank` entries raises on every rank.  The result
        equals `from_global([CSRGraph.metapath(R, self_loops) for R in relations], ...)` bit for bit."""
        from .graph import _pattern_count, _pattern_fill, _require_cuda, _require_ids_in_range
        rels = list(relations)
        if not rels or any(R.n_rows != rels[0].n_rows for R in rels):
            raise ValueError("PartitionedMetapaths.from_relations: relations over the same N nodes")
        _require_cuda(*[R.rowptr for R in rels])
        _require_ids_in_range(*rels)  # every rank holds the same relations: a refusal is every rank's
        pairs = [(R, R.transpose()) for R in rels]

        def count(m, lo, hi):
            return _pattern_count(pairs[m][0], pairs[m][1], lo, hi, self_loops)

        bounds, rowptrs = metapath_row_plan(count, rels[0].n_rows, len(rels), rank, world, max_nnz_per_rank, group)
        lo, hi = bounds[rank], bounds[rank + 1]
        cols = [_pattern_fill(R, Rt, lo, hi, self_loops, rp, int(rp[-1].item())) for (R, Rt), rp in zip(pairs, rowptrs)]
        return cls(rowptrs, cols, bounds, rank, world, widths, device=kw.pop("device", rels[0].rowptr.device),
                   group=group, **kw)

    def __len__(self) -> int:
        return self._view.n_graphs

    def __getitem__(self, m: int):
        """Metapath m's block in the combined column space: (rowptr [n_local + 1], int32 col in [0, n_comb))."""
        v = self._view
        if not 0 <= m < v.n_graphs:
            raise IndexError(m)
        r = v.n_local
        rp = v.rowptr[m * r:(m + 1) * r + 1]
        return rp - rp[0], v.col[int(rp[0]):int(rp[-1])] - m * v.n_comb

    @property
    def n_local(self) -> int:
        return self.union.n_local

    @property
    def row_range(self):
        return self.union.row_range

    @property
    def dtype(self) -> torch.dtype:
        return self.union.dtype

    @property
    def halo_rows(self) -> int:
        return self.union.plan.n_halo

    @property
    def halo_rows_per_graph(self) -> List[int]:
        return list(self._view.halo_rows_per_graph)

    @property
    def slot_shift(self) -> List[int]:
        return list(self._view.slot_shift)

    def op(self, F: int) -> PartitionedSpmm:
        return self.union.op(F)

    def attention(self):
        """(batched CSRGraph [M*n_local, M*n_comb] in the combined column space, device int64 [M] slot shifts) for the
        batched-rectangular attention kernels.  Raises on every rank when some metapath row has no edge."""
        from .graph import CSRGraph
        self._view.require_edges()
        if self._graph is None:
            v = self._view
            g = CSRGraph(v.rowptr, v.col, None, v.n_graphs * v.n_local, v.n_graphs * v.n_comb)
            g.transpose()      # built once with the block: the backward's pass 2 walks it
            g.gat_long_rows()
            g.transpose().gat_long_rows()
            self._graph = g
            self._shift = torch.tensor(v.slot_shift, dtype=torch.int64, device=v.rowptr.device)
        return self._graph, self._shift

    def local_index(self, idx_global: torch.Tensor) -> torch.Tensor:
        return self.union.local_index(idx_global)

    def close(self):
        """Free the union's peer buffers (collective: every rank calls it)."""
        self.union.close()


# ---- GTN's learned metapath composition over one row partition ----------------------------------

class PeerRowReduce:
    """Ordered cross-rank sums of fp32 row buffers over NVLink peer memory, one peer-mapped buffer per reduce SITE
    (a named place in a step that runs every step, in the same order on every rank).

      all_reduce(site, x [N, F])               every rank gets Σ_q x_q, all N rows
      reduce_scatter(site, x [N, F], relu)     this rank gets relu?(Σ_q x_q) of its own rows [lo, hi)
      all_gather(site, x_local [n_local, F])   every rank gets the owners' blocks stacked in rank order, [N, F]

    A call writes this rank's operand into its own buffer of the site, raises its arrival flag on every peer, waits
    for theirs, and reduces with `gnn_peer_reduce_rows_f32`, which adds the ranks' rows in rank order 0..P-1 in fp32
    (the all-gather copies the owners' blocks with `gnn_peer_copy_async` instead); then it raises its "consumed" flag.
    A buffer is rewritten only after every peer has raised "consumed" for the previous call of that site.  Every wait
    is bounded: a lost peer sets a status word (`check_status`) instead of hanging the GPU.  Nothing is read back to
    the host.  At world 1 no buffer exists: the reduction is the same kernel over one source, a copy (or ReLU).

    sites: {name: (rows, cols)} of this rank's buffer; every rank passes the same names.  Construction is collective
    (the buffers are exported with CUDA IPC and mapped by every peer)."""

    def __init__(self, sites: Dict[str, tuple], bounds: List[int], rank: int, world: int, device, group=None,
                 timeout_ms: int = 20000):
        self.bounds, self.rank, self.world, self.group = [int(b) for b in bounds], int(rank), int(world), group
        self.dev, self.timeout_ms = torch.device(device), int(timeout_ms)
        self._sites: Dict[str, dict] = {}
        self._bufs: List[_PeerBuffer] = []
        self._flags: Optional[_PeerFlags] = None
        if self.world == 1:
            return
        try:
            # flag arrays 2k (arrive) and 2k + 1 (consumed) for site k
            self._flags = _PeerFlags(2 * len(sites), self.rank, self.world, group, self.dev, self.timeout_ms)
            self._bufs.append(self._flags.buf)
            for k, (name, (rows, cols)) in enumerate(sorted(sites.items())):
                ld = (int(cols) + 3) // 4 * 4  # 16-byte rows: the reduce kernel reads float4 vectors
                buf = _PeerBuffer(max(int(rows), 1) * ld * 4, self.rank, self.world, group)
                self._bufs.append(buf)
                self._sites[name] = {"buf": buf, "rows": int(rows), "cols": int(cols), "ld": ld, "flag": 2 * k,
                                     "step": 0}
        except Exception:
            self.close()
            raise

    def _site(self, name: str, x: torch.Tensor) -> dict:
        site = self._sites.get(name)
        if site is None:
            raise _lib.GnnError(f"PeerRowReduce: no reduce site {name!r} (built for {sorted(self._sites)})")
        if x.dtype != torch.float32 or x.dim() != 2 or x.shape[0] > site["rows"] or x.shape[1] > site["cols"]:
            raise _lib.GnnError(f"PeerRowReduce: site {name!r} holds fp32 [{site['rows']}, {site['cols']}], got "
                                f"{x.dtype} {tuple(x.shape)}")
        return site

    def _publish(self, site: dict, x: torch.Tensor, stream):
        """x into this rank's buffer of the site once every peer has read its previous contents; then the flags."""
        s = site["step"]
        if s > 0:
            self._flags.wait(site["flag"] + 1, s, stream)
        if x.shape[0]:
            _raw_view(site["buf"].own, x.shape[0], site["ld"], torch.float32, self.dev)[:, :x.shape[1]].copy_(x)
        self._flags.signal(site["flag"], s + 1, stream)
        self._flags.wait(site["flag"], s + 1, stream)

    def _done(self, site: dict, stream):
        site["step"] += 1
        self._flags.signal(site["flag"] + 1, site["step"], stream)

    def _reduce(self, name: str, x: torch.Tensor, row_lo: int, row_hi: int, relu: bool) -> torch.Tensor:
        from .functional import peer_reduce_rows_raw
        F = int(x.shape[1])
        out = torch.empty((row_hi - row_lo, F), dtype=torch.float32, device=self.dev)
        if self.world == 1:
            x = x.contiguous()
            return peer_reduce_rows_raw([x.data_ptr()], F, F, row_lo, row_hi, out, relu)
        site = self._site(name, x)
        stream = torch.cuda.current_stream(self.dev)
        self._publish(site, x, stream)
        peer_reduce_rows_raw(site["buf"].ptrs, site["ld"], F, row_lo, row_hi, out, relu)
        self._done(site, stream)
        return out

    def all_reduce(self, name: str, x: torch.Tensor) -> torch.Tensor:
        return self._reduce(name, x, 0, int(x.shape[0]), False)

    def reduce_scatter(self, name: str, x: torch.Tensor, relu: bool = False) -> torch.Tensor:
        return self._reduce(name, x, self.bounds[self.rank], self.bounds[self.rank + 1], relu)

    def all_gather(self, name: str, x_local: torch.Tensor) -> torch.Tensor:
        F = int(x_local.shape[1])
        if self.world == 1:
            return x_local.contiguous().clone()
        site = self._site(name, x_local)
        if site["ld"] != site["cols"] or F != site["cols"]:
            raise _lib.GnnError(f"PeerRowReduce.all_gather: site {name!r} needs contiguous rows of {F} columns")
        stream = torch.cuda.current_stream(self.dev)
        out = torch.empty((self.bounds[-1], F), dtype=torch.float32, device=self.dev)
        self._publish(site, x_local, stream)
        lib, row_bytes = _lib.load(), F * 4
        for q in range(self.world):
            rows = self.bounds[q + 1] - self.bounds[q]
            if rows:
                _lib.check(lib.gnn_peer_copy_async(out.data_ptr() + self.bounds[q] * row_bytes, site["buf"].ptrs[q],
                                                   rows * row_bytes, stream.cuda_stream), "gnn_peer_copy_async")
        self._done(site, stream)
        return out

    def check_status(self):
        """Raise if a flag wait of an earlier call timed out (synchronises)."""
        if self._flags is not None:
            self._flags.check_status("reduce")

    def close(self):
        """Free the peer buffers (collective)."""
        if self._bufs:
            _close_peer_buffers(self._bufs, self.dev, self.group)
            self._bufs = []
            self._sites = {}


GTN_MAX_CHANNELS = 8  # gnn_spgemm_values_f32 takes up to 8 channels: the [N, C] reduce sites hold 8 columns


class PartitionedRelationStack:
    """One rank's share of a `layers.gtn.RelationStack` that every rank holds, for `GTN_Model.forward(ps, X_local,
    target_local)`: rank p owns rows [lo, hi) of every composed H_l (the same bounds for all layers), of X and of the
    output.  The union pattern U and its values V stay whole on every rank (they are small).

      P_1 = pattern(U[lo:hi]·U),  D_l = P_l without the entries (r, lo + r),  P_{l+1} = pattern(D_l·U)
      gcn   the CSR of (D_L + I)ᵀ restricted to the local rows: N rows, columns the local row index i - lo, self-loops
            for j in [lo, hi)

    The composition needs no communication.  GTN's column normalisation and the degrees of its final gcn_conv sum
    along columns, so each rank computes partial [N, C] sums over its rows and `PeerRowReduce.all_reduce` adds them in
    rank order; the gcn_conv aggregates only the local rows' XW into a partial [N, C·w_out], which a reduce-scatter with
    the ReLU fused turns into this rank's rows (its backward is the all-gather of the output gradient).

    Bounds: every rank builds the chain P_1 .. P_L for its rows of an even split (`shard_bounds`), filling
    P_1 .. P_{L-1} and counting P_L; `metapath_row_plan` (one "metapath" per layer) exchanges the per-row counts and
    returns bounds balanced on Σ_l rowptr_l and this rank's rowptrs of every layer, from which the final block is
    filled layer by layer without counting again.  A block of more than `max_nnz_per_rank` entries over the L layers
    raises the same GnnError on every rank.

    width = num_channels * w_out of the model (it sizes the output sites).  Collective construction; every rank runs
    the same sequence of forward and backward calls (the reduce sites count calls with flags in peer memory)."""

    def __init__(self, stack, rank: int, world: int, num_layers: int, width: int, max_nnz_per_rank: Optional[int] = None,
                 group=None, timeout_ms: int = 20000):
        from .graph import CSRGraph, _pattern_count, _pattern_fill
        from .layers.gtn import _drop_diagonal, _gcn_pattern, _plan
        L, n = int(num_layers), stack.n
        if L < 1 or int(width) <= 0:
            raise ValueError(f"PartitionedRelationStack: num_layers >= 1 and width > 0 needed, got {L}, {width}")
        if int(world) > 1 and int(width) % 4:
            raise ValueError(f"PartitionedRelationStack: width {width} must be a multiple of 4 across ranks "
                             "(the output's all-gather copies whole 16-byte rows)")
        self.stack, self.rank, self.world, self.group = stack, int(rank), int(world), group
        self.num_layers, self.width, self.num_edge, self.n = L, int(width), stack.num_edge, n
        U = stack.U
        U.transpose()  # B of every product is read through its transpose
        chain = {}

        def count(m, lo, hi):
            """rowptr of rows [lo, hi) of P_{m+1}; P_1 .. P_{L-1} of the even split are filled for the next count."""
            A, a_lo, a_hi = (U, lo, hi) if m == 0 else (chain["D"], 0, hi - lo)
            rp = _pattern_count(A, U, a_lo, a_hi, False)
            if m < L - 1:
                P = CSRGraph(rp, _pattern_fill(A, U, a_lo, a_hi, False, rp, int(rp[-1].item())), None, hi - lo, n)
                chain["D"] = _drop_diagonal(P, lo)[0]
            return rp

        self.bounds, rowptrs = metapath_row_plan(count, n, L, self.rank, self.world, max_nnz_per_rank, group,
                                                 what="PartitionedRelationStack", items="layers")
        chain.clear()  # the even split's fills are not needed any more
        lo, hi = self.row_range
        n_loc = hi - lo
        u0, u1 = int(U.rowptr[lo].item()), int(U.rowptr[hi].item())
        self.U_rows = (CSRGraph(U.rowptr[lo:hi + 1] - u0, U.col[u0:u1], None, n_loc, n), u0, u1)
        _plan(self.U_rows[0])
        _plan(self.U_rows[0].transpose())
        self.P, self.D, self.keep = [], [], []
        A, a_lo, a_hi = U, lo, hi
        for rp in rowptrs:
            P = CSRGraph(rp, _pattern_fill(A, U, a_lo, a_hi, False, rp, int(rp[-1].item())), None, n_loc, n)
            D, keep = _drop_diagonal(P, lo)
            for g in (P, D):  # transposes the backward and the column sums walk, and their SpMM plans
                _plan(g)
                _plan(g.transpose())
            self.P.append(P)
            self.D.append(D)
            self.keep.append(keep)
            A, a_lo, a_hi = D, 0, n_loc
        self.gcn = _gcn_pattern(self.D[-1], self.keep[-1], n, lo)
        sites = {"deg": (n, GTN_MAX_CHANNELS), "deg_bwd": (n, GTN_MAX_CHANNELS), "out": (n, self.width),
                 "out_bwd": (max(self.bounds[p + 1] - self.bounds[p] for p in range(self.world)), self.width)}
        for l in range(1, L):
            sites[f"norm{l}"] = sites[f"norm{l}_bwd"] = (n, GTN_MAX_CHANNELS)
        self.reduce = PeerRowReduce(sites, self.bounds, self.rank, self.world, U.device, group, timeout_ms)

    @property
    def row_range(self):
        return self.bounds[self.rank], self.bounds[self.rank + 1]

    @property
    def n_local(self) -> int:
        return self.bounds[self.rank + 1] - self.bounds[self.rank]

    @property
    def nnz_per_layer(self) -> List[int]:
        """nnz of this rank's block of every P_l."""
        return [P.nnz for P in self.P]

    def local_index(self, idx_global: torch.Tensor) -> torch.Tensor:
        """The global node ids of `idx_global` this rank owns, as local row indices."""
        return _local_index(idx_global, *self.row_range)

    def check_status(self):
        """Raise if a flag wait of an earlier step timed out (synchronises)."""
        self.reduce.check_status()

    def close(self):
        """Free the peer buffers (collective: every rank calls it)."""
        self.reduce.close()


# ---- a feature table sharded across ranks ---------------------------------------------------
_TABLE_DTYPES = {torch.float32: 4, torch.bfloat16: 2}


def shard_bounds(n_rows: int, world: int) -> List[int]:
    """Row-balanced contiguous blocks: shard p holds the rows [n*p // world, n*(p+1) // world) (empty shards when
    n_rows < world)."""
    n_rows, world = int(n_rows), int(world)
    if n_rows < 0 or world < 1:
        raise ValueError(f"shard_bounds: bad size (rows={n_rows}, world={world})")
    return [n_rows * p // world for p in range(world + 1)]


def locate_rows(ids: torch.Tensor, bounds: List[int]):
    """(shard, row within the shard) of every global id, by the sharded gather's rule: the last shard s with
    bounds[s] <= id.  Ids outside [0, bounds[-1]) get shard -1 (the gather skips them)."""
    ids = ids.to(torch.int64)
    b = torch.tensor(bounds, dtype=torch.int64, device=ids.device)
    s = torch.searchsorted(b, ids, right=True) - 1
    valid = (ids >= 0) & (ids < b[-1])
    s = torch.where(valid, s.clamp(0, len(bounds) - 2), torch.full_like(s, -1))
    local = torch.where(valid, ids - b[s.clamp(min=0)], torch.full_like(ids, -1))
    return s, local


def agree_layout(F: int, ld: int, dtype, bounds, error: Optional[str], rank: int, world: int, group=None):
    """The first step of building a ShardedTable (a collective): every rank states its block's width, padded row
    stride, dtype and the row bounds of all shards, plus any local refusal, and every rank raises the same GnnError
    if a rank refused or the ranks disagree — no rank is left waiting in a later collective, and no rank addresses
    a peer's shard by bounds the peer does not hold."""
    mine = (int(F), int(ld), str(dtype), tuple(int(b) for b in bounds), error)
    every = [None] * world
    dist.all_gather_object(every, mine, group=group)
    problems = [f"rank {q}: {v[-1]}" for q, v in enumerate(every) if v[-1]]
    if len({v[:3] for v in every}) > 1:
        problems.append("ranks disagree on (F, ld, dtype): " +
                        ", ".join(f"rank {q} {tuple(v[:3])}" for q, v in enumerate(every)))
    if len({v[3] for v in every}) > 1:
        problems.append("ranks disagree on the bounds: " +
                        ", ".join(f"rank {q} {list(v[3])}" for q, v in enumerate(every)))
    if problems:
        raise _lib.GnnError("ShardedTable: " + "; ".join(problems))


def _table_refusal(X: torch.Tensor) -> Optional[str]:
    if not torch.is_tensor(X) or X.dim() != 2:
        return "a 2-D feature tensor is needed"
    if not X.is_cuda:
        return "the table is on the CPU (the sharded gather reads device memory)"
    if X.dtype not in _TABLE_DTYPES:
        return f"dtype {X.dtype} (float32 or bfloat16)"
    if X.requires_grad:
        return "the table requires grad (features are inputs: there is no backward into a sharded table)"
    return None


class ShardedTable:
    """A read-only feature table split into contiguous row blocks (shards), one per rank: the table argument of
    `functional.gather_reduce_multi_raw` / `gather_reduce_multi_split_raw` and of `GraphSage.forward_sampled`, in
    place of a tensor too large for one GPU.  Shard s holds the global rows [bounds[s], bounds[s+1]); the gather
    reads each sampled row from its owner's memory (a peer's through a CUDA IPC mapping, over NVLink), and every
    reduced row is bit-identical to the same gather over the concatenated table.

    `ShardedTable(X_block, bounds, rank, world)` (a collective: every rank of `group` calls it) copies this rank's
    rows into a peer-mapped buffer of 16-byte aligned rows and maps every peer's; `from_global` cuts the block out of
    a table every rank holds; `local([t0, t1, ...])` builds the same object from tensors of one process on one
    device, without IPC.  Like a tensor it has `shape` (global rows, F), `dtype`, `device`, `stride()` and
    `requires_grad` (always False); `abs_max` is max |x| over the whole table."""

    def __init__(self, X_block: torch.Tensor, bounds, rank: int, world: int, group=None):
        self.bounds, self.rank, self.world, self.group = [int(b) for b in bounds], int(rank), int(world), group
        if self.world > _lib.MAX_SHARDS:
            raise _lib.GnnError(f"ShardedTable: {self.world} shards, at most {_lib.MAX_SHARDS}")
        err = _table_refusal(X_block)
        if err is None and (len(self.bounds) != self.world + 1 or
                            X_block.shape[0] != self.bounds[self.rank + 1] - self.bounds[self.rank]):
            err = f"block of {X_block.shape[0]} rows does not match bounds {self.bounds}"
        F = int(X_block.shape[1]) if torch.is_tensor(X_block) and X_block.dim() == 2 else -1
        dtype = X_block.dtype if torch.is_tensor(X_block) else None
        ld = self._padded_ld(F, dtype)
        agree_layout(F, ld, dtype, self.bounds, err, self.rank, self.world, group)
        self._set_layout(F, ld, dtype, X_block.device)
        n = X_block.shape[0]
        self._buf = _PeerBuffer(n * ld * _TABLE_DTYPES[dtype], self.rank, self.world, group)
        # the local fill either succeeds on every rank or every rank frees its buffer and raises (no rank is left in
        # a collective the others skipped)
        err = None
        try:
            if n:  # pad columns are zero, as pad_table leaves them: a 16-byte store of the gather may carry them out
                full = _raw_view(self._buf.own, n, ld, dtype, self.device)
                full[:, F:].zero_()
                full[:, :F].copy_(X_block)
            amax = X_block.detach().abs().max().float() if n else torch.zeros((), device=self.device)
            amax = amax.reshape(1).clone()
            torch.cuda.synchronize(self.device)
        except Exception as e:
            err = f"{type(e).__name__}: {e}"
        every = [None] * self.world
        dist.all_gather_object(every, err, group=group)
        failed = [f"rank {q}: {e}" for q, e in enumerate(every) if e]
        if failed:
            self._buf.close()
            raise _lib.GnnError("ShardedTable: filling the shards failed: " + "; ".join(failed))
        dist.all_reduce(amax, op=dist.ReduceOp.MAX, group=group)
        self.abs_max = float(amax.item())
        dist.barrier(group=group)  # no rank reads a shard before its owner has written it
        self._keep = []
        self._make_desc(self._buf.ptrs)

    @classmethod
    def from_global(cls, X: torch.Tensor, rank: int, world: int, group=None) -> "ShardedTable":
        """This rank's rows of a table every rank holds, row-balanced bounds (`shard_bounds`)."""
        bounds = shard_bounds(X.shape[0], world)
        return cls(X[bounds[rank]:bounds[rank + 1]], bounds, rank, world, group)

    @classmethod
    def local(cls, shards) -> "ShardedTable":
        """The shards as tensors of this process on one device (copied into 16-byte aligned rows; no IPC, no
        collective).  The kernel cannot tell these allocations from peer mappings."""
        from .functional import pad_table
        shards = list(shards)
        if not 1 <= len(shards) <= _lib.MAX_SHARDS:
            raise _lib.GnnError(f"ShardedTable: {len(shards)} shards, 1 to {_lib.MAX_SHARDS}")
        for t in shards:
            err = _table_refusal(t)
            if err:
                raise _lib.GnnError("ShardedTable: " + err)
        if len({(t.shape[1], t.dtype, t.device) for t in shards}) != 1:
            raise _lib.GnnError("ShardedTable: the shards differ in F, dtype or device")
        self = cls.__new__(cls)
        self.rank, self.world, self.group, self._buf = 0, 1, None, None
        self.bounds = [0]
        for t in shards:
            self.bounds.append(self.bounds[-1] + int(t.shape[0]))
        F, dtype = int(shards[0].shape[1]), shards[0].dtype
        self._set_layout(F, self._padded_ld(F, dtype), dtype, shards[0].device)
        self._keep = [pad_table(t.detach()) if t.shape[0] else None for t in shards]  # row stride self.ld
        self.abs_max = max([float(t.abs().max()) for t in self._keep if t is not None] or [0.0])
        self._make_desc([0 if t is None else t.data_ptr() for t in self._keep])
        return self

    @staticmethod
    def _padded_ld(F: int, dtype) -> int:
        per16 = 16 // _TABLE_DTYPES.get(dtype, 4)
        return (max(F, 0) + per16 - 1) // per16 * per16

    def _set_layout(self, F, ld, dtype, device):
        self.F, self.ld, self.dtype, self.device = int(F), int(ld), dtype, torch.device(device)
        self.shape = torch.Size((self.bounds[-1], self.F))
        self.requires_grad = False

    def _make_desc(self, ptrs):
        d = _lib.ShardedTableDesc()
        d.struct_size = C.sizeof(_lib.ShardedTableDesc)
        d.n_shards = len(self.bounds) - 1
        for s, p in enumerate(ptrs):
            d.base[s] = p or None
        for s, b in enumerate(self.bounds):
            d.row_begin[s] = b
        self.desc = d

    @property
    def n_shards(self) -> int:
        return len(self.bounds) - 1

    def stride(self, dim: Optional[int] = None):
        return (self.ld, 1) if dim is None else (self.ld, 1)[dim]

    def close(self):
        """Unmap and free the shard buffers (collective for a table built across ranks, like
        PartitionedGraph.close)."""
        if self._buf is not None:
            # gathers are asynchronous: this rank's last ones may still read peer shards, and peers may still read
            # this rank's shard, so every rank finishes its work before any mapping is closed or buffer freed
            torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)
            self._buf.close()
            self._buf = None
        self._keep = []
        self.desc = None


# ---- training across ranks ------------------------------------------------------------------
# A model holds replicated weights and rank-local activations.  With the loss rule below, the SUM over the ranks of
# the per-rank gradients is the 1-GPU gradient, so one SUM all_reduce of the gradients before the optimizer step
# keeps the replicas identical (given identical initial weights: broadcast_parameters).

def broadcast_parameters(module: torch.nn.Module, group=None):
    """Send the parameters and buffers of the group's first rank to every rank (call once, before training)."""
    src = 0 if group is None else dist.get_global_rank(group, 0)
    with torch.no_grad():
        for t in list(module.parameters()) + list(module.buffers()):
            dist.broadcast(t.data, src=src, group=group)


def allreduce_gradients(module: torch.nn.Module, group=None):
    """SUM every parameter's .grad over the ranks: one all_reduce of the gradients flattened in parameter order
    (a missing .grad counts as zeros).  Call between backward() and optimizer.step().
    When any gradient is narrower than fp32 (a bf16 model), the flattened gradients are reduced in fp32 (or wider, if
    some gradient is) and each sum is rounded once to its parameter's dtype: a bf16 ring sum would round at every hop.
    A model whose gradients are all fp32 (or all fp64) is reduced as is."""
    params = [p for p in module.parameters() if p.requires_grad]
    if not params:
        return
    grads = [(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params]
    if all(g.dtype.itemsize >= 4 for g in grads):
        flat = torch.cat(grads)
    else:
        acc = torch.float32
        for g in grads:
            acc = torch.promote_types(acc, g.dtype)
        flat = torch.cat([g.to(acc) for g in grads])
    dist.all_reduce(flat, group=group)
    off = 0
    for p in params:
        n = p.numel()
        g = flat[off:off + n].view_as(p)
        if p.grad is None:
            p.grad = g.to(p.dtype, copy=True)
        else:
            p.grad.copy_(g)  # rounds once when the gradient is not fp32
        off += n


def global_count(n_local: int, device, group=None) -> int:
    """Σ over the ranks of n_local (e.g. the global number of training rows): one all_reduce."""
    t = torch.tensor([int(n_local)], dtype=torch.int64, device=device)
    dist.all_reduce(t, group=group)
    return int(t.item())


def partitioned_cross_entropy(logits_local: torch.Tensor, target_local: torch.Tensor, n_global: int) -> torch.Tensor:
    """The loss rule of partitioned training: Σ of the per-row cross-entropy over this rank's rows, divided by
    the GLOBAL row count (`global_count`).  The sum of these losses over the ranks is the mean cross-entropy over
    all rows — `nn.CrossEntropyLoss()(output[idx_train], labels[idx_train])` of the 1-GPU model — and the sum of
    their gradients (`allreduce_gradients`) is its gradient."""
    return torch.nn.functional.cross_entropy(logits_local, target_local, reduction="sum") / float(max(n_global, 1))
