"""Multi-GPU sharding of the MI step: one process per GPU, units partitioned by
pre-computed pair-count cost (longest-processing-time bin packing), NO
collective on the data path -- units are independent (SURVEY 8e).  The only
cross-unit step is the global ECDF / mip pass (giremi.py:415-429), which needs
every site's mean MI in one place: per-rank results are gathered to rank 0 and
put back into the reference's row order (unit -> pair).

local_run also splits a unit too deep for one GPU by rows of its pair grid, as
multigpu.DevicePool does in one process (multigpu.plan_pieces, the same plan on
every rank).  A piece reads the plane rows of the later pieces from the other
processes' devices, and the first piece's owner gathers every piece's MI slice
for the per-site pass, both through CUDA IPC handles (Batch.export_piece); only
those handles, a few hundred bytes, travel through object collectives.

torch.distributed is plumbing here (gather of result buffers); it works with
the "nccl" backend (device tensors) and with "gloo" (host tensors, used by the
CPU tests)."""
from __future__ import annotations

import numpy as np

import time

from . import api
from ._lib import PAIR_REC
from .api import partition_lpt, unit_costs
from .encode import PlaneBatch
from .multigpu import (MergedResult, merge_shards, piece_batch, place_pieces, plane_copies,  # noqa: F401
                       plan_pieces, row_order, upload_piece_rows)


def plan(units, world_size):
    """bin_of[unit], load[bin] for `world_size` GPUs."""
    return partition_lpt(unit_costs(units), world_size)


def local_shard(pb: PlaneBatch, rank, world_size):
    """(sub-batch of the units assigned to `rank`, their global indices ascending)."""
    bin_of, _ = plan(pb.units, world_size)
    index = np.nonzero(bin_of == rank)[0]
    return pb.subset(index), index


def _gather_bytes(buf: np.ndarray, dst, group, device):
    """Gathers one variable-length byte buffer per rank onto `dst` (list of
    numpy arrays there, None elsewhere)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    n = torch.tensor([buf.size], dtype=torch.int64, device=device)
    sizes = [torch.zeros(1, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(sizes, n, group=group)
    sizes = [int(s.item()) for s in sizes]
    cap = max(max(sizes), 1)
    mine = torch.zeros(cap, dtype=torch.uint8, device=device)
    if buf.size:
        mine[:buf.size] = torch.from_numpy(buf.copy()).to(device)
    parts = [torch.empty(cap, dtype=torch.uint8, device=device) for _ in range(world)] if rank == dst else None
    dist.gather(mine, parts, dst=dst, group=group)
    if rank != dst:
        return None
    return [p[:s].cpu().numpy() for p, s in zip(parts, sizes)]


def gather_to_rank0(pb_global: PlaneBatch, local_result, local_index, group=None, device="cpu"):
    """Collects every rank's StepResult on rank 0 and restores global order.

    pb_global is only used for its unit table (site offsets / counts); every
    rank holds it (descriptors are tiny), only rank 0 gets a MergedResult."""
    import torch.distributed as dist
    rank = dist.get_rank(group)
    world = dist.get_world_size(group)
    rec = np.ascontiguousarray(local_result.records)
    payloads = [
        rec.view(np.uint8).reshape(-1),
        np.ascontiguousarray(local_result.site_mean, dtype=np.float64).view(np.uint8).reshape(-1),
        np.ascontiguousarray(local_result.site_cnt, dtype=np.uint32).view(np.uint8).reshape(-1),
        np.ascontiguousarray(local_result.unit_rec_off, dtype=np.uint64).view(np.uint8).reshape(-1),
        np.ascontiguousarray(local_index, dtype=np.int64).view(np.uint8).reshape(-1),
    ]
    gathered = [_gather_bytes(p, 0, group, device) for p in payloads]
    if rank != 0:
        return None
    parts = []
    for r in range(world):
        off = gathered[3][r].view(np.uint64)
        index = gathered[4][r].view(np.int64)
        assert len(off) == len(index) + 1
        parts.append((index, gathered[0][r].view(PAIR_REC), gathered[1][r].view(np.float64),
                      gathered[2][r].view(np.uint32), off, None))
    # ranks hold ascending global indices and emit in (unit, i, j) order: the merge is index bookkeeping
    return merge_shards(pb_global.units, pb_global.n_sites, parts)


class LocalRun:
    """One rank's share of a split-aware step (local_run): `result` (api.StepResult, or None when the rank has no
    ordinary unit) of its ordinary units `index` (global, ascending); `pieces` [(unit, first row, end row, records,
    counts | None)] of split units it ran, records numbered as in the piece (i, j from its first row); `means`
    {unit: (site_mean, site_cnt)} of the split units whose first piece it holds.  Host times in ms: `shard_ms` of
    the ordinary units, `pieces_ms` of the piece batch from creation to results on the host (copies included),
    `split_means_ms` of the per-site passes; `piece_kernel_ms` is the piece batch's device time."""

    def __init__(self, result, index, pieces=(), means=None, shard_ms=0.0, pieces_ms=0.0, piece_kernel_ms=None,
                 split_means_ms=0.0):
        self.result, self.index = result, np.asarray(index, dtype=np.int64)
        self.pieces, self.means = list(pieces), dict(means or {})
        self.shard_ms, self.pieces_ms, self.piece_kernel_ms = shard_ms, pieces_ms, piece_kernel_ms
        self.split_means_ms = split_means_ms


def local_run(pb_global: PlaneBatch, rank, world, min_common, mode, ctx, group=None) -> LocalRun:
    """The step of `rank`'s share of pb_global on ctx, with deep units split over the ranks (plan_pieces, the same on
    every rank: nothing is exchanged to plan).  With no unit split it is local_shard + one mi_step_batched and makes
    no collective call.  Otherwise every rank of `group` must call it with the same arguments but its own rank and
    context: each builds the batch of its pieces and uploads their own rows, takes the rows after them from the
    ranks holding the later pieces (CUDA IPC: the handles go through all_gather_object), runs, and the owner of a
    unit's first piece computes its per-site means from every piece's MI slice.  No rank closes its piece batch
    before all are done with it (barrier)."""
    shards, pieces, splits = plan_pieces(pb_global.units, world)
    index = shards[rank]
    t0 = time.perf_counter()
    result = api.mi_step_batched(pb_global.subset(index), min_common, mode, ctx=ctx) if len(index) or not splits \
        else None
    run = LocalRun(result, index, shard_ms=1e3 * (time.perf_counter() - t0))
    if not splits:
        return run
    import torch.distributed as dist
    mine = pieces[rank]
    t0 = time.perf_counter()
    batch = piece_batch(ctx, pb_global, mine) if mine else None
    try:
        if batch is not None:
            upload_piece_rows(batch, pb_global, mine)
        exported = _export_pieces(batch, mine, world, group)
        for dst, k, q, src, n in plane_copies(pb_global.units, pieces)[rank]:
            if k == rank:
                batch.copy_planes_from(dst, batch, src, n)
            else:
                batch.copy_planes_from_ipc(dst, exported[k][q], src, n)
        if batch is not None:
            batch.run(min_common, mode)
            res = batch.download(copy=True)
            run.piece_kernel_ms = res.kernel_ms
            run.pieces = [(u, a, e, res.unit_records(q), res.unit_counts(q) if res.counts is not None else None)
                          for q, (u, a, e) in enumerate(mine)]
        run.pieces_ms = 1e3 * (time.perf_counter() - t0)
        exported = _export_pieces(batch, mine, world, group)         # again, after the run
        t0 = time.perf_counter()
        for u in splits:
            order = row_order(pieces, u)
            if order[0][2] != rank:
                continue
            S, off = int(pb_global.units['n_sites'][u]), int(pb_global.units['site_off'][u])
            run.means[u] = api.split_means_ipc(ctx, pb_global.site_flags[off:off + S],
                                               [exported[k][q] for _a, _e, k, q in order])
        run.split_means_ms = 1e3 * (time.perf_counter() - t0)
        dist.barrier(group=group)            # every import from this rank's batch is done
    finally:
        if batch is not None:
            batch.close()
    return run


def _export_pieces(batch, mine, world, group):
    """export_piece bytes of every rank's pieces [rank][position], each behind all its batch has queued so far."""
    import torch.distributed as dist
    out = [None] * world
    dist.all_gather_object(out, [batch.export_piece(q) for q in range(len(mine))], group=group)
    return out


def gather_run_to_rank0(pb_global: PlaneBatch, run: LocalRun, group=None, device="cpu"):
    """gather_to_rank0 for local_run: every rank's ordinary shard (with its 3x3 tables under EMIT_COUNTS), its
    pieces' records and tables and its split units' means reach rank 0, which merges them (merge_shards with the
    split units placed) into the result of one process's step over pb_global.  Only rank 0 gets a MergedResult;
    its split_units maps each split unit to [(rank, first row, end row)] of its pieces."""
    import torch.distributed as dist
    rank = dist.get_rank(group)
    world = dist.get_world_size(group)
    r = run.result
    n_local = len(run.index)

    def raw(a, dtype):
        return np.ascontiguousarray(a, dtype=dtype).view(np.uint8).reshape(-1)

    if r is None:
        shard = [np.empty(0, PAIR_REC), np.empty(0), np.empty(0, np.uint32), np.zeros(n_local + 1, np.uint64), None]
    else:
        shard = [r.records, r.site_mean, r.site_cnt, r.unit_rec_off, r.counts]
    pieces = run.pieces
    piece_rec = np.concatenate([p[3] for p in pieces]) if pieces else np.empty(0, PAIR_REC)
    with_counts = [p for p in pieces if p[4] is not None]
    piece_cnt = np.concatenate([np.asarray(p[4]).reshape(-1, 9) for p in with_counts]) if with_counts \
        else np.empty((0, 9), np.uint32)
    units = sorted(run.means)
    means = np.concatenate([run.means[u][0] for u in units]) if units else np.empty(0)
    cnts = np.concatenate([run.means[u][1] for u in units]) if units else np.empty(0, np.uint32)
    payloads = [raw(shard[0], PAIR_REC), raw(shard[1], np.float64), raw(shard[2], np.uint32),
                raw(shard[3], np.uint64), raw(run.index, np.int64),
                raw(shard[4] if shard[4] is not None else np.empty((0, 9)), np.uint32),
                raw(piece_rec, PAIR_REC), raw(piece_cnt, np.uint32), raw(means, np.float64), raw(cnts, np.uint32)]
    gathered = [_gather_bytes(p, 0, group, device) for p in payloads]
    # what the byte buffers hold: per piece (unit, first row, end row, rows, tables shipped); the means' units
    meta = ([(int(u), int(a), int(e), len(rec), c is not None) for u, a, e, rec, c in pieces],
            units, shard[4] is not None)
    metas = [None] * world if rank == 0 else None
    dist.gather_object(meta, metas, dst=0, group=group)
    if rank != 0:
        return None
    parts, split_pieces, split_means = [], [], {}
    for k in range(world):
        index = gathered[4][k].view(np.int64)
        if len(index):
            off = gathered[3][k].view(np.uint64)
            counts = gathered[5][k].view(np.uint32).reshape(-1, 9) if metas[k][2] else None
            parts.append((index, gathered[0][k].view(PAIR_REC), gathered[1][k].view(np.float64),
                          gathered[2][k].view(np.uint32), off, counts))
        rec, tab = gathered[6][k].view(PAIR_REC), gathered[7][k].view(np.uint32).reshape(-1, 9)
        at = tab_at = 0
        for u, a, e, n, has_counts in metas[k][0]:
            c = None
            if has_counts:
                c, tab_at = tab[tab_at:tab_at + n], tab_at + n
            split_pieces.append((k, u, a, e, rec[at:at + n], c))
            at += n
        mean, cnt = gathered[8][k].view(np.float64), gathered[9][k].view(np.uint32)
        at = 0
        for u in metas[k][1]:
            S = int(pb_global.units['n_sites'][u])
            split_means[u] = (mean[at:at + S], cnt[at:at + S])
            at += S
    return merge_shards(pb_global.units, pb_global.n_sites, parts, *place_pieces(split_pieces, split_means))
