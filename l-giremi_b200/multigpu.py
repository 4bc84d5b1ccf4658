"""One host process driving every GPU of the box (SURVEY 8b / 8e: "CUDA context only in the
parent"; north_star part 4).

The reference's CLI forks `-t` workers that each run the whole per-region analysis
(giremi.py:375-380).  With the MI step on GPUs the workers only extract and encode; the PARENT
owns the devices: it partitions the (footprint, strand) units of all chunks by pre-computed
pair-count cost (longest-processing-time bin packing, lgmi_partition_lpt), submits one shard per
GPU from a thread pool (the C-ABI calls release the GIL; a handle is used by one thread at a time),
and merges the results back into the reference's row order.  Units are independent:
no collective.  A unit whose cost alone exceeds a device's share is split by rows of its pair
grid into pieces on several devices (split_plan); its planes cross the host link once, in
row ranges, and each piece fetches the rows it also needs from the other pieces' devices.
`shard.py` is the same thing for one PROCESS per GPU (torch.distributed launches:
bench.py --gpus N); its local_run splits units the same way, the other processes' pieces reached
through CUDA IPC handles."""
from __future__ import annotations

from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import api
from ._lib import PAIR_REC
from .encode import PlaneBatch


class MergedResult:
    """Results of several shards put back in global unit order: the fields of api.StepResult
    that callers read (records, site_mean, site_cnt, unit_rec_off, counts).  split_units maps each
    unit that was split to its pieces [(device index, first row, end row)] in row order."""

    def __init__(self, records, site_mean, site_cnt, unit_rec_off, n_candidates, counts=None, shard_ms=None,
                 shard_units=None, split_units=None):
        self.records, self.site_mean, self.site_cnt = records, site_mean, site_cnt
        self.unit_rec_off, self.n_candidates, self.counts = unit_rec_off, n_candidates, counts
        self.n_records = len(records)
        self.shard_ms, self.shard_units, self.split_units = shard_ms, shard_units, split_units or {}

    def unit_records(self, unit):
        return self.records[int(self.unit_rec_off[unit]):int(self.unit_rec_off[unit + 1])]

    def unit_counts(self, unit):
        if self.counts is None:
            return np.zeros((0, 9), dtype=np.uint32)
        return self.counts[int(self.unit_rec_off[unit]):int(self.unit_rec_off[unit + 1])]


def place_pieces(pieces, means):
    """merge_shards' `split` and `split_units` arguments from the split units' pieces `pieces` = [(device, unit,
    first row, end row, records, counts | None)] in any order and their means {unit: (site_mean, site_cnt)}."""
    ps, units = sorted(pieces, key=lambda p: (p[1], p[2])), sorted({p[1] for p in pieces})
    split = [(u, [(a, rec, c) for _k, v, a, _e, rec, c in ps if v == u]) + tuple(means[u]) for u in units]
    return split, {u: [(k, a, e) for k, v, a, e, _r, _c in ps if v == u] for u in units}


def merge_shards(units, n_sites, parts, split=(), split_units=None) -> MergedResult:
    """`parts` = [(global unit indices ascending, records, site_mean, site_cnt, unit_rec_off, counts | None)]
    per shard, each in its own local order -> one result in global order.  `split` = [(global unit,
    [(first row, records, counts | None)] of its pieces in row order, site_mean, site_cnt)] for the units
    that were split (a piece's i and j count from its first row) and `split_units`, as place_pieces gives them."""
    n_units = len(units)
    site_mean = np.full(n_sites, np.nan)
    site_cnt = np.zeros(n_sites, dtype=np.uint32)
    per_unit = np.zeros(n_units, dtype=np.int64)
    site_off = units['site_off'].astype(np.int64)
    n_s = units['n_sites'].astype(np.int64)
    # a split unit: its pieces' rows back to back, i and j shifted to the unit's own site numbers
    joined = []
    for unit, pieces, mean, cnt in split:
        rec = np.concatenate([np.asarray(r) for _a, r, _c in pieces]) if pieces else np.empty(0, PAIR_REC)
        if len(rec):
            shift = np.concatenate([np.full(len(r), a, dtype=np.int64) for a, r, _c in pieces])
            rec['i'] = (rec['i'].astype(np.int64) + shift).astype(np.uint16)
            rec['j'] = (rec['j'].astype(np.int64) + shift).astype(np.uint16)
        cnts = None
        if any(c is not None for _a, _r, c in pieces):
            cnts = np.concatenate([np.asarray(c).reshape(-1, 9) for _a, r, c in pieces]) \
                if len(rec) else np.zeros((0, 9), dtype=np.uint32)
        per_unit[unit] = len(rec)
        a, n = int(site_off[unit]), int(n_s[unit])
        site_mean[a:a + n] = mean
        site_cnt[a:a + n] = cnt
        joined.append((int(unit), rec, cnts))
    for index, _rec, mean, cnt, off, _counts in parts:
        index = np.asarray(index, dtype=np.int64)
        per_unit[index] = np.diff(np.asarray(off).astype(np.int64))
        # the shard's sites are its units' sites back to back, in shard order
        ns = n_s[index]
        if ns.sum():
            dst = np.repeat(site_off[index] - np.concatenate(([0], np.cumsum(ns)[:-1])), ns) + np.arange(int(ns.sum()))
            site_mean[dst] = np.asarray(mean)[:len(dst)]
            site_cnt[dst] = np.asarray(cnt)[:len(dst)]
    unit_rec_off = np.zeros(n_units + 1, dtype=np.uint64)
    unit_rec_off[1:] = np.cumsum(per_unit)
    total = int(unit_rec_off[-1])
    records = np.empty(total, dtype=PAIR_REC)
    want_counts = any(p[5] is not None for p in parts) or any(c is not None for _u, _r, c in joined)
    counts = np.empty((total, 9), dtype=np.uint32) if want_counts else None
    for unit, rec, cnts in joined:
        a = int(unit_rec_off[unit])
        records[a:a + len(rec)] = rec
        records['unit'][a:a + len(rec)] = unit
        if counts is not None and cnts is not None:
            counts[a:a + len(rec)] = cnts
    for index, rec, _mean, _cnt, off, cnts in parts:
        index = np.asarray(index, dtype=np.int64)
        if not len(index):
            continue
        off = np.asarray(off).astype(np.int64)
        n = np.diff(off)
        # row r of the shard (unit k = its position in the shard) goes to unit_rec_off[index[k]] + (r - off[k])
        shift = np.repeat(unit_rec_off[index].astype(np.int64) - off[:-1], n)
        dst = shift + np.arange(int(n.sum()))
        rec = np.asarray(rec)
        records[dst] = rec
        records['unit'][dst] = np.repeat(index, n).astype(np.uint32)
        if counts is not None and cnts is not None and len(dst):
            counts[dst] = cnts
    return MergedResult(records, site_mean, site_cnt, unit_rec_off, int((n_s * (n_s - 1) // 2).sum()), counts,
                        split_units=split_units)


SPLIT_ROWS = 128   # piece boundaries fall on multiples of this many rows (lgmi_batch_create_rows)


def _rows_pairs(S, rows):
    """Pairs (i, j), i < j < S, with i < rows, for an array of row counts."""
    rows = np.asarray(rows, dtype=np.int64)
    return rows * S - rows * (rows + 1) // 2


def split_rows(S, m):
    """Row boundaries 0 = b_0 < ... < b_m = S of m pieces of a unit of S sites, at multiples of SPLIT_ROWS, with the
    largest piece's pair count as small as that granularity allows (the slowest device sets the time)."""
    S = int(S)
    ends = np.minimum(np.arange(1, -(-S // SPLIT_ROWS) + 1, dtype=np.int64) * SPLIT_ROWS, S)
    blocks = np.diff(np.concatenate(([0], _rows_pairs(S, ends))))    # pairs of each 128-row block
    nb = len(blocks)
    m = max(1, min(int(m), nb))

    def cut(cap):   # greedy: each piece takes blocks while it stays within cap, leaving one block per later piece
        bounds, t = [0], 0
        for p in range(m - 1):
            acc, t = blocks[t], t + 1
            while t < nb - (m - 1 - p) and acc + blocks[t] <= cap:
                acc, t = acc + blocks[t], t + 1
            bounds.append(int(ends[t - 1]))
        return bounds + [S], int(blocks[t:].sum())

    lo, hi = int(blocks.max()), int(blocks.sum())     # the smallest cap for which the last piece fits too
    while lo < hi:
        mid = (lo + hi) // 2
        if cut(mid)[1] <= mid:
            hi = mid
        else:
            lo = mid + 1
    return cut(lo)[0]


def split_plan(units, n_dev):
    """Which units to split, and how, for n_dev devices: {unit: row boundaries}.  A unit of more than
    SPLIT_ROWS sites whose cost (api.unit_costs) exceeds total / n_dev is cut into
    min(n_dev, ceil(cost * n_dev / total), ceil(S / SPLIT_ROWS)) pieces of about equal pair counts."""
    if n_dev < 2 or not len(units):
        return {}
    cost = api.unit_costs(units).astype(np.float64)
    total = cost.sum()
    S = units['n_sites'].astype(np.int64)
    out = {}
    for u in np.flatnonzero((S > SPLIT_ROWS) & (cost * n_dev > total)):
        m = min(n_dev, int(np.ceil(cost[u] * n_dev / total)), int(-(-S[u] // SPLIT_ROWS)))
        if m >= 2:
            out[int(u)] = split_rows(S[u], m)
    return out


def plan_pieces(units, n_dev):
    """LPT partition of the ordinary units and of the pieces of the split units together.  Returns
    (shards, pieces, splits): shards[k] the ascending ordinary units of device k, pieces[k] its pieces as
    (unit, first row, end row), splits the split_plan."""
    splits = split_plan(units, n_dev)
    whole = np.array([u for u in range(len(units)) if u not in splits], dtype=np.int64)
    items = [(int(u), 0, 0) for u in whole]
    cost = [api.unit_costs(units[whole])] if len(whole) else []
    chunk = 64
    for u, b in splits.items():
        S, R = int(units['n_sites'][u]), int(units['n_reads'][u])
        for a, e in zip(b[:-1], b[1:]):
            items.append((u, a, e))
            cost.append(np.array([(_rows_pairs(S, e) - _rows_pairs(S, a)) * ((R + chunk - 1) // chunk)], np.uint64))
    bin_of, _load = api.partition_lpt(np.concatenate(cost) if cost else np.zeros(0, np.uint64), n_dev)
    shards = [whole[bin_of[:len(whole)] == k] for k in range(n_dev)]
    pieces = [[items[t] for t in range(len(whole), len(items)) if bin_of[t] == k] for k in range(n_dev)]
    return shards, pieces, splits


def piece_units(units, pieces):
    """The descriptor table of the batch of `pieces` [(unit, first row, end row)] of `units`: each piece the suffix
    unit of sites [a, S) of its unit, planes and sites back to back."""
    desc = np.zeros(len(pieces), dtype=units.dtype)
    word = site = 0
    for q, (u, a, _e) in enumerate(pieces):
        S, W = int(units['n_sites'][u]), int(units['row_words'][u])
        desc[q] = (word, S - a, int(units['n_reads'][u]), W, site)
        word += 3 * (S - a) * W
        site += S - a
    return desc


def row_order(pieces, unit):
    """The pieces of `unit` in plan_pieces' `pieces` as (first row, end row, device, position in its batch), in row
    order: the first one's device computes the unit's per-site means."""
    return sorted((a, e, k, q) for k, mine in enumerate(pieces) for q, (u, a, e) in enumerate(mine) if u == unit)


def plane_copies(units, pieces):
    """For each device k, in issue order, the copies [(dst_word, src_device, src_position, src_word, n_words)] that
    bring each piece of pieces[k] the rows after its own, from the later pieces of its unit, once all own rows are
    uploaded (upload_piece_rows).  src_word is lgmi_piece_export's plane_word of the source, n_words its plane_words."""
    off = [piece_units(units, mine)['plane_off'] for mine in pieces]
    every = [(ks, qs, v, c, ce) for ks, theirs in enumerate(pieces) for qs, (v, c, ce) in enumerate(theirs)]
    copies = [[] for _ in pieces]
    for k, q, u, a, e in every:
        W = int(units['row_words'][u])
        copies[k] += [(int(off[k][q]) + 3 * (c - a) * W, ks, qs, int(off[ks][qs]), 3 * (ce - c) * W)
                      for ks, qs, v, c, ce in every if v == u and c >= e]
    return copies


def piece_batch(ctx, pb: PlaneBatch, pieces):
    """The batch of `pieces` [(unit, first row, end row)] of pb's units on ctx (api.Batch with row limits): each the
    suffix unit of sites [a, S) of its unit (piece_units), with row limit e - a.  Its planes are left empty: they come
    from upload_piece_rows and from copies of the other pieces' rows (plane_copies)."""
    desc = piece_units(pb.units, pieces)
    off, S = pb.units['site_off'], pb.units['n_sites']
    flags = np.concatenate([pb.site_flags[int(off[u]) + a:int(off[u]) + int(S[u])] for u, a, _e in pieces])
    # (np.empty: the batch only reads the planes' size; their words come from upload_rows / copies)
    words = int((3 * desc['n_sites'].astype(np.int64) * desc['row_words']).sum())
    return api.Batch(ctx, PlaneBatch(desc, np.empty(words, dtype=np.uint32), flags),
                     row_limit=[e - a for _u, a, e in pieces])


def upload_piece_rows(batch, pb: PlaneBatch, pieces):
    """Uploads each piece's own rows [a, e) of pb's planes (and the flags) to its place in piece_batch's batch."""
    for q, (u, a, e) in enumerate(pieces):
        W, base = int(pb.units['row_words'][u]), int(pb.units['plane_off'][u])
        batch.upload_rows(int(batch.pb.units['plane_off'][q]), pb.planes[base + 3 * a * W:base + 3 * e * W])


class DevicePool:
    """Contexts on `devices` (default: every visible GPU), owned by the calling process."""

    def __init__(self, devices=None):
        if devices is None:
            import os
            env = os.environ.get("LGMI_DEVICES", "")                  # e.g. "0,1,2,3"; default: every visible GPU
            devices = [int(d) for d in env.split(",") if d != ""] or list(range(max(1, api.device_count())))
        self.devices = [int(d) for d in devices]
        self.contexts = [api.Context(d) for d in self.devices]       # raises without a GPU: no CPU path
        self._threads = ThreadPoolExecutor(max_workers=len(self.devices)) if len(self.devices) > 1 else None

    def __len__(self):
        return len(self.devices)

    def close(self):
        if self._threads is not None:
            self._threads.shutdown()
            self._threads = None
        for c in self.contexts:
            c.close()
        self.contexts = []

    def run(self, pb: PlaneBatch, min_common_reads=5, mode=api.MODE_HET_ONLY):
        """The MI step of `pb` over all devices; same result as api.mi_step_batched on one."""
        n_dev = len(self.devices)
        shards, pieces, splits = plan_pieces(pb.units, n_dev)
        self.last_piece_ms, self.last_split_means_ms = [None] * n_dev, None   # (what the last run measured)
        if not splits and (n_dev == 1 or pb.n_units < 2 * n_dev):
            return api.mi_step_batched(pb, min_common_reads, mode, ctx=self.contexts[0])
        import time
        batches = self._piece_batches(pb, pieces) if splits else [None] * n_dev

        def work(k):
            index, b = shards[k], batches[k]
            t0 = time.perf_counter()
            res = None
            if b is not None:
                b.run(min_common_reads, mode)
            if len(index):
                res = api.mi_step_batched(pb.subset(index), min_common_reads, mode, ctx=self.contexts[k])
            mine = []
            if b is not None:
                r = b.download(copy=True)
                self.last_piece_ms[k] = r.kernel_ms
                mine = [(k, u, a, e, r.unit_records(q), r.unit_counts(q) if r.counts is not None else None)
                        for q, (u, a, e) in enumerate(pieces[k])]
            return res, mine, 1e3 * (time.perf_counter() - t0)

        try:
            done = list(self._threads.map(work, range(n_dev)))
            means = {}
            t0 = time.perf_counter()
            for u in splits:
                order = row_order(pieces, u)
                S, off = int(pb.units['n_sites'][u]), int(pb.units['site_off'][u])
                means[u] = api.split_means(self.contexts[order[0][2]], pb.site_flags[off:off + S],
                                           [(batches[k], q) for _a, _e, k, q in order])
            self.last_split_means_ms = 1e3 * (time.perf_counter() - t0)
        finally:
            for b in batches:
                if b is not None:
                    b.close()
        parts = [(shards[k], r.records, r.site_mean, r.site_cnt, r.unit_rec_off, r.counts)
                 for k, (r, _p, _ms) in enumerate(done) if r is not None]
        merged = merge_shards(pb.units, pb.n_sites, parts, *place_pieces([p for r in done for p in r[1]], means))
        merged.shard_ms = [ms for _r, _p, ms in done]
        # units per device; a split unit counts on the device of its first piece, which computes its means
        owners = [row_order(pieces, u)[0][2] for u in splits]
        merged.shard_units = [len(s) + owners.count(k) for k, s in enumerate(shards)]
        return merged

    def _piece_batches(self, pb, pieces):
        """One batch of pieces per device (None where there is none), planes in place: each piece's own rows
        uploaded from the host, the rows after them copied from the devices of the later pieces of its unit."""
        batches = [piece_batch(ctx, pb, mine) if mine else None for ctx, mine in zip(self.contexts, pieces)]
        try:
            # the host link once: every piece uploads its own rows, one thread per device
            list(self._threads.map(lambda k: upload_piece_rows(batches[k], pb, pieces[k]),
                                   [k for k, mine in enumerate(pieces) if mine]))
            # then, from this thread, each piece's rows after its own from the pieces that uploaded them: a copy
            # waits on an event recorded behind the upload already queued on the source's stream
            for k, copies in enumerate(plane_copies(pb.units, pieces)):
                for dst, ks, _qs, src, n in copies:
                    batches[k].copy_planes_from(dst, batches[ks], src, n)
        except BaseException:
            for b in batches:
                if b is not None:
                    b.close()
            raise
        return batches


_pool = None


def get_pool() -> DevicePool:
    """Process-wide pool over every visible GPU, created on first use (in the parent, after the
    extraction workers have been forked and have returned)."""
    global _pool
    if _pool is None or not _pool.contexts:
        _pool = DevicePool()
    return _pool
