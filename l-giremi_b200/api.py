"""Host-side mirror of the reference's MI interface, backed by liblgmi.so.

Same names, argument meaning, return shapes, row order and error behaviour as

  giremi.mutual_information.mismatch_pair_mutual_info        (:6-45)
  giremi.mutual_information.mean_mismatch_pair_mutual_info   (:48-60)
  giremi.stat.ecdf                                           (stat.py:7-29)

plus the batched step (`mi_step_batched`) that replaces the per-unit loop of
giremi.mismatch.region_mismatch_analysis (mismatch.py:387-404) with one submit.
Nothing here computes MI on the CPU; without the CUDA library or a GPU every
entry point raises."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import (MODE_ALL_PAIRS, MODE_COMPACT_OUTPUT, MODE_EMIT_COUNTS, MODE_HET_ONLY, MODE_GRAPH, MODE_SKIP_NONHET,
                   MODE_SPLIT_RECORDS, MODE_TIGHT_INPUT,
                   PAIR_REC, SITE_TYPE_CODE, LgmiError, Result, array_at, check, ptr)
from .encode import PlaneBatch, encode_batch, encode_mismatches, pack_units


class Context:
    """One liblgmi handle == one process on one GPU."""

    def __init__(self, device=0):
        self._lib = _lib.load()
        h = C.c_void_p()
        rc = self._lib.lgmi_create(int(device), C.byref(h))
        if rc != 0:
            msg = self._lib.lgmi_last_error(None)
            raise LgmiError(rc, msg.decode() if msg else "")
        self.handle = h
        self.device = int(device)

    def close(self):
        if getattr(self, "handle", None):
            self._lib.lgmi_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr):
        """Launch on a caller-owned cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream)."""
        check(self._lib.lgmi_set_stream(self.handle, C.c_void_p(cuda_stream_ptr or 0)), self.handle)

    def set_dense_threshold(self, min_sites, min_reads):
        """Units at least this large take the int8 tensor-core path (batches created afterwards)."""
        check(self._lib.lgmi_set_dense_threshold(self.handle, int(min_sites), int(min_reads)), self.handle)

    def set_dense_path(self, blocks):
        """Deep units: 4 = four Gram blocks + "other" cells from the listed reads while those are rare (decided on
        the device per unit and run; default), 9 = always nine blocks (lgmi_set_dense_path)."""
        check(self._lib.lgmi_set_dense_path(self.handle, int(blocks)), self.handle)

    def set_tile_path(self, tensor_cores):
        """Mid-depth units counted on the tensor cores (True / non-zero, default: k_tile_gram_ws + k_tile_finish)
        or by tiled popcount (False / 0: k_tile_mi)."""
        check(self._lib.lgmi_set_tile_path(self.handle, int(tensor_cores)), self.handle)

    @property
    def launch_count(self):
        return int(self._lib.lgmi_launch_count(self.handle))

    def pinned_empty(self, shape, dtype):
        """numpy array backed by cudaHostAlloc memory (kept alive by the returned object)."""
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        p = C.c_void_p()
        check(self._lib.lgmi_pinned_alloc(self.handle, max(1, count * dtype.itemsize), C.byref(p)), self.handle)
        arr = array_at(p.value, dtype, count).reshape(shape) if count else np.empty(shape, dtype)
        return _Pinned(self, p.value, arr)


class _Pinned:
    def __init__(self, ctx, address, array):
        self.ctx, self.address, self.array = ctx, address, array

    def free(self):
        if self.address and self.ctx.handle:
            self.ctx._lib.lgmi_pinned_free(self.ctx.handle, C.c_void_p(self.address))
        self.address = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


_default_ctx = None


def device_count() -> int:
    """CUDA devices this process sees (0 without a driver)."""
    return int(_lib.load().lgmi_device_count())


def default_device() -> int:
    """Which GPU a process gets when nobody said: LGMI_DEVICE, else LOCAL_RANK (torchrun), else -- inside a
    multiprocessing pool worker, as when the reference's `l-giremi -t N` runs the name-level drop-ins in its
    forked workers (giremi.py:375-380) -- worker index modulo the number of GPUs, so that N workers use
    min(N, 8) GPUs instead of all sharing device 0."""
    import multiprocessing as mp
    import os
    for key in ("LGMI_DEVICE", "LOCAL_RANK"):
        if os.environ.get(key, "") != "":
            return int(os.environ[key])
    ident = getattr(mp.current_process(), "_identity", ())
    if ident:
        return (int(ident[0]) - 1) % max(1, device_count())
    return 0


def get_context(device=None) -> Context:
    """Process-wide context, created on first use (after any fork: CUDA must be
    initialised in the process that uses it)."""
    global _default_ctx
    if _default_ctx is None or _default_ctx.handle is None:
        _default_ctx = Context(default_device() if device is None else device)
    return _default_ctx


class StepResult:
    """Host view of one batch's outputs (copies: safe after the batch is reused)."""

    def __init__(self, res: Result, n_units, copy=True):
        self.n_candidates = int(res.n_candidates)
        self.n_evaluated = int(res.n_evaluated)
        self.n_records = int(res.n_records)
        self.kernel_ms = float(res.kernel_ms)
        self.pairs_kernel_ms = float(res.pairs_kernel_ms)
        self.dense_kernel_ms = float(res.dense_kernel_ms)
        self.n_dense_units = int(res.n_dense_units)
        self.n_dense_four = int(res.n_dense_four)
        self.dense_macs = int(res.dense_macs)
        self.gram_kernel_ms = float(res.gram_kernel_ms)
        self.gram_macs = int(res.gram_macs)
        off = array_at(res.unit_rec_off, np.uint64, n_units + 1)
        self.rec_mi = self.rec_ij = None
        if not res.records and res.rec_mi:                   # MODE_SPLIT_RECORDS: two arrays instead of 16-byte rows
            self.rec_mi = array_at(res.rec_mi, np.float64, self.n_records)
            # (i | j << 16 as uint32, or -- MODE_COMPACT_OUTPUT, no unit above 256 sites -- i | j << 8 as uint16)
            self.rec_ij = array_at(res.rec_ij, np.uint16 if int(res.rec_ij_bytes) == 2 else np.uint32, self.n_records)
            if copy:
                self.rec_mi, self.rec_ij = self.rec_mi.copy(), self.rec_ij.copy()
            rec = None
        else:
            rec = array_at(res.records, PAIR_REC, self.n_records)
        mean = array_at(res.site_mean, np.float64, int(res.n_sites))
        cnt = array_at(res.site_cnt, np.uint32, int(res.n_sites)) if res.site_cnt else None
        counts = array_at(res.counts, np.uint32, self.n_records * 9).reshape(-1, 9) if res.counts else None
        if copy:
            rec = rec.copy() if rec is not None else None
            mean, off = mean.copy(), off.copy()
            cnt = cnt.copy() if cnt is not None else None
            counts = counts.copy() if counts is not None else None
        self._records, self.site_mean, self._site_cnt, self.unit_rec_off, self.counts = rec, mean, cnt, off, counts
        self._site_off = None                                # per-unit first site: set by the owner of the unit table

    @property
    def site_cnt(self):
        """Rows each site appears in.  Not shipped under MODE_COMPACT_OUTPUT: then counted here from the
        rows (needs the unit table's site offsets, which Pipeline.step attaches)."""
        if self._site_cnt is None:
            if self._site_off is None:
                raise ValueError("site_cnt was not downloaded (MODE_COMPACT_OUTPUT) and the unit table is unknown")
            rec = self.records
            base = self._site_off[rec['unit']]
            n = len(self.site_mean)
            self._site_cnt = (np.bincount(base + rec['i'], minlength=n) +
                              np.bincount(base + rec['j'], minlength=n)).astype(np.uint32)
        return self._site_cnt

    @property
    def records(self):
        """Rows as (unit, i, j, mi); assembled on the host from the split arrays when the step
        ran with MODE_SPLIT_RECORDS."""
        if self._records is None:
            rec = np.empty(self.n_records, dtype=PAIR_REC)
            rec['mi'] = self.rec_mi
            if self.rec_ij.dtype == np.uint16:
                rec['i'], rec['j'] = self.rec_ij & 0xff, self.rec_ij >> 8
            else:
                rec['i'], rec['j'] = self.rec_ij & 0xffff, self.rec_ij >> 16
            n = np.diff(self.unit_rec_off.astype(np.int64))
            rec['unit'] = np.repeat(np.arange(len(n), dtype=np.uint32), n)
            self._records = rec
        return self._records

    def unit_records(self, unit):
        a, b = int(self.unit_rec_off[unit]), int(self.unit_rec_off[unit + 1])
        return self.records[a:b]

    def unit_counts(self, unit):
        a, b = int(self.unit_rec_off[unit]), int(self.unit_rec_off[unit + 1])
        if self.counts is None and self.n_records == 0:      # nothing survived: the library returns no table buffer
            return np.zeros((0, 9), dtype=np.uint32)
        return self.counts[a:b]


class Batch:
    """Device-side batch: create once, then upload / run / download repeatedly.

    row_limit (one entry per unit, or None): a unit with a non-zero entry is a piece of a split unit -- the suffix
    of sites [a, S) of a unit, of which only the pairs (i, j) with i < row_limit are evaluated and emitted
    (lgmi_batch_create_rows).  Its site_mean / site_cnt entries stay NaN / 0: split_means gives them."""

    def __init__(self, ctx: Context, pb: PlaneBatch, row_limit=None):
        self.ctx, self.pb = ctx, pb
        self._lib = ctx._lib
        h = C.c_void_p()
        if row_limit is None:
            check(self._lib.lgmi_batch_create(ctx.handle, ptr(pb.units), pb.n_units, pb.planes.size,
                                              pb.n_sites, C.byref(h)), ctx.handle)
        else:
            self.row_limit = np.ascontiguousarray(row_limit, dtype=np.uint32)
            assert self.row_limit.size == pb.n_units
            check(self._lib.lgmi_batch_create_rows(ctx.handle, ptr(pb.units), pb.n_units, ptr(self.row_limit),
                                                   pb.planes.size, pb.n_sites, C.byref(h)), ctx.handle)
        self.handle = h

    def upload(self, planes=None, site_flags=None):
        planes = self.pb.planes if planes is None else planes
        site_flags = self.pb.site_flags if site_flags is None else site_flags
        assert planes.dtype == np.uint32 and planes.size == self.pb.planes.size
        assert site_flags.dtype == np.uint8 and site_flags.size == self.pb.n_sites
        self._keep = (planes, site_flags)
        check(self._lib.lgmi_batch_upload(self.handle, ptr(planes), ptr(site_flags)), self.ctx.handle)

    def upload_rows(self, word_begin, words, site_flags=None):
        """Uploads the host words `words` to the plane words [word_begin, word_begin + len(words)) of the batch,
        and every flag byte; the rest of the planes comes from elsewhere, e.g. copy_planes_from.  The host arrays
        must stay untouched until the next sync."""
        words = np.ascontiguousarray(words, dtype=np.uint32)
        site_flags = self.pb.site_flags if site_flags is None else site_flags
        assert site_flags.dtype == np.uint8 and site_flags.size == self.pb.n_sites
        self._keep_rows = getattr(self, "_keep_rows", []) + [words, site_flags]
        check(self._lib.lgmi_batch_upload_rows(self.handle, ptr(words), int(word_begin), int(word_begin) + words.size,
                                               ptr(site_flags)), self.ctx.handle)

    def copy_planes_from(self, dst_word, src: "Batch", src_word, n_words):
        """Device-to-device copy of n_words plane words of `src` (any device) to dst_word of this batch, behind
        whatever src's stream has queued (lgmi_batch_copy_planes)."""
        check(self._lib.lgmi_batch_copy_planes(self.handle, int(dst_word), src.handle, int(src_word), int(n_words)),
              self.ctx.handle)

    def export_piece(self, k) -> bytes:
        """Piece k of this batch as the bytes another process imports (lgmi_piece_export: CUDA IPC handles of the
        batch's blocks and of an event recorded behind everything queued so far, i.e. the upload or the run).  The
        batch must outlive every importer's use of them."""
        out = _lib.PieceIpc()
        check(self._lib.lgmi_piece_export(self.handle, int(k), C.byref(out)), self.ctx.handle)
        return bytes(out)

    def copy_planes_from_ipc(self, dst_word, piece: bytes, src_word, n_words):
        """copy_planes_from with the source a piece exported by another process (export_piece's bytes): n_words
        plane words of its batch from src_word, behind its event (lgmi_batch_copy_planes_ipc)."""
        src = _lib.PieceIpc.from_buffer_copy(piece)
        check(self._lib.lgmi_batch_copy_planes_ipc(self.handle, int(dst_word), C.byref(src), int(src_word),
                                                   int(n_words)), self.ctx.handle)

    def run(self, min_common, mode=MODE_ALL_PAIRS):
        check(self._lib.lgmi_batch_run(self.handle, int(min_common), int(mode)), self.ctx.handle)

    def sync(self) -> Result:
        res = Result()
        check(self._lib.lgmi_batch_sync(self.handle, C.byref(res)), self.ctx.handle)
        return res

    def download(self, copy=True) -> StepResult:
        res = Result()
        check(self._lib.lgmi_batch_download(self.handle, C.byref(res)), self.ctx.handle)
        return StepResult(res, self.pb.n_units, copy=copy)

    def algorithmic_bytes(self) -> int:
        v = C.c_uint64()
        check(self._lib.lgmi_batch_algorithmic_bytes(self.handle, C.byref(v)), self.ctx.handle)
        return int(v.value)

    def device_ptrs(self):
        p = [C.c_void_p() for _ in range(4)]
        check(self._lib.lgmi_batch_device_ptrs(self.handle, *[C.byref(x) for x in p]), self.ctx.handle)
        return tuple(x.value for x in p)

    def close(self):
        if getattr(self, "handle", None):
            self._lib.lgmi_batch_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            if self.ctx.handle:
                self.close()
        except Exception:
            pass


class Pipeline:
    """Host-buffers-in / host-buffers-out step with the H2D copy, the kernels and
    the D2H copy of consecutive groups of units overlapped (lgmi_pipeline_*).
    Same result as Batch.upload + run + download."""

    def __init__(self, ctx: Context, pb: PlaneBatch, n_chunks=4):
        self.ctx, self.pb = ctx, pb
        self._lib = ctx._lib
        h = C.c_void_p()
        check(self._lib.lgmi_pipeline_create(ctx.handle, ptr(pb.units), pb.n_units, pb.planes.size, pb.n_sites,
                                             int(n_chunks), C.byref(h)), ctx.handle)
        self.handle = h

    def _inputs(self, mode, planes, site_flags, packed, tight):
        packed = packed or tight
        if planes is None:
            planes = self.pb.packed2(tight=tight) if packed else self.pb.planes
        site_flags = self.pb.site_flags if site_flags is None else site_flags
        if tight:
            mode |= MODE_TIGHT_INPUT
            want = int((2 * self.pb.units['n_sites'].astype(np.int64) * ((self.pb.units['n_reads'].astype(np.int64) + 31) // 32)).sum())
        else:
            want = self.pb.planes.size // 3 * 2 if packed else self.pb.planes.size
        assert planes.dtype == np.uint32 and planes.size == want
        assert site_flags.dtype == np.uint8 and site_flags.size == self.pb.n_sites
        return planes, site_flags, mode, packed

    def step(self, min_common, mode=MODE_HET_ONLY, planes=None, site_flags=None, copy=True, packed=False,
             tight=False) -> StepResult:
        """One pipelined step.  packed=True: `planes` is the two-plane form (PlaneBatch.packed2(),
        two thirds of the bytes); tight=True: its rows without the 128-read padding
        (PlaneBatch.packed2(tight=True), MODE_TIGHT_INPUT); mode | MODE_SPLIT_RECORDS: rows come back as
        rec_mi / rec_ij; mode | MODE_COMPACT_OUTPUT: the same with 2-byte (i, j) entries where no unit has
        more than 256 sites, and no per-site count over the wire."""
        self.begin(min_common, mode, planes, site_flags, packed, tight)
        return self.finish(copy=copy)

    def begin(self, min_common, mode=MODE_HET_ONLY, planes=None, site_flags=None, packed=False, tight=False):
        """First half of step(): queues the uploads and kernels of every group and returns
        (lgmi_pipeline_begin*).  The input arrays must stay alive and untouched until finish()."""
        planes, site_flags, mode, packed = self._inputs(mode, planes, site_flags, packed, tight)
        fn = self._lib.lgmi_pipeline_begin_packed if packed else self._lib.lgmi_pipeline_begin
        check(fn(self.handle, ptr(planes), ptr(site_flags), int(min_common), int(mode)), self.ctx.handle)
        self._pending = (planes, site_flags)

    def collect(self):
        """First part of finish() on its own: waits for the groups' kernels and queues their downloads
        (lgmi_pipeline_collect); the previous result's arrays are rewritten from here on."""
        check(self._lib.lgmi_pipeline_collect(self.handle), self.ctx.handle)

    def finish(self, copy=True) -> StepResult:
        """Second half of step(): waits for the groups, copies the rows back (lgmi_pipeline_finish)."""
        res = Result()
        check(self._lib.lgmi_pipeline_finish(self.handle, C.byref(res)), self.ctx.handle)
        self._pending = None
        out = StepResult(res, self.pb.n_units, copy=copy)
        out._site_off = self.pb.units['site_off'].astype(np.int64)
        return out

    def close(self):
        if getattr(self, "handle", None):
            self._lib.lgmi_pipeline_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            if self.ctx.handle:
                self.close()
        except Exception:
            pass


def stream_schedule(n_steps, depth, collect=True):
    """The order of calls that keeps `depth` steps in flight over `depth` pipelines (step k on pipeline
    k % depth): yields ('begin', k), ('collect', k), ('finish', k).  After begin(k) the downloads of step
    k - depth + 2 are queued (collect) and step k - depth + 1 is waited for (finish), so that both directions
    of the host link always have work queued; the tail finishes what is left, in order."""
    depth = max(1, int(depth))
    for k in range(n_steps):
        yield 'begin', k
        if collect and depth > 2 and k >= depth - 2:
            yield 'collect', k - depth + 2
        if k >= depth - 1:
            yield 'finish', k - depth + 1
    for k in range(max(0, n_steps - depth + 1), n_steps):
        yield 'finish', k


def stream_steps(pipes, inputs, min_common, mode=MODE_HET_ONLY, copy=True, packed=False, tight=False, collect=True):
    """Batch after batch through the pipelined step with len(pipes) steps in flight (stream_schedule): `pipes`
    are Pipeline objects built for the same unit table, `inputs` an iterable of (planes, site_flags) host arrays
    (pinned for the copies to be asynchronous; they must stay untouched until their step has been yielded).
    Yields (k, StepResult) in input order; each result is the synchronous step's, bit for bit.  With copy=False
    a result's arrays are only valid until the generator is advanced again."""
    depth = len(pipes)
    held = {}                                                # step -> its input arrays, alive until finished
    it = iter(inputs)
    k = 0
    for planes, site_flags in it:
        held[k] = (planes, site_flags)
        pipes[k % depth].begin(min_common, mode, planes, site_flags, packed=packed, tight=tight)
        if collect and depth > 2 and k >= depth - 2:
            pipes[(k - depth + 2) % depth].collect()
        if k >= depth - 1:
            j = k - depth + 1
            res = pipes[j % depth].finish(copy=copy)
            del held[j]
            yield j, res
        k += 1
    for j in range(max(0, k - depth + 1), k):
        res = pipes[j % depth].finish(copy=copy)
        del held[j]
        yield j, res


def split_means(ctx: Context, site_flags, pieces):
    """Per-site mean MI and row count of a split unit (lgmi_split_means): `pieces` = [(Batch, unit index in it)]
    in row order, each already run; `site_flags` the unit's flag bytes.  The same bits as an unsplit run."""
    flags = np.ascontiguousarray(site_flags, dtype=np.uint8)
    n = flags.size
    handles = (C.c_void_p * len(pieces))(*[b.handle.value for b, _k in pieces])
    units = np.array([k for _b, k in pieces], dtype=np.uint32)
    mean = np.empty(n, dtype=np.float64)
    cnt = np.empty(n, dtype=np.uint32)
    check(ctx._lib.lgmi_split_means(ctx.handle, n, ptr(flags), len(pieces), C.cast(handles, C.c_void_p), ptr(units),
                                    ptr(mean), ptr(cnt)), ctx.handle)
    return mean, cnt


def split_means_ipc(ctx: Context, site_flags, pieces):
    """split_means over pieces in any process: `pieces` = export_piece bytes of every piece in row order, each
    exported after its run (lgmi_split_means_ipc).  The same bits as split_means."""
    flags = np.ascontiguousarray(site_flags, dtype=np.uint8)
    n = flags.size
    arr = (_lib.PieceIpc * len(pieces))(*[_lib.PieceIpc.from_buffer_copy(p) for p in pieces])
    mean = np.empty(n, dtype=np.float64)
    cnt = np.empty(n, dtype=np.uint32)
    check(ctx._lib.lgmi_split_means_ipc(ctx.handle, n, ptr(flags), len(pieces), C.cast(arr, C.c_void_p), ptr(mean),
                                        ptr(cnt)), ctx.handle)
    return mean, cnt


PIPELINE_MIN_CANDIDATES = 2_000_000   # below this one submit is as fast as a pipelined one


def mi_step_batched(pb: PlaneBatch, min_common_reads=5, mode=MODE_HET_ONLY, ctx=None, n_chunks=None) -> StepResult:
    """All units of `pb` in one submit: pair MI -> het filter -> per-site mean
    (mismatch.py:387-404 for every unit at once).  Host buffers in, host
    buffers out.  Large batches go through the pipelined step (copies and
    kernels overlapped); the result is the same either way."""
    ctx = ctx or get_context()
    if n_chunks is None:
        n_chunks = 4 if pb.n_candidates >= PIPELINE_MIN_CANDIDATES and pb.n_units >= 16 else 1
    if n_chunks > 1:
        p = Pipeline(ctx, pb, n_chunks)
        try:
            return p.step(min_common_reads, mode, copy=True)
        finally:
            p.close()
    b = Batch(ctx, pb)
    try:
        b.upload()
        b.run(min_common_reads, mode)
        return b.download(copy=True)
    finally:
        b.close()


# --------------------------------------------------------------------------- #
# drop-in functions (reference signatures)
# --------------------------------------------------------------------------- #
def mismatch_pair_mutual_info(mismatches, min_common_reads=5):
    """Drop-in for giremi.mutual_information.mismatch_pair_mutual_info (:6-45):
    returns ``[[p1, type1, p2, type2, mi], ...]`` in ``combinations`` order for
    every pair sharing at least ``min_common_reads`` reads."""
    if len(mismatches) < 2:
        return []
    eu = encode_mismatches(mismatches)
    res = mi_step_batched(pack_units([eu]), min_common_reads, MODE_ALL_PAIRS)
    rec = res.records
    if eu.bad_sites and len(rec):
        bad = np.fromiter(eu.bad_sites, dtype=np.int64)
        if np.isin(rec['i'], bad).any() or np.isin(rec['j'], bad).any():
            raise IndexError('list index out of range')   # mutual_information.py:30/32
    pos, typ = eu.positions, eu.types
    return [[pos[i], typ[i], pos[j], typ[j], mi]
            for i, j, mi in zip(rec['i'].tolist(), rec['j'].tolist(), rec['mi'].tolist())]


def mean_mismatch_pair_mutual_info(mismatch_pair_mi):
    """Drop-in for giremi.mutual_information.mean_mismatch_pair_mutual_info
    (:48-60): ``[[pos, mean], ...]`` in first-appearance order.  The grouping
    is index bookkeeping on the host; the summation and division run on the
    device with CPython's float-sum semantics."""
    order, values = {}, []
    for p1, _t1, p2, _t2, mi in mismatch_pair_mi:
        for p in (p1, p2):
            k = order.get(p)
            if k is None:
                k = order[p] = len(values)
                values.append([])
            values[k].append(mi)
    if not values:
        return []
    offsets = np.zeros(len(values) + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([len(v) for v in values])
    flat = np.array([x for v in values for x in v], dtype=np.float64)
    out = np.empty(len(values), dtype=np.float64)
    ctx = get_context()
    check(ctx._lib.lgmi_site_mean_csr(ctx.handle, ptr(offsets), ptr(flat), len(values), ptr(out)), ctx.handle)
    return [[p, m] for p, m in zip(order.keys(), out.tolist())]


def ecdf(x):
    """Drop-in for giremi.stat.ecdf (stat.py:7-29): returns a callable mapping a
    sample (scalar or array) to ``y[searchsorted(sort(x), sample)]``.

    The sort and the ordinates ``[0] ++ linspace(1/n, 1, n)`` are computed ONCE, on the
    device, when the callable is built (lgmi_ecdf_table); evaluating it is an index
    into that table.  The CLI calls it once per row through DataFrame.apply
    (giremi.py:424-428): a device round trip per call would be far slower than the
    reference.  Large sample arrays go to the device in one launch (lgmi_ecdf_eval)."""
    xs = np.ascontiguousarray(np.array(x, dtype=np.float64).reshape(-1))
    if xs.size == 0:
        raise ZeroDivisionError('division by zero')      # 1/n at stat.py:19
    ctx = get_context()
    table_x = np.empty(xs.size, dtype=np.float64)
    table_y = np.empty(xs.size + 1, dtype=np.float64)
    check(ctx._lib.lgmi_ecdf_table(ctx.handle, ptr(xs), xs.size, ptr(table_x), ptr(table_y)), ctx.handle)

    def childfunc(sample):
        s = np.asarray(sample, dtype=np.float64)
        if s.size >= ECDF_DEVICE_MIN_SAMPLES:
            flat = np.ascontiguousarray(s).reshape(-1)
            out = np.empty(flat.size, dtype=np.float64)
            check(ctx._lib.lgmi_ecdf_eval(ctx.handle, ptr(table_x), table_x.size, ptr(flat), flat.size, ptr(out)),
                  ctx.handle)
            return out.reshape(s.shape)
        out = table_y[np.searchsorted(table_x, s, side='left')]   # numpy orders NaN last, as the table does
        return np.float64(out) if s.ndim == 0 else out

    return childfunc


ECDF_DEVICE_MIN_SAMPLES = 4096   # sample arrays at least this long are evaluated on the device


def mip_and_calls(mean_mi, site_types, threshold=0.05, ctx=None):
    """Vectorised global pass (giremi.py:415-429 and :97-114): returns
    (mip, call) with call 1 = positive label, 2 = negative label, 0 = neither.
    `site_types` is an array of type codes or of type names."""
    mean = np.ascontiguousarray(mean_mi, dtype=np.float64)
    st = np.asarray(site_types)
    if st.dtype.kind in "US" or st.dtype == object:
        st = np.array([SITE_TYPE_CODE[t] for t in st.tolist()], dtype=np.uint8)
    flags = np.ascontiguousarray(st, dtype=np.uint8)
    mip = np.empty(mean.size, dtype=np.float64)
    call = np.empty(mean.size, dtype=np.uint8)
    ctx = ctx or get_context()
    check(ctx._lib.lgmi_ecdf(ctx.handle, ptr(mean), ptr(flags), mean.size, float(threshold), ptr(mip), ptr(call)),
          ctx.handle)
    return mip, call


# --------------------------------------------------------------------------- #
# site x splice-site MI: the reference's second mutual_info_score call site
# --------------------------------------------------------------------------- #
class SiteSpliceArrays:
    """Input of lgmi_site_splice_mi (include/lgmi.h), plus the names its integer ids stand for.

    entries  site k owns entries [entry_off[k], entry_off[k+1]): read entry_read[p], allele index entry_allele[p]
             (within the site); one per list entry, so a read listed twice is there twice
    splices  read r has the splice ids splice_id[splice_off[r] .. splice_off[r+1]), ascending and unique
    triples  (tri_site, tri_allele, tri_splice), one per requested pair, in order
    names    read_names[r], site_labels[k], allele_names[k][a], splice_labels[id]"""

    def __init__(self, entry_off, entry_read, entry_allele, splice_off, splice_id, tri_site, tri_allele, tri_splice,
                 read_names, site_labels, allele_names, splice_labels):
        u32 = lambda a: np.ascontiguousarray(a, dtype=np.uint32)
        self.entry_off = np.ascontiguousarray(entry_off, dtype=np.uint64)
        self.entry_read, self.entry_allele = u32(entry_read), u32(entry_allele)
        self.splice_off = np.ascontiguousarray(splice_off, dtype=np.uint64)
        self.splice_id = u32(splice_id)
        self.tri_site, self.tri_allele, self.tri_splice = u32(tri_site), u32(tri_allele), u32(tri_splice)
        self.read_names, self.site_labels = read_names, site_labels
        self.allele_names, self.splice_labels = allele_names, splice_labels

    @property
    def n_sites(self):
        return self.entry_off.size - 1

    @property
    def n_reads(self):
        return self.splice_off.size - 1


def read_splice_csr(read, splice, n_reads):
    """(splice_off, splice_id) of records (read[k], splice[k]): per read its splice ids ascending, each once (the
    reference's membership test is by set, calculate_site_splice_mi.py:122)."""
    read = np.asarray(read, dtype=np.int64)
    splice = np.asarray(splice, dtype=np.int64)
    n_ids = int(splice.max()) + 1 if splice.size else 1
    key = np.unique(read * n_ids + splice)
    off = np.zeros(n_reads + 1, dtype=np.uint64)
    off[1:] = np.cumsum(np.bincount(key // n_ids, minlength=n_reads))
    return off, (key % n_ids).astype(np.uint32)


def site_splice_mi_arrays(a: SiteSpliceArrays, ctx=None, tables=False):
    """MI of every triple of `a` in one synchronous device call (lgmi_site_splice_mi); with tables=True also the
    integer 2x2 tables [N-x-y+xy, y-xy, x-xy, xy] as an (n, 4) uint32 array."""
    ctx = ctx or get_context()
    n = a.tri_site.size
    mi = np.empty(n, dtype=np.float64)
    table = np.empty((n, 4), dtype=np.uint32) if tables else None
    check(ctx._lib.lgmi_site_splice_mi(ctx.handle, a.n_sites, ptr(a.entry_off), ptr(a.entry_read),
                                       ptr(a.entry_allele), a.n_reads, ptr(a.splice_off), ptr(a.splice_id), n,
                                       ptr(a.tri_site), ptr(a.tri_allele), ptr(a.tri_splice), ptr(mi), ptr(table)),
          ctx.handle)
    return (mi, table) if tables else mi


def site_splice_arrays(sites, splices, pairs) -> SiteSpliceArrays:
    """The arrays of `site_splice_mutual_info`'s arguments: names interned once, lists flattened without a Python
    step per entry.  Only the requested sites and splice sites are kept.  A missing site or allele raises KeyError,
    as the reference's lookups do (calculate_site_splice_mi.py:116-117)."""
    import itertools

    import pandas as pd
    site_labels = list(dict.fromkeys(p[0] for p in pairs))
    site_of = {label: k for k, label in enumerate(site_labels)}
    allele_names, lists, list_site, list_allele = [], [], [], []
    for k, label in enumerate(site_labels):
        alleles = sites[label]
        allele_names.append(list(alleles))
        for a, names in enumerate(alleles.values()):
            lists.append(names)
            list_site.append(k)
            list_allele.append(a)
    lens = np.fromiter(map(len, lists), dtype=np.int64, count=len(lists))
    names = np.fromiter(itertools.chain.from_iterable(lists), dtype=object, count=int(lens.sum()))
    entry_read, read_names = pd.factorize(names, use_na_sentinel=False)
    entry_off = np.zeros(len(site_labels) + 1, dtype=np.uint64)
    entry_off[1:] = np.cumsum(np.bincount(np.asarray(list_site, dtype=np.int64), weights=lens,
                                          minlength=len(site_labels)).astype(np.int64))
    entry_allele = np.repeat(np.asarray(list_allele, dtype=np.uint32), lens)
    splice_labels = list(dict.fromkeys(p[2] for p in pairs))
    slists = [splices.get(label, ()) for label in splice_labels]
    slens = np.fromiter(map(len, slists), dtype=np.int64, count=len(slists))
    snames = np.fromiter(itertools.chain.from_iterable(slists), dtype=object, count=int(slens.sum()))
    sread = pd.Index(read_names).get_indexer(snames)
    sid = np.repeat(np.arange(len(slists), dtype=np.int64), slens)
    keep = sread >= 0                                   # reads listed at no requested site cannot count
    splice_off, splice_id = read_splice_csr(sread[keep], sid[keep], len(read_names))
    spl_of = {label: k for k, label in enumerate(splice_labels)}
    allele_of = [{seq: a for a, seq in enumerate(names)} for names in allele_names]
    tri_site = [site_of[p[0]] for p in pairs]
    tri_allele = [allele_of[k][p[1]] for k, p in zip(tri_site, pairs)]
    tri_splice = [spl_of[p[2]] for p in pairs]
    return SiteSpliceArrays(entry_off, entry_read, entry_allele, splice_off, splice_id, tri_site, tri_allele,
                            tri_splice, list(read_names), site_labels, allele_names, splice_labels)


def site_splice_mutual_info(sites, splices, pairs, ctx=None):
    """The loop of giremi/script/calculate_site_splice_mi.py:106-125 as ONE device call.

    `sites`   {site label: {allele: [read names]}}      (:88-92)
    `splices` {splice label: [read names]}              (:95-102)
    `pairs`   iterable of (site label, allele, splice label)   (rows of the pair table)

    Returns the MI of every pair, in order: over all list entries of the site (a read listed twice counts twice,
    :117-120), labels "carries the allele" x "has the splice site" by read NAME (:121-122).  The 2x2 tables are
    counted on the device from interned read ids for the requested pairs only (lgmi_site_splice_mi); at most 64
    alleles per site."""
    pairs = [tuple(p) for p in pairs]
    if not pairs:
        return []
    return site_splice_mi_arrays(site_splice_arrays(sites, splices, pairs), ctx=ctx).tolist()


# --------------------------------------------------------------------------- #
# partitioning
# --------------------------------------------------------------------------- #
def unit_costs(units) -> np.ndarray:
    s = units['n_sites'].astype(np.uint64)
    r = units['n_reads'].astype(np.uint64)
    return (s * (s - np.minimum(s, 1)) // 2 * ((r + 63) // 64)).astype(np.uint64)


def partition_lpt(costs, n_bins):
    """Longest-processing-time greedy partition (SURVEY 8e); returns
    (bin_of[unit], bin_load[bin]).  Pure host bookkeeping, no device needed."""
    lib = _lib.load()
    costs = np.ascontiguousarray(costs, dtype=np.uint64)
    bin_of = np.empty(costs.size, dtype=np.uint32)
    load = np.zeros(int(n_bins), dtype=np.uint64)
    rc = lib.lgmi_partition_lpt(ptr(costs), costs.size, int(n_bins), ptr(bin_of), ptr(load))
    if rc != 0:
        raise LgmiError(rc, "lgmi_partition_lpt: bad argument")
    return bin_of, load
