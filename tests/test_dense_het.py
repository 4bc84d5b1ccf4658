"""The het-anchored form of the deep units (k_gram_i8 over the het sites' rows only) under HET_ONLY | SKIP_NONHET.

Each case runs a batch in HET_ONLY | SKIP_NONHET, with and without EMIT_COUNTS, and compares it with the same batch
in HET_ONLY, which keeps the all-pairs form: records, 3x3 tables, site_mean and site_cnt bit for bit.  The unit is
also checked against the C oracle, and dense_macs against the het plan's tile count."""
import importlib

import numpy as np
import pytest

from conftest import assert_mi_close
from parity import c_oracle, oracle_unit, signed

enc = importlib.import_module("l-giremi_b200.encode")
synth = importlib.import_module("l-giremi_b200.synth")

BM, BN, BK = 128, 256, 128
TYPE_MASK, HET_SNP = 3, 2
SMALL_DEEP = (2, 1)                      # a dense threshold every unit with pairs reaches
RAISED = (1 << 20, 1 << 30)              # ... and one no unit reaches


@pytest.fixture()
def ctx(lg, gpu_ctx):
    yield gpu_ctx
    gpu_ctx.set_dense_threshold(*lg.DENSE_DEFAULT)
    gpu_ctx.set_dense_path(4)


def labels(seed, S, R, cov=0.6):
    return synth.make_deep_unit(seed, S, R, cov, keep_labels=True)[1]


def unit(lab, het):
    types = ["snp"] * lab.shape[0]
    for s in het:
        types[s] = "het_snp"
    return enc.EncodedUnit([1000 + 37 * s for s in range(lab.shape[0])], types, lab)


def het_macs(S, R, het, blocks):
    """Multiply-accumulates of the het tile list: het row blocks x column blocks holding a pair (het[h], s)."""
    H = len(het)
    n = 0
    for I in range(-(-H // BM)):
        rows = het[I * BM:(I + 1) * BM]
        for J in range(-(-S // BN)):
            cols = range(J * BN, min(S, (J + 1) * BN))
            if len(cols) > 1 or len(rows) > 1 or rows[0] != cols[0]:
                n += 1
    return n * blocks * BM * BN * (4 * -(-R // 128) * 32)


def same(a, b):
    assert a.n_records == b.n_records
    assert np.array_equal(a.records.view(np.uint8), b.records.view(np.uint8))
    assert np.array_equal(a.unit_rec_off, b.unit_rec_off)
    assert (a.counts is None) == (b.counts is None)
    if a.counts is not None:
        assert np.array_equal(a.counts, b.counts)
    assert np.array_equal(a.site_mean.view(np.uint64), b.site_mean.view(np.uint64))
    assert np.array_equal(a.site_cnt, b.site_cnt)


def check(lg, ctx, pb, het_units, run=None):
    """pb in SKIP_NONHET (+- EMIT_COUNTS) against HET_ONLY (+- EMIT_COUNTS); het_units: {unit: (S, R, het list,
    blocks)} of the deep units that take the het form.  Returns the SKIP_NONHET | EMIT_COUNTS result."""
    run = run or (lambda m: lg.mi_step_batched(pb, 6, m, ctx=ctx, n_chunks=1))
    out = None
    for extra in (0, lg.MODE_EMIT_COUNTS):
        ref = run(lg.MODE_HET_ONLY | extra)
        got = run(lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET | extra)
        same(got, ref)
        if het_units:
            assert got.dense_macs == sum(het_macs(*v) for v in het_units.values())
            assert got.dense_macs < ref.dense_macs
        out = got
    return out


def check_oracle(res, pb, u, eu, mc=6):
    i, j, mi, tab, mean, cnt = oracle_unit(eu, mc)
    is_het = np.array([t == "het_snp" for t in eu.types], dtype=bool)
    keep = is_het[i] | is_het[j] if len(i) else np.zeros(0, bool)
    rec = res.unit_records(u)
    assert rec["i"].tolist() == i[keep].tolist() and rec["j"].tolist() == j[keep].tolist()
    assert np.array_equal(res.unit_counts(u).astype(np.int64), tab[keep])
    assert_mi_close(rec["mi"], mi[keep], 0.9)
    off = int(pb.units["site_off"][u])
    S = eu.n_sites
    assert np.array_equal(np.isnan(res.site_mean[off:off + S]), np.isnan(mean))
    assert_mi_close(res.site_mean[off:off + S][~np.isnan(mean)], mean[~np.isnan(mean)], 0.9, "site mean")


HET_SETS = {
    0: [],
    1: [0],
    2: [0, 999],
    127: list(range(0, 999, 7))[:126] + [999],
    128: list(range(1, 1000, 7))[:128],
    129: list(range(0, 999, 7))[:128] + [999],
}


@pytest.mark.gpu
@pytest.mark.parametrize("H", sorted(HET_SETS))
def test_deep_het_form_at_the_default_threshold(lg, ctx, H):
    """1 000 sites (not a multiple of 256) x 8 200 reads: a deep unit at the default threshold, four blocks."""
    lab = labels(71 + H, 1000, 8200)
    het = HET_SETS[H]
    assert len(het) == H and len(set(het)) == H
    eu = unit(lab, het)
    pb = lg.pack_units([eu])
    res = check(lg, ctx, pb, {0: (1000, 8200, het, 4)})
    assert res.n_dense_units == 1 and res.n_dense_four == 1
    if H == 0:
        assert res.n_records == 0 and np.all(np.isnan(res.site_mean))
    check_oracle(res, pb, 0, eu)


@pytest.mark.gpu
@pytest.mark.parametrize("blocks", [4, 9])
def test_deep_het_form_small_shapes(lg, ctx, blocks):
    """A lowered threshold sends small units to the tensor-core path: four and nine blocks, het sites at 0 and S-1,
    beside a unit that is all het (the form is not taken)."""
    ctx.set_dense_threshold(*SMALL_DEEP)
    ctx.set_dense_path(blocks)
    rng = np.random.default_rng(5)
    shapes = [(600, 300), (257, 700), (130, 128), (3, 200)]
    eus, het_units = [], {}
    for u, (S, R) in enumerate(shapes):
        lab = labels(100 + u, S, R)
        het = sorted({0, S - 1} | set(rng.choice(S, S // 10, replace=False).tolist()))
        if u == 3:
            het = list(range(S))                            # all het: the all-pairs form is cheaper
        else:
            het_units[u] = (S, R, het, blocks)
        eus.append(unit(lab, het))
    pb = lg.pack_units(eus)
    res = check(lg, ctx, pb, None)
    tri3 = lg.mi_step_batched(lg.pack_units([eus[3]]), 6, lg.MODE_HET_ONLY, ctx=ctx, n_chunks=1).dense_macs
    assert res.dense_macs == sum(het_macs(*v) for v in het_units.values()) + tri3
    assert res.n_dense_units == len(shapes) and res.n_dense_four == (len(shapes) if blocks == 4 else 0)
    for u, eu in enumerate(eus):
        check_oracle(res, pb, u, eu)


@pytest.mark.gpu
def test_deep_het_form_falls_back_to_nine_blocks(lg, ctx):
    """A site with more "other" reads than its list holds sends the unit to nine blocks on the device; the het form
    follows it there."""
    lab = labels(12, 200, 8300)
    covered = np.flatnonzero(lab[7] != 255)
    lab[7, covered[:400]] = 0                                # 400 > max(256, 8300 / 64) "other" reads at site 7
    het = [0, 7, 50, 199]
    eu = unit(lab, het)
    pb = lg.pack_units([eu])
    res = check(lg, ctx, pb, {0: (200, 8300, het, 9)})
    assert res.n_dense_units == 1 and res.n_dense_four == 0
    check_oracle(res, pb, 0, eu)


@pytest.mark.gpu
def test_deep_het_form_in_a_mixed_batch_and_every_entry_point(lg, ctx):
    """A deep unit among small and mid-depth units: one submit, the pipelined step (also begin / collect / finish),
    a graph replay and a timed run agree; one Batch uploaded twice with different het flags gives each upload's
    result."""
    rng = np.random.default_rng(3)
    eus = []
    for u, (S, R) in enumerate([(40, 200), (120, 900), (300, 8200), (64, 256), (90, 3000)]):
        lab = labels(300 + u, S, R)
        het = sorted(rng.choice(S, max(1, S // 10), replace=False).tolist())
        eus.append(unit(lab, het))
    pb = lg.pack_units(eus)
    deep_het = [s for s, t in enumerate(eus[2].types) if t == "het_snp"]
    one = check(lg, ctx, pb, {2: (300, 8200, deep_het, 4)})
    for u, eu in enumerate(eus):
        check_oracle(one, pb, u, eu)
    mode = lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET | lg.MODE_EMIT_COUNTS
    p = lg.Pipeline(ctx, pb, n_chunks=3)
    try:
        same(p.step(6, mode), one)
        p.begin(6, mode)
        p.collect()
        same(p.finish(), one)
    finally:
        p.close()
    b = lg.Batch(ctx, pb)
    try:
        b.upload()
        b.run(6, mode | lg.MODE_GRAPH)
        graph = b.download()
        b.run(6, mode)
        timed = b.download()
        same(graph, one)
        same(timed, one)
        assert timed.dense_kernel_ms > 0 and timed.gram_kernel_ms >= 0
        # new flags through the same batch: another het set of the same layout (the tables' contents change, the
        # captured graph stays), then one of two row blocks, past half the triangle (the all-pairs form)
        off = int(pb.units["site_off"][2])
        for new_het, taken in ((list(range(1, 300, 3))[:90], True), (list(range(0, 300, 2))[:140], False)):
            flags = pb.site_flags.copy()
            flags[off:off + 300] = (flags[off:off + 300] & ~np.uint8(TYPE_MASK)) | np.uint8(1)     # snp
            flags[off + np.array(new_het)] = (flags[off + np.array(new_het)] & ~np.uint8(TYPE_MASK)) | HET_SNP
            pb2 = lg.PlaneBatch(pb.units, pb.planes, flags)
            ref2 = lg.mi_step_batched(pb2, 6, lg.MODE_HET_ONLY | lg.MODE_EMIT_COUNTS, ctx=ctx, n_chunks=1)
            for m in (mode | lg.MODE_GRAPH, mode):
                b.upload(site_flags=flags)
                b.run(6, m)
                got = b.download()
                same(got, ref2)
                assert (got.dense_macs < ref2.dense_macs) == taken
        b.upload()                                           # and back
        b.run(6, mode | lg.MODE_GRAPH)
        same(b.download(), one)
    finally:
        b.close()


def het_flags(pb, u, S, het):
    """pb's flag bytes with unit u's het sites replaced by `het` (the others snp)."""
    off = int(pb.units["site_off"][u])
    flags = pb.site_flags.copy()
    flags[off:off + S] = (flags[off:off + S] & ~np.uint8(TYPE_MASK)) | np.uint8(1)
    flags[off + np.array(het, dtype=np.int64)] = (flags[off + np.array(het, dtype=np.int64)] & ~np.uint8(TYPE_MASK)) | HET_SNP
    return flags


class _DeviceBytes:
    """A device buffer of the batch, seen by torch through the CUDA array interface."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 3}


@pytest.mark.gpu
def test_deep_het_form_device_written_flags_and_late_reupload(lg, ctx):
    """A caller that writes the flags into the device buffer itself keeps the all-pairs form: after a graph run on
    uploaded flags, device_ptrs and other het sites written on the device, the next graph run gives the new flags'
    result (the graph captured with the old het plan is not replayed).  And dense_macs reports the form the run
    took even when other flags are uploaded between the run and the download."""
    torch = pytest.importorskip("torch")
    lab = labels(41, 1000, 8200)
    het_a = list(range(0, 1000, 11))
    het_b = list(range(5, 1000, 13))
    eu = unit(lab, het_a)
    pb = lg.pack_units([eu])
    flags_b = het_flags(pb, 0, 1000, het_b)
    pb_b = lg.PlaneBatch(pb.units, pb.planes, flags_b)
    mode = lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET | lg.MODE_EMIT_COUNTS
    ref_a = lg.mi_step_batched(pb, 6, lg.MODE_HET_ONLY | lg.MODE_EMIT_COUNTS, ctx=ctx, n_chunks=1)
    ref_b = lg.mi_step_batched(pb_b, 6, lg.MODE_HET_ONLY | lg.MODE_EMIT_COUNTS, ctx=ctx, n_chunks=1)
    b = lg.Batch(ctx, pb)
    try:
        b.upload()
        b.run(6, mode | lg.MODE_GRAPH)
        got_a = b.download()
        same(got_a, ref_a)
        assert got_a.dense_macs == het_macs(1000, 8200, het_a, 4) < ref_a.dense_macs
        _, d_flags, _, _ = b.device_ptrs()
        dst = torch.as_tensor(_DeviceBytes(d_flags, pb.n_sites), device="cuda")
        dst.copy_(torch.from_numpy(flags_b).cuda())
        torch.cuda.synchronize()
        b.run(6, mode | lg.MODE_GRAPH)
        got_b = b.download()
        same(got_b, ref_b)
        assert got_b.dense_macs == ref_b.dense_macs                  # the all-pairs form
        # run on uploaded flags A, upload B, then download: A's result and A's het form
        b.upload()
        b.run(6, mode)
        b.upload(site_flags=flags_b)
        late = b.download()
        same(late, ref_a)
        assert late.dense_macs == het_macs(1000, 8200, het_a, 4)
    finally:
        b.close()


@pytest.mark.gpu
def test_cfg3_het_form_equals_popcount_and_oracle(lg, ctx):
    """The full cfg3 unit (2 000 sites x 100 000 reads, the bench's seed) in HET_ONLY | SKIP_NONHET | EMIT_COUNTS:
    the het form against the all-pairs form and the popcount path bit for bit, and a 20-site sample against the
    oracle."""
    pb, lab = synth.make_deep_unit(20261021, 2000, 100000, 0.6, keep_labels=True)
    het = np.flatnonzero((pb.site_flags & TYPE_MASK) == HET_SNP).tolist()
    mode = lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET | lg.MODE_EMIT_COUNTS
    res = check(lg, ctx, pb, {0: (2000, 100000, het, 4)})
    ctx.set_dense_threshold(*RAISED)
    popc = lg.mi_step_batched(pb, 6, mode, ctx=ctx, n_chunks=1)
    assert popc.n_dense_units == 0
    same(res, popc)
    rng = np.random.default_rng(9)
    idx = np.sort(np.concatenate([rng.choice(het, 6, replace=False),
                                  rng.choice(np.setdiff1d(np.arange(2000), het), 14, replace=False)]))
    i, j, mi, tab = c_oracle.unit_pairs_from_labels(signed(lab[idx]), None, 6)
    keep = np.isin(idx[i], het) | np.isin(idx[j], het)
    rec = res.records
    key = rec["i"].astype(np.int64) * 65536 + rec["j"]
    want = idx[i][keep].astype(np.int64) * 65536 + idx[j][keep]
    at = np.searchsorted(key, want)
    assert np.array_equal(key[at], want)
    assert np.array_equal(res.counts[at].astype(np.int64), tab[keep])
    assert_mi_close(rec["mi"][at], mi[keep], 0.9)
