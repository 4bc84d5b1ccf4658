"""GPU parity tests: liblgmi.so (through its C ABI, via the ctypes binding)
against the oracle and the golden fixtures generated from the real reference.

  * pair sets, 3x3 counts, threshold calls, record order: bit-exact
  * MI, mean MI, mip: 1e-10 relative (conftest.MI_RTOL / MI_ATOL), with a floor
    on the fraction that must be bit-identical
"""
import importlib
import math
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, assert_mi_close, golden_mismatches, unhex

sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import c_oracle  # noqa: E402
from fuzz import random_mismatches  # noqa: E402
from parity import _other_heavy_unit, _synth_unit, check_batch, oracle_unit, signed  # noqa: E402

pytestmark = pytest.mark.gpu

synth = importlib.import_module("l-giremi_b200.synth")
enc = importlib.import_module("l-giremi_b200.encode")


# --------------------------------------------------------------------------- drop-in functions
def rows_equal(got, want_hex):
    want = [[r[0], r[1], r[2], r[3], unhex(r[4])] for r in want_hex]
    assert [r[:4] for r in got] == [r[:4] for r in want]
    assert all(isinstance(r[4], float) for r in got)
    assert_mi_close([r[4] for r in got], [r[4] for r in want], 0.97)


def test_kat_drop_in_functions(lg, gpu_ctx, golden):
    kat = golden("kat.json")
    for name in ("ab", "cb", "db", "ef_min6", "ef_min7", "abc"):
        unit = kat[name]
        m = golden_mismatches(unit)
        rows = lg.mismatch_pair_mutual_info(m, unit["min_common"])
        rows_equal(rows, unit["rows"])
        kept = [r for r in rows if r[1] == 'het_snp' or r[3] == 'het_snp']
        means = lg.mean_mismatch_pair_mutual_info(kept) if kept else []
        assert [p for p, _ in means] == [p for p, _ in unit["means"]]
        assert_mi_close([v for _, v in means], [unhex(v) for _, v in unit["means"]], 0.9)
    # the survey's known answers, literally
    m = golden_mismatches(kat["abc"])
    got = {(r[0], r[2]): r[4] for r in lg.mismatch_pair_mutual_info(m, 6)}
    assert got == {(10, 20): 0.6931471805599454, (10, 30): 0.4620981203732968, (20, 30): 0.4620981203732968}
    assert lg.mismatch_pair_mutual_info(golden_mismatches(kat["ef_min6"]), 6)[0][4] == 0.0
    assert lg.mismatch_pair_mutual_info({}, 6) == []
    assert lg.mismatch_pair_mutual_info({10: m[10]}, 6) == []
    assert lg.mean_mismatch_pair_mutual_info([]) == []


def test_default_min_common_is_five(lg, gpu_ctx):
    reads = ['r%d' % k for k in range(10)]
    a = {'ref': 'A', 'type': 'het_snp', 'depth': {'A': 3, 'G': 2}, 'nt': {'A': reads[:3], 'G': reads[3:5]}}
    b = {'ref': 'A', 'type': 'mismatch', 'depth': {'A': 2, 'G': 3}, 'nt': {'A': reads[:2], 'G': reads[2:5]}}
    assert len(lg.mismatch_pair_mutual_info({1: a, 2: b})) == 1          # 5 common, default 5: kept
    assert len(lg.mismatch_pair_mutual_info({1: a, 2: b}, 6)) == 0


def test_index_error_like_reference(lg, gpu_ctx):
    ok = {'ref': 'A', 'type': 'het_snp', 'depth': {'A': 6, 'C': 6},
          'nt': {'A': ['r%d' % k for k in range(6)], 'C': ['r%d' % k for k in range(6, 12)]}}
    bad = {'ref': 'A', 'type': 'mismatch', 'depth': {'G': 12}, 'nt': {'G': ['r%d' % k for k in range(12)]}}
    with pytest.raises(IndexError):
        lg.mismatch_pair_mutual_info({10: bad, 20: ok}, 6)
    assert lg.mismatch_pair_mutual_info({10: bad, 20: ok}, 13) == []


@pytest.mark.parametrize("fixture", ["units_fuzz.json", "units_synth.json"])
def test_golden_units_drop_in(lg, gpu_ctx, golden, fixture):
    for unit in golden(fixture):
        m = golden_mismatches(unit)
        rows = lg.mismatch_pair_mutual_info(m, unit["min_common"])
        rows_equal(rows, unit["rows"])
        kept = [r for r in rows if r[1] == 'het_snp' or r[3] == 'het_snp']
        means = lg.mean_mismatch_pair_mutual_info(kept) if kept else []
        assert [p for p, _ in means] == [p for p, _ in unit["means"]]
        assert_mi_close([v for _, v in means], [unhex(v) for _, v in unit["means"]])


def test_golden_units_batched(lg, gpu_ctx, golden):
    """All golden units with the same min_common in ONE submit."""
    units = golden("units_fuzz.json") + golden("units_synth.json")
    for mc in sorted(set(u["min_common"] for u in units)):
        group = [u for u in units if u["min_common"] == mc]
        eus = [lg.encode_mismatches(golden_mismatches(u)) for u in group]
        ok = [k for k, eu in enumerate(eus) if not eu.bad_sites]
        full = check_batch(lg, gpu_ctx, [eus[k] for k in ok], mc)
        for n, k in enumerate(ok):
            rec = full.unit_records(n)
            pos, typ = eus[k].positions, eus[k].types
            rows = [[pos[i], typ[i], pos[j], typ[j], mi] for i, j, mi in
                    zip(rec['i'].tolist(), rec['j'].tolist(), rec['mi'].tolist())]
            rows_equal(rows, group[k]["rows"])
            # mean MI against the reference's own output
            off = int(np.sum([eus[q].n_sites for q in ok[:n]]))
            want = dict((p, unhex(v)) for p, v in group[k]["means"])
            got = {p: v for p, v in zip(pos, full.site_mean[off:off + len(pos)].tolist()) if not math.isnan(v)}
            assert list(got) == sorted(want)
            assert_mi_close([got[p] for p in got], [want[p] for p in got])


# --------------------------------------------------------------------------- batched kernel vs oracle
def test_fuzz_batch_all_quirks(lg, gpu_ctx):
    rng = np.random.default_rng(2026)
    ms = [random_mismatches(rng) for _ in range(300)]
    eus = [lg.encode_mismatches(m) for m in ms]
    eus = [e for e in eus if not e.bad_sites]
    for mc in (1, 3, 6):
        check_batch(lg, gpu_ctx, eus, mc)


def test_ragged_and_degenerate_units(lg, gpu_ctx):
    """Empty units, single-site units, R not a multiple of 32/128, exactly
    2048 / 2049 pairs per unit (work-item boundary), units spanning many items."""
    rng = np.random.default_rng(77)
    shapes = [(0, 0), (1, 9), (2, 1), (2, 6), (3, 31), (5, 32), (7, 33), (9, 127), (11, 128), (4, 129),
              (64, 40), (65, 40), (66, 70), (130, 17), (50, 200), (23, 1000), (300, 90)]
    eus = []
    for S, R in shapes:
        if S == 0:
            eus.append(enc.EncodedUnit([], [], np.zeros((0, 0), np.uint8)))
            continue
        a, k = synth.draw_alleles(rng, 1, S, R, float(rng.uniform(0.2, 0.9))) if R >= 2 and S >= 1 else (None, None)
        if a is None:
            lab = np.full((S, R), 2, np.uint8)
            eus.append(enc.EncodedUnit(list(range(S)), ['het_snp'] * S, lab))
            continue
        lab = synth.labels_from_alleles(a[0])
        eus.append(enc.EncodedUnit([1000 + 37 * s for s in range(S)],
                                   [("mismatch", "snp", "het_snp")[int(x)] for x in k[0]], lab))
    for mc in (1, 6, 20):
        check_batch(lg, gpu_ctx, eus, mc)


def test_min_common_is_strict_less_than(lg, gpu_ctx):
    """A pair with exactly min_common common reads is kept (mutual_information.py:19)."""
    for n in (1, 5, 6, 7, 32, 33, 128, 129):
        lab = np.full((2, n + 3), 255, np.uint8)
        lab[0, :n] = [2 if k % 2 else 1 for k in range(n)]
        lab[1, :n] = [2 if k % 3 else 1 for k in range(n)]
        lab[0, n] = 2          # covered by one site only
        lab[1, n + 1] = 1
        eu = enc.EncodedUnit([10, 20], ['het_snp', 'mismatch'], lab)
        pb = lg.pack_units([eu])
        assert lg.mi_step_batched(pb, n, lg.MODE_ALL_PAIRS, ctx=gpu_ctx).n_records == 1
        assert lg.mi_step_batched(pb, n + 1, lg.MODE_ALL_PAIRS, ctx=gpu_ctx).n_records == 0
        res = lg.mi_step_batched(pb, n + 1, lg.MODE_HET_ONLY, ctx=gpu_ctx)
        assert np.isnan(res.site_mean).all() and res.site_cnt.tolist() == [0, 0]


def test_heavy_tail_batch(lg, gpu_ctx):
    pb, raw = synth.make_heavy_tail(20261022, 120, keep_raw=True, s_max=400, r_max=5000)
    eus = [enc.EncodedUnit([1000 + 37 * s for s in range(a.shape[0])],
                           [("mismatch", "snp", "het_snp")[int(x)] for x in k], synth.labels_from_alleles(a))
           for a, k in raw]
    full = check_batch(lg, gpu_ctx, eus, 6)
    # the generator's own packing is the same bytes as pack_units
    again = lg.mi_step_batched(pb, 6, lg.MODE_ALL_PAIRS, ctx=gpu_ctx)
    assert np.array_equal(again.records, full.records)


@pytest.mark.parametrize("cov", [0.01, 0.05, 0.1, 0.25, 0.5])
def test_cfg5_grid_against_oracle(lg, gpu_ctx, cov):
    """BASELINE.json configs[4] at oracle size: the mi_min_common_read x coverage grid on 50-site x
    200-read units -- from 'no pair has enough common reads' to 'every pair survives'."""
    rng = np.random.default_rng(int(cov * 1000) + 11)
    eus = [_synth_unit(rng, 50, 200, cov) for _ in range(12)]
    survivors = []
    for mc in (6, 10, 20, 50):
        survivors.append(check_batch(lg, gpu_ctx, eus, mc).n_records)
    assert survivors == sorted(survivors, reverse=True)      # a larger threshold never keeps more pairs
    if cov <= 0.05:
        assert survivors[-1] == 0                            # <= 10 covered reads per site: nothing reaches 50


def test_deep_unit_large_counts(lg, gpu_ctx):
    """R = 30 000: counts beyond 2^14, ln table grown on demand."""
    rng = np.random.default_rng(5)
    a, k = synth.draw_alleles(rng, 1, 24, 30000, 0.7)
    eu = enc.EncodedUnit(list(range(24)), [("mismatch", "snp", "het_snp")[int(x)] for x in k[0]],
                         synth.labels_from_alleles(a[0]))
    check_batch(lg, gpu_ctx, [eu], 6, min_exact=0.9)


def test_many_sites_multi_item_unit(lg, gpu_ctx):
    """S = 700 (244 650 pairs, ~120 work items): ordered compaction across CTAs
    and the multi-item per-site mean path."""
    rng = np.random.default_rng(6)
    a, k = synth.draw_alleles(rng, 1, 700, 64, 0.3)
    eu = enc.EncodedUnit(list(range(700)), [("mismatch", "snp", "het_snp")[int(x)] for x in k[0]],
                         synth.labels_from_alleles(a[0]))
    small = enc.EncodedUnit([1, 2, 3], ['het_snp', 'mismatch', 'snp'], synth.labels_from_alleles(a[0][:3]))
    check_batch(lg, gpu_ctx, [small, eu, small], 6)


def test_mid_units_popcount_and_tensor_paths_agree(lg, gpu_ctx):
    """Mid-depth units (more than 64 sites or 256 reads): k_tile_gram_ws + k_tile_finish (tcgen05, the default) and
    k_tile_mi (popcount, path 0) must give the same records, tables and means bit for bit, and both match the oracle.
    Shapes straddle the 128-site row blocks, the 48-site column blocks and the 128-read k-blocks; (47, 9000) is the
    deepest unit below the default dense threshold (48 sites x 8192 reads)."""
    rng = np.random.default_rng(20261031)
    shapes = [(65, 40), (48, 257), (49, 300), (129, 129), (97, 1000), (2, 700), (3, 4097), (257, 70), (200, 385),
              (145, 128), (47, 9000)]
    eus = [_synth_unit(rng, S, R, cov) for (S, R), cov in zip(shapes, [0.5, 0.3, 0.7, 0.5, 0.2, 1.0, 0.6, 0.4, 0.5, 0.9, 0.3])]
    eus.insert(3, enc.EncodedUnit([1, 2, 3], ['het_snp', 'mismatch', 'snp'], eus[0].labels[:3, :30]))   # a small unit between
    pb = lg.pack_units(eus)
    out = {}
    try:
        for path in (2, 0):
            gpu_ctx.set_tile_path(path)
            full = check_batch(lg, gpu_ctx, eus, 6, min_exact=0.9)
            assert full.n_dense_units == 0
            het = lg.mi_step_batched(pb, 9, lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET | lg.MODE_EMIT_COUNTS, ctx=gpu_ctx)
            out[path] = (full, het)
    finally:
        gpu_ctx.set_tile_path(2)                                # (the default)
    for a, b in zip(out[2], out[0]):
        assert np.array_equal(a.records, b.records) and np.array_equal(a.counts, b.counts)
        assert np.array_equal(a.site_mean, b.site_mean, equal_nan=True) and np.array_equal(a.site_cnt, b.site_cnt)
        assert np.array_equal(a.unit_rec_off, b.unit_rec_off)


# --------------------------------------------------------------------------- tensor-core path (K3)
@pytest.fixture()
def dense_everything(lg, gpu_ctx):
    """Every unit with a pair goes through k_dense_x + k_gram_i8."""
    gpu_ctx.set_dense_threshold(2, 1)
    yield gpu_ctx
    gpu_ctx.set_dense_threshold(*lg.DENSE_DEFAULT)


def test_dense_path_small_shapes(lg, dense_everything):
    """int8 tcgen05 Gram kernel forced onto small and ragged units: one tile, several
    tiles per plane pair, S and R off every block boundary, third alleles present.
    Counts bit-exact against the oracle, MI within tolerance, same records as the
    popcount path."""
    ctx = dense_everything
    rng = np.random.default_rng(31)
    shapes = [(2, 6), (3, 127), (70, 300), (129, 129), (257, 1000), (300, 90), (513, 260)]
    eus = [_synth_unit(rng, S, R, float(rng.uniform(0.3, 0.9))) for S, R in shapes]
    for mc in (1, 6):
        full = check_batch(lg, ctx, eus, mc)
        assert full.n_dense_units == len(eus) and full.dense_macs > 0
    dense = lg.mi_step_batched(lg.pack_units(eus), 6, lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS, ctx=ctx)
    ctx.set_dense_threshold(1 << 20, 1 << 30)
    popc = lg.mi_step_batched(lg.pack_units(eus), 6, lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS, ctx=ctx)
    assert popc.n_dense_units == 0
    assert np.array_equal(dense.records, popc.records) and np.array_equal(dense.counts, popc.counts)
    assert np.array_equal(dense.site_mean, popc.site_mean, equal_nan=True)


@pytest.mark.parametrize("blocks", [4, 9])
def test_dense_forms_agree_and_fall_back(lg, dense_everything, blocks):
    """lgmi_set_dense_path: four Gram blocks + the "other" cells from the listed reads, or nine blocks.  Units with
    few "other" reads take the four-block form, a unit with a site above max(256, R/64) of them falls back to nine
    blocks on the device; counts, MI and means against the oracle, and the same records as the popcount path."""
    ctx = dense_everything
    ctx.set_dense_path(blocks)
    try:
        rng = np.random.default_rng(131)
        sparse = [_synth_unit(rng, S, R, 0.6) for S, R in ((40, 700), (130, 1500), (300, 520), (65, 20000))]
        some = _other_heavy_unit(rng, 90, 30000, 0.6, 0.004)      # ~100 "other" reads per site: listed (cap 468)
        many = _other_heavy_unit(rng, 70, 3000, 0.7, 0.4)          # het sites: ~600 per site, over the cap of 256 -> nine blocks
        lab = rng.integers(0, 3, size=(50, 900)).astype(np.uint8)
        lab[lab == 0] = 255                                          # no "other" label at all: not covered instead
        none = enc.EncodedUnit(list(range(50)), ["het_snp" if s % 7 == 0 else "mismatch" for s in range(50)], lab)
        eus = sparse + [some, many, none]
        for mc in (3, 6):
            full = check_batch(lg, ctx, eus, mc, min_exact=0.9)
            assert full.n_dense_units == len(eus)
            assert full.n_dense_four == (len(eus) - 1 if blocks == 4 else 0)
        dense = lg.mi_step_batched(lg.pack_units(eus), 6, lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS, ctx=ctx)
        ctx.set_dense_threshold(1 << 20, 1 << 30)
        popc = lg.mi_step_batched(lg.pack_units(eus), 6, lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS, ctx=ctx)
        assert popc.n_dense_units == 0
        assert np.array_equal(dense.records, popc.records) and np.array_equal(dense.counts, popc.counts)
        assert np.array_equal(dense.site_mean, popc.site_mean, equal_nan=True)
    finally:
        ctx.set_dense_path(4)


def test_dense_four_blocks_more_than_2048_sites(lg, dense_everything):
    """k_other_fix walks the partners 2 048 at a time and k_dense_prep the sites 256 at a time: a unit of 2 100 sites
    (S_pad 2 304: two passes, a ragged last block) in both dense forms against the popcount path, bit for bit, and a
    sample of its sites against the oracle."""
    ctx = dense_everything
    rng = np.random.default_rng(132)
    eu = _other_heavy_unit(rng, 2100, 700, 0.4, 0.01)
    pb = lg.pack_units([eu])
    mode = lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS
    out = {}
    try:
        for blocks in (4, 9):
            ctx.set_dense_path(blocks)
            out[blocks] = lg.mi_step_batched(pb, 6, mode, ctx=ctx)
            assert out[blocks].n_dense_units == 1 and out[blocks].n_dense_four == (1 if blocks == 4 else 0)
    finally:
        ctx.set_dense_path(4)
    ctx.set_dense_threshold(1 << 20, 1 << 30)
    popc = lg.mi_step_batched(pb, 6, mode, ctx=ctx)
    assert popc.n_dense_units == 0 and popc.n_records > 100000
    for blocks in (4, 9):
        d = out[blocks]
        assert np.array_equal(d.records, popc.records) and np.array_equal(d.counts, popc.counts)
        assert np.array_equal(d.site_mean, popc.site_mean, equal_nan=True) and np.array_equal(d.site_cnt, popc.site_cnt)
    idx = np.sort(rng.choice(2100, 24, replace=False))
    i, j, mi, tab = c_oracle.unit_pairs_from_labels(signed(eu.labels[idx]), None, 6)
    rec = out[4].records
    key = rec['i'].astype(np.int64) * 65536 + rec['j']
    want = idx[i].astype(np.int64) * 65536 + idx[j]
    at = np.searchsorted(key, want)
    assert np.array_equal(key[at], want)
    assert np.array_equal(out[4].counts[at].astype(np.int64), tab)
    assert_mi_close(rec['mi'][at], mi, 0.9)


def test_dense_path_deep_unit(lg, gpu_ctx):
    """A unit over the default threshold (520 sites x 12 000 reads) mixed with small
    units in one batch: the deep one takes the tensor cores, the others do not."""
    rng = np.random.default_rng(32)
    deep = _synth_unit(rng, 520, 12000, 0.6)
    narrow = _synth_unit(rng, 60, 9000, 0.5)          # few sites, deep: one padded 256-site block
    tiled = _synth_unit(rng, 30, 9000, 0.5)           # below the site threshold: 16 x 16 popcount tiles
    small = [_synth_unit(rng, 40, 150, 0.5) for _ in range(3)]
    full = check_batch(lg, gpu_ctx, [small[0], deep, small[1], narrow, tiled, small[2]], 6, min_exact=0.9)
    assert full.n_dense_units == 2
    assert full.dense_kernel_ms > 0.0


def test_cfg3_full_size_dense_equals_popcount_and_oracle(lg, gpu_ctx):
    """BASELINE.json configs[2] at full size (2 000 sites x 100 000 reads, 1 999 000 pairs):
    the tensor-core path and the popcount path give the same records, tables and means
    bit for bit, and a random sub-unit of 20 sites matches the oracle."""
    pb, lab = synth.make_deep_unit(20261021, 2000, 100000, 0.6, keep_labels=True)
    mode = lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS
    dense = lg.mi_step_batched(pb, 6, mode, ctx=gpu_ctx)
    assert dense.n_dense_units == 1 and dense.n_candidates == 1_999_000
    gpu_ctx.set_dense_threshold(1 << 20, 1 << 30)
    try:
        popc = lg.mi_step_batched(pb, 6, mode, ctx=gpu_ctx)
    finally:
        gpu_ctx.set_dense_threshold(*lg.DENSE_DEFAULT)
    assert popc.n_dense_units == 0
    assert np.array_equal(dense.records, popc.records)
    assert np.array_equal(dense.counts, popc.counts)
    assert np.array_equal(dense.site_mean, popc.site_mean, equal_nan=True)
    assert np.array_equal(dense.site_cnt, popc.site_cnt)
    # every table sums to the pair's common-read count and the marginals are consistent
    rec = dense.records
    assert np.all(dense.counts.sum(axis=1) >= 6)
    key = rec['i'].astype(np.int64) * 65536 + rec['j']
    assert np.all(np.diff(key) > 0)
    rng = np.random.default_rng(9)
    idx = np.sort(rng.choice(2000, 20, replace=False))
    i, j, mi, tab = c_oracle.unit_pairs_from_labels(signed(lab[idx]), None, 6)
    at = np.searchsorted(key, idx[i].astype(np.int64) * 65536 + idx[j])
    assert np.array_equal(key[at], idx[i].astype(np.int64) * 65536 + idx[j])      # same pairs survive
    assert np.array_equal(dense.counts[at].astype(np.int64), tab)
    assert_mi_close(rec['mi'][at], mi, 0.9)


def test_small_units_block_boundaries(lg, gpu_ctx):
    """Small units (<= 64 sites, <= 256 reads: k_count_fast + k_pairs_fast) from 2 to 64 sites and 6 to 256
    reads, on both sides of 128 reads (one or two k-blocks of plane words), plus fuzz units: records, 3x3
    tables and means against the oracle at min_common 1, 6 and 20."""
    rng = np.random.default_rng(41)
    shapes = [(2, 6), (3, 40), (9, 128), (10, 129), (11, 200), (20, 256), (30, 31), (31, 255), (39, 100), (40, 128),
              (41, 129), (50, 200), (59, 256), (60, 200), (61, 200), (64, 256)]
    eus = [_synth_unit(rng, S, R, float(rng.uniform(0.3, 0.95))) for S, R in shapes]
    eus += [lg.encode_mismatches(random_mismatches(rng)) for _ in range(60)]
    eus = [e for e in eus if not e.bad_sites]
    for mc in (1, 6, 20):
        check_batch(lg, gpu_ctx, eus, mc)


def test_small_units_many_others_fall_back(lg, gpu_ctx):
    """More than 7 'other' reads in a cell does not fit the packed form: the unit is flagged and
    the generic kernel takes it."""
    rng = np.random.default_rng(42)
    lab = rng.choice(np.array([0, 1, 2, 255], np.uint8), size=(12, 150), p=[0.3, 0.3, 0.3, 0.1])
    eu = enc.EncodedUnit(list(range(12)), ['het_snp', 'mismatch'] * 6, lab)
    ok = _synth_unit(rng, 20, 100, 0.6)
    check_batch(lg, gpu_ctx, [ok, eu, ok], 6)


# --------------------------------------------------------------------------- pipelined step
@pytest.mark.parametrize("n_chunks", [1, 2, 5, 64])
def test_pipelined_step_equals_one_submit(lg, gpu_ctx, n_chunks):
    """lgmi_pipeline_*: groups of units on their own streams, outputs merged -- bit for bit
    what upload + run + download of the whole batch gives, in every mode, step after step."""
    pb, _ = synth.make_heavy_tail(20261024, 90, s_max=200, r_max=3000)
    pipe = lg.Pipeline(gpu_ctx, pb, n_chunks)
    b = lg.Batch(gpu_ctx, pb)
    b.upload()
    for mode in (lg.MODE_HET_ONLY, lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS, lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET):
        for mc in (6, 3):
            b.run(mc, mode)
            want = b.download()
            got = pipe.step(mc, mode)
            assert got.n_records == want.n_records and got.n_candidates == want.n_candidates
            assert np.array_equal(got.records, want.records)
            assert np.array_equal(got.unit_rec_off, want.unit_rec_off)
            assert np.array_equal(got.site_mean, want.site_mean, equal_nan=True)
            assert np.array_equal(got.site_cnt, want.site_cnt)
            if mode & lg.MODE_EMIT_COUNTS:
                assert np.array_equal(got.counts, want.counts)
            # packed two-plane input and split-record output: same rows, same means
            packed = pipe.step(mc, mode | lg.MODE_SPLIT_RECORDS, packed=True)
            assert packed.rec_mi is not None and packed.rec_ij.dtype == np.uint32
            assert np.array_equal(packed.records, want.records)
            assert np.array_equal(packed.site_mean, want.site_mean, equal_nan=True)
            assert np.array_equal(packed.unit_rec_off, want.unit_rec_off)
            if mode & lg.MODE_EMIT_COUNTS:
                assert np.array_equal(packed.counts, want.counts)
            # the tight two-plane input (no 128-read padding) and the compact output (4-byte (i, j) here: a unit
            # has more than 256 sites... or not; no per-site count over the wire: recounted from the rows)
            tight = pipe.step(mc, mode | lg.MODE_COMPACT_OUTPUT, tight=True)
            assert tight.rec_ij.dtype == (np.uint16 if int(pb.units['n_sites'].max()) <= 256 else np.uint32)
            assert np.array_equal(tight.records, want.records)
            assert np.array_equal(tight.site_mean, want.site_mean, equal_nan=True)
            if mode & lg.MODE_HET_ONLY:                         # site_cnt counts het-kept rows: the rows of these modes
                assert np.array_equal(tight.site_cnt, want.site_cnt)
            # the launch chain as a CUDA graph: same bits, replayed
            for _ in range(2):
                b.run(mc, mode | lg.MODE_GRAPH)
                g = b.download()
                assert np.array_equal(g.records, want.records) and np.array_equal(g.site_mean, want.site_mean, equal_nan=True)
                assert g.kernel_ms == 0.0
    pipe.close()
    b.close()


def test_compact_rows_use_two_byte_site_indices(lg, gpu_ctx):
    """MODE_COMPACT_OUTPUT with no unit above 256 sites: (i, j) as i | j << 8 in a uint16 array."""
    pb = synth.make_uniform_planes(77, 300, 50, 200, 0.5)
    pipe = lg.Pipeline(gpu_ctx, pb, 3)
    want = pipe.step(6, lg.MODE_HET_ONLY)
    got = pipe.step(6, lg.MODE_HET_ONLY | lg.MODE_COMPACT_OUTPUT, tight=True)
    assert got.rec_ij.dtype == np.uint16 and got._site_cnt is None
    assert np.array_equal(got.records, want.records)
    assert np.array_equal(got.site_cnt, want.site_cnt) and np.array_equal(got.site_mean, want.site_mean, equal_nan=True)
    pipe.close()


def test_two_pipelines_with_steps_in_flight(lg, gpu_ctx):
    """lgmi_pipeline_begin* / lgmi_pipeline_finish: two pipelines over DIFFERENT batches on one context, the
    next step begun before the previous one is collected, round after round -- every result equals the
    synchronous step of its own batch, bit for bit; a second begin or a finish without a begin is an
    error and leaves the pipeline usable."""
    pbs = [synth.make_heavy_tail(20261101 + k, 70, s_max=150, r_max=2500)[0] for k in range(2)]
    pipes = [lg.Pipeline(gpu_ctx, pb, 3) for pb in pbs]
    mode = lg.MODE_HET_ONLY | lg.MODE_COMPACT_OUTPUT
    want = [p.step(6, mode, tight=True) for p in pipes]
    assert not np.array_equal(want[0].site_mean, want[1].site_mean, equal_nan=True)
    with pytest.raises(lg.LgmiError) as e:
        pipes[0].finish()
    assert e.value.code == -4
    inputs = [pb.packed2(tight=True) for pb in pbs]
    pipes[0].begin(6, mode, inputs[0], tight=True)
    with pytest.raises(lg.LgmiError) as e:
        pipes[0].begin(6, mode, inputs[0], tight=True)
    assert e.value.code == -4
    for r in range(1, 8):                                         # begin (r), then collect (r - 1)
        k = r & 1
        pipes[k].begin(6, mode, inputs[k], tight=True)
        got = pipes[k ^ 1].finish()
        w = want[k ^ 1]
        assert got.n_records == w.n_records
        assert np.array_equal(got.records, w.records)
        assert np.array_equal(got.unit_rec_off, w.unit_rec_off)
        assert np.array_equal(got.site_mean, w.site_mean, equal_nan=True)
    got = pipes[1].finish()
    assert np.array_equal(got.records, want[1].records)
    # three in flight with the downloads of the next step queued before the previous one is waited for:
    # begin(k + 2); collect(k + 1); finish(k)
    pbs.append(synth.make_heavy_tail(20261103, 40, s_max=120, r_max=2000)[0])
    pipes.append(lg.Pipeline(gpu_ctx, pbs[2], 2))
    inputs.append(pbs[2].packed2(tight=True))
    want.append(pipes[2].step(6, mode, tight=True))
    with pytest.raises(lg.LgmiError) as e:
        pipes[2].collect()
    assert e.value.code == -4
    for k in range(9):
        pipes[k % 3].begin(6, mode, inputs[k % 3], tight=True)
        if k >= 1:
            pipes[(k - 1) % 3].collect()
            pipes[(k - 1) % 3].collect()                          # (idempotent)
        if k >= 2:
            got, w = pipes[(k - 2) % 3].finish(), want[(k - 2) % 3]
            assert np.array_equal(got.records, w.records) and np.array_equal(got.unit_rec_off, w.unit_rec_off)
            assert np.array_equal(got.site_mean, w.site_mean, equal_nan=True)
    for k in (7, 8):
        got, w = pipes[k % 3].finish(), want[k % 3]
        assert np.array_equal(got.records, w.records) and np.array_equal(got.site_mean, w.site_mean, equal_nan=True)
    # the same through the host helper: lg.stream_steps over three pipelines of one shape
    same = [lg.Pipeline(gpu_ctx, pbs[2], 1) for _ in range(3)]
    feed = ((inputs[2], pbs[2].site_flags) for _ in range(7))
    seen = []
    for k, got in lg.stream_steps(same, feed, 6, mode, tight=True):
        seen.append(k)
        assert np.array_equal(got.records, want[2].records) and np.array_equal(got.site_mean, want[2].site_mean, equal_nan=True)
    assert seen == list(range(7))
    for p in same:
        p.close()
    # and the synchronous call still works on both afterwards
    for p, w in zip(pipes, want):
        assert np.array_equal(p.step(6, mode, tight=True).records, w.records)
        p.close()


def test_pipeline_needs_back_to_back_units(lg, gpu_ctx):
    pb = synth.make_uniform_planes(3, 4, 5, 40, 0.5)
    bad = lg.PlaneBatch(pb.units[::-1].copy(), pb.planes, pb.site_flags)
    with pytest.raises(lg.LgmiError) as e:
        lg.Pipeline(gpu_ctx, bad, 2)
    assert e.value.code == -6


# --------------------------------------------------------------------------- full-size properties (cfg2)
@pytest.fixture(scope="module")
def cfg2(lg):
    return synth.make_uniform(20261020, 20000, 50, 200, 0.5, chunk=500)


def test_cfg2_full_size_properties(lg, gpu_ctx, cfg2):
    pb = cfg2.plane_batch()
    assert pb.n_candidates == 24_500_000
    b = lg.Batch(gpu_ctx, pb)
    b.upload()
    b.run(6, lg.MODE_ALL_PAIRS)
    r1 = b.download()
    b.run(6, lg.MODE_ALL_PAIRS)
    r2 = b.download()
    assert np.array_equal(r1.records, r2.records)                         # deterministic, bit for bit
    assert np.array_equal(r1.site_mean, r2.site_mean, equal_nan=True)
    rec = r1.records
    # reference row order: unit, then i, then j
    key = rec['unit'].astype(np.int64) * (1 << 32) + rec['i'].astype(np.int64) * (1 << 16) + rec['j']
    assert np.all(np.diff(key) > 0)
    assert np.all(rec['i'] < rec['j']) and rec['j'].max() < 50
    assert np.array_equal(np.searchsorted(rec['unit'], np.arange(20001)), r1.unit_rec_off.astype(np.int64))
    assert np.all(rec['mi'] >= 0.0) and np.all(rec['mi'] <= math.log(3) + 1e-12)
    # per-site mean recomputed on the host from the emitted records (any order-insensitive check)
    flags = pb.site_flags & 3
    site = np.arange(20000 * 50).reshape(20000, 50)
    gi, gj = site[rec['unit'], rec['i']], site[rec['unit'], rec['j']]
    keep = (flags[gi] == 2) | (flags[gj] == 2)
    tot = np.bincount(gi[keep], rec['mi'][keep], 20000 * 50) + np.bincount(gj[keep], rec['mi'][keep], 20000 * 50)
    cnt = np.bincount(gi[keep], minlength=20000 * 50) + np.bincount(gj[keep], minlength=20000 * 50)
    assert np.array_equal(cnt, r1.site_cnt)
    with np.errstate(invalid='ignore', divide='ignore'):
        assert np.allclose(tot / cnt, r1.site_mean, rtol=1e-12, atol=1e-15, equal_nan=True)
    # a random sample of units against the oracle
    rng = np.random.default_rng(1)
    for g in rng.choice(20000, 40, replace=False).tolist():
        i, j, mi, tab, mean, cnt_o = oracle_unit(cfg2.encoded(g), 6)
        u = r1.unit_records(g)
        assert u['i'].tolist() == i.tolist() and u['j'].tolist() == j.tolist()
        assert_mi_close(u['mi'], mi)
        assert_mi_close(r1.site_mean[g * 50:(g + 1) * 50], mean)
    b.close()


def _order_and_mean_properties(pb, res):
    """Size-independent checks on a full-size result: reference row order, offsets, MI range, and the
    per-site counts / means recomputed on the host from the emitted rows."""
    rec = res.records
    key = rec['unit'].astype(np.int64) * (1 << 32) + rec['i'].astype(np.int64) * (1 << 16) + rec['j']
    assert np.all(np.diff(key) > 0)
    S = pb.units['n_sites'].astype(np.int64)
    assert np.all(rec['i'] < rec['j']) and np.all(rec['j'] < S[rec['unit']])
    assert np.array_equal(np.searchsorted(rec['unit'], np.arange(pb.n_units + 1)), res.unit_rec_off.astype(np.int64))
    assert np.all(rec['mi'] >= 0.0) and np.all(rec['mi'] <= math.log(3) + 1e-12)
    off = pb.units['site_off'].astype(np.int64)
    flags = pb.site_flags & 3
    gi, gj = off[rec['unit']] + rec['i'], off[rec['unit']] + rec['j']
    keep = (flags[gi] == 2) | (flags[gj] == 2)
    tot = np.bincount(gi[keep], rec['mi'][keep], pb.n_sites) + np.bincount(gj[keep], rec['mi'][keep], pb.n_sites)
    cnt = np.bincount(gi[keep], minlength=pb.n_sites) + np.bincount(gj[keep], minlength=pb.n_sites)
    assert np.array_equal(cnt, res.site_cnt)
    with np.errstate(invalid='ignore', divide='ignore'):
        assert np.allclose(tot / cnt, res.site_mean, rtol=1e-12, atol=1e-15, equal_nan=True)


def test_cfg4_full_size_properties_and_oracle_sample(lg, gpu_ctx):
    """BASELINE.json configs[3] at full size (20 000 heavy-tailed units, 32 M pairs, every kernel path in one
    batch): order / offsets / means as properties, deterministic, mid-depth units identical on the tensor-core
    and the popcount path, and a sample of units of every path against the oracle."""
    pb, raw = synth.make_heavy_tail(20261023, 20000, keep_raw=True)
    S, R = pb.units['n_sites'].astype(np.int64), pb.units['n_reads'].astype(np.int64)
    out = {}
    try:
        for path in (2, 0):
            gpu_ctx.set_tile_path(path)
            b = lg.Batch(gpu_ctx, pb)
            b.upload()
            b.run(6, lg.MODE_ALL_PAIRS)
            out[path] = b.download()
            if path:
                b.run(6, lg.MODE_ALL_PAIRS)
                again = b.download()
                assert np.array_equal(again.records, out[path].records)                  # deterministic
            b.close()
    finally:
        gpu_ctx.set_tile_path(2)                                # (the default)
    res = out[2]                             # many tiles per CTA here: the tile-to-tile hand-over of k_tile_gram_ws
    assert np.array_equal(res.records, out[0].records)
    assert np.array_equal(res.site_mean, out[0].site_mean, equal_nan=True)
    assert np.array_equal(res.site_cnt, out[0].site_cnt)
    _order_and_mean_properties(pb, res)
    rng = np.random.default_rng(2)
    small = np.flatnonzero((S <= 64) & (R <= 256) & (S >= 2))
    mid = np.flatnonzero(((S > 64) | (R > 256)) & (S * S * R < 4e8) & (S >= 2))
    big = np.flatnonzero(((S > 64) | (R > 256)) & (S * S * R >= 4e8) & (S * S * R < 6e9))
    picks = rng.choice(small, 12, replace=False).tolist() + rng.choice(mid, 16, replace=False).tolist() + \
        rng.choice(big, min(4, len(big)), replace=False).tolist()
    for g in picks:
        a, k = raw[g]
        eu = enc.EncodedUnit([1000 + 37 * s for s in range(a.shape[0])],
                             [("mismatch", "snp", "het_snp")[int(x)] for x in k], synth.labels_from_alleles(a))
        i, j, mi, tab, mean, cnt_o = oracle_unit(eu, 6)
        u = res.unit_records(g)
        assert u['i'].tolist() == i.tolist() and u['j'].tolist() == j.tolist(), "pair set of unit %d" % g
        assert_mi_close(u['mi'], mi)
        o = int(pb.units['site_off'][g])
        assert_mi_close(res.site_mean[o:o + eu.n_sites], mean)
        assert res.site_cnt[o:o + eu.n_sites].tolist() == cnt_o.tolist()


@pytest.mark.parametrize("cov", [0.01, 0.05, 0.1, 0.25, 0.5])
def test_cfg5_full_size_oracle_sample(lg, gpu_ctx, cov):
    """BASELINE.json configs[4] at full size: 20 000 units per grid point; per point the size-independent
    properties, and 6 sampled units against the oracle (pair set, MI, means)."""
    sb = synth.make_uniform(20261030 + int(cov * 1000), 20000, 50, 200, cov)
    pb = sb.plane_batch()
    b = lg.Batch(gpu_ctx, pb)
    b.upload()
    rng = np.random.default_rng(int(cov * 1000))
    picks = rng.choice(20000, 6, replace=False).tolist()
    survivors = []
    for mc in (6, 10, 20, 50):
        b.run(mc, lg.MODE_ALL_PAIRS)
        res = b.download()
        survivors.append(res.n_records)
        _order_and_mean_properties(pb, res)
        for g in picks:
            i, j, mi, tab, mean, cnt_o = oracle_unit(sb.encoded(g), mc)
            u = res.unit_records(g)
            assert u['i'].tolist() == i.tolist() and u['j'].tolist() == j.tolist()
            assert_mi_close(u['mi'], mi)
            assert_mi_close(res.site_mean[g * 50:(g + 1) * 50], mean)
    assert survivors == sorted(survivors, reverse=True)
    b.close()


def test_read_permutation_and_label_swap_invariance(lg, gpu_ctx):
    """MI does not depend on read order, nor on which of two alleles is called
    major when no third allele is present."""
    rng = np.random.default_rng(12)
    a, k = synth.draw_alleles(rng, 1, 40, 333, 0.6)
    lab = synth.labels_from_alleles(a[0])
    types = [("mismatch", "snp", "het_snp")[int(x)] for x in k[0]]
    eu0 = enc.EncodedUnit(list(range(40)), types, lab)
    eu1 = enc.EncodedUnit(list(range(40)), types, lab[:, rng.permutation(333)])
    swapped = lab.copy()
    bi = ~(lab == 0).any(axis=1)
    swapped[bi] = np.where(lab[bi] == 2, 1, np.where(lab[bi] == 1, 2, lab[bi]))
    eu2 = enc.EncodedUnit(list(range(40)), types, swapped)
    res = lg.mi_step_batched(lg.pack_units([eu0, eu1, eu2]), 6, lg.MODE_ALL_PAIRS, ctx=gpu_ctx)
    r0, r1, r2 = (res.unit_records(u) for u in range(3))
    assert np.array_equal(r0['i'], r1['i']) and np.array_equal(r0['j'], r1['j'])
    assert np.array_equal(r0['mi'], r1['mi'])                 # integer counts are identical -> same bits
    assert np.array_equal(r0['i'], r2['i'])
    assert_mi_close(r2['mi'], r0['mi'])


# --------------------------------------------------------------------------- global pass
def test_ecdf_drop_in_matches_reference(lg, gpu_ctx, golden):
    for case in golden("ecdf.json")["functions"]:
        fn = lg.ecdf([unhex(v) for v in case["x"]])
        samples = np.array([unhex(v) for v in case["samples"]])
        want = np.array([unhex(v) for v in case["y"]])
        assert np.array_equal(fn(samples), want)              # bit-exact: same linspace arithmetic
        one = fn(float(samples[0]))
        assert np.ndim(one) == 0 and isinstance(one, np.floating) and one == want[0]      # scalar in, scalar out
        assert np.ndim(fn(np.float64(samples[0]))) == 0
    k = golden("kat.json")["ecdf"]
    assert lg.ecdf(k["x"])(np.array(k["samples"])).tolist() == [0, 0, 0.25, 0.75, 0.75, 1.0]
    with pytest.raises(ZeroDivisionError):
        lg.ecdf([])


def test_mip_and_threshold_calls_match_reference(lg, gpu_ctx, golden):
    tab = golden("ecdf.json")["site_table"]
    mean = np.array([unhex(v) for v in tab["mean"]])
    mip, call = lg.mip_and_calls(mean, tab["type"], tab["threshold"], ctx=gpu_ctx)
    want = np.array([unhex(v) for v in tab["mip"]])
    assert np.array_equal(mip, want, equal_nan=True)
    assert (call == 1).tolist() == tab["positive"]
    assert (call == 2).tolist() == tab["negative"]


def test_mip_large_random_vs_oracle(lg, gpu_ctx):
    rng = np.random.default_rng(3)
    n = 300_000
    mean = rng.random(n).round(4)                             # plenty of ties
    mean[rng.random(n) < 0.3] = np.nan
    code = rng.choice(np.array([0, 1, 2], np.uint8), n, p=[0.85, 0.05, 0.10])
    for thr in (0.05, 0.5):
        mip, call = lg.mip_and_calls(mean, code, thr, ctx=gpu_ctx)
        wmip, wcall = c_oracle.mip_calls(mean, code, thr)
        assert np.array_equal(mip, wmip, equal_nan=True)
        assert np.array_equal(call, wcall)
    # no het SNP at all -> everything NaN / no call
    mip, call = lg.mip_and_calls(mean, np.zeros(n, np.uint8), 0.05, ctx=gpu_ctx)
    assert np.isnan(mip).all() and not call.any()


def test_end_to_end_calls_identical(lg, gpu_ctx, cfg2):
    """units -> MI -> mean -> mip -> call on the GPU vs the oracle chain, on 300
    units: every site's call at mi_p_threshold must be identical."""
    idx = list(range(300))
    eus = [cfg2.encoded(g) for g in idx]
    res = lg.mi_step_batched(lg.pack_units(eus), 6, lg.MODE_HET_ONLY, ctx=gpu_ctx)
    want_mean = np.concatenate([oracle_unit(eu, 6)[4] for eu in eus])
    assert_mi_close(res.site_mean, want_mean)
    code = np.concatenate([[c_oracle.TYPE_CODE[t] for t in eu.types] for eu in eus]).astype(np.uint8)
    mip, call = lg.mip_and_calls(res.site_mean, code, 0.05, ctx=gpu_ctx)
    wmip, wcall = c_oracle.mip_calls(want_mean, code, 0.05)
    assert np.array_equal(call, wcall)
    assert_mi_close(mip, wmip)


# --------------------------------------------------------------------------- errors
def test_argument_errors(lg, gpu_ctx):
    pb = synth.make_uniform_planes(1, 2, 5, 40, 0.5)
    bad = lg.PlaneBatch(pb.units.copy(), pb.planes, pb.site_flags)
    bad.units['row_words'][0] = 3
    with pytest.raises(lg.LgmiError) as e:
        lg.Batch(gpu_ctx, bad)
    assert e.value.code == -2
    b = lg.Batch(gpu_ctx, pb)
    with pytest.raises(lg.LgmiError) as e:
        b.run(6)                                               # nothing uploaded
    assert e.value.code == -4
    b.upload()
    with pytest.raises(lg.LgmiError):
        b.run(6, lg.MODE_SKIP_NONHET)                          # needs HET_ONLY
    b.close()
    assert gpu_ctx.launch_count > 0
