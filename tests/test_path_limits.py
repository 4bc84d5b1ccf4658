"""Each count path on both sides of the capacity limits of its packed counts, against the C oracle.

Every count path keeps its counts in a narrow field or a capped list, and the plan (or the kernel itself) sends a
unit elsewhere before that storage would overflow.  An off-by-one or a wrong cadence there gives wrong integers, not
a fault, on inputs real data has (highly expressed genes, sites with many third alleles).  The units here are built
label by label to sit exactly at each limit and one past it: pair sets and 3x3 tables bit-exact against the oracle,
MI and means within conftest's tolerance, and bit for bit against a second device path wherever one exists.

Labels are uint8 matrices [sites, reads]: 2 major, 1 minor, 0 "other" (a third allele), 255 not covered.  The last
test checks on the CPU that every construction hits its target, so that a later edit of a generator cannot move a
unit off its limit unnoticed.
"""
import importlib

import numpy as np
import pytest

from conftest import assert_mi_close
from parity import _check_split, c_oracle, check_batch, oracle_unit, signed

enc = importlib.import_module("l-giremi_b200.encode")

TYPES = ("mismatch", "snp", "het_snp")
RAISED = (1 << 20, 1 << 30)             # a dense threshold no unit reaches


# --------------------------------------------------------------------------- constructions
def _rows(rng, S, R, third=0.0):
    """Background labels [S, R], one site at a time from 16-bit draws (no float arrays of the unit's size): per site
    a coverage in [0.3, 0.95] and a share of reads whose allele follows one read haplotype shared by all sites (so
    that pairs are linked and MI is not just noise); `third` of the covered reads are "other"."""
    hap = rng.integers(0, 2, R, dtype=np.uint8)
    lab = np.empty((S, R), np.uint8)
    t = int(third * 32768)
    for s in range(S):
        cov = int(rng.uniform(0.3, 0.95) * 65536)
        link = int(rng.uniform(0.0, 0.9) * 65536)
        c, li, a = (rng.integers(0, 65536, R, dtype=np.uint16) for _ in range(3))
        row = (1 + np.where(li < link, hap, a & 1)).astype(np.uint8)
        if t:
            row[(a >> 1) < t] = 0
        row[c >= cov] = 255
        lab[s] = row
    return lab


def _full_pair(rng, lab, i, j, third):
    """Sites i and j covered on every read; j repeats i's label on about 80 % of them."""
    R = lab.shape[1]
    a, b, c = (rng.integers(0, 65536, R, dtype=np.uint16) for _ in range(3))
    t = int(third * 32768)
    lab[i] = 1 + (a & 1)
    lab[i][(a >> 1) < t] = 0
    lab[j] = lab[i]
    redraw = b < 13107
    lab[j][redraw] = 1 + (c[redraw] & 1)
    lab[j][redraw & ((c >> 1) < t)] = 0


def _unit(rng, lab, types=None):
    S = lab.shape[0]
    if types is None:
        types = [TYPES[int(k)] for k in rng.integers(0, 3, S)]
    return enc.EncodedUnit([1000 + 37 * s for s in range(S)], types, lab)


def table(lab, i, j):
    """The oracle's 3x3 table of sites i, j (label order other, minor, major), on the host."""
    T = np.zeros((3, 3), np.int64)
    for a in range(3):
        for b in range(3):
            T[a, b] = np.count_nonzero((lab[i] == a) & (lab[j] == b))
    return T


def n_other(lab):
    return np.count_nonzero(lab == 0, axis=1)


# (a) the small path: kOthCap = 7 "other" reads per site
K_OTH_CAP = 7
SMALL_SHAPES = [(12, 200), (12, 256), (64, 200), (64, 256)]
A_ONE_WORD = np.arange(7)                                    # site 0: seven in read word 0
B_SEVEN_WORDS = 32 * np.arange(7) + 5                        # site 1: one in each of words 0 .. 6
C_TWO_HALVES = np.array([122, 123, 124, 125, 128, 129, 130])  # site 2: four below read 128, three above
Z_READS = np.arange(64, 71)                                  # the last site's seven (word 2)
EXTRA_SAME_WORD, EXTRA_OTHER_WORD = 7, 40                    # site 0's eighth


def small_unit(S, R, extra=None, a_het=True):
    """S <= 64, R <= 256 with five sites at exactly seven "other" reads and crafted partners that bring each of the
    five packed cells of a pair to 7:  T[0][0] of (0, 3) (both "other" on the same reads), T[0][1] / T[0][2] of
    (0, 4) / (0, 5) (the site first, its partner minor / major there), T[1][0] / T[2][0] of (6, S-1) / (7, S-1)
    (the site second).  Every other site is a partner of sites 0 and S-1 on their "other" reads with probability
    its coverage, so that pairs of both parities (both 16-bit halves of ocell) get "other" cells.  `extra`: a read
    that becomes site 0's eighth "other" read, with sites 4 and 5 minor / major on it (cells of 8: over the cap)."""
    rng = np.random.default_rng(1000 * S + R)
    lab = _rows(rng, S, R)                                   # no "other" label anywhere else
    types = [TYPES[int(k)] for k in rng.integers(0, 3, S)]
    Z = S - 1
    lab[0, A_ONE_WORD] = 0
    lab[1, B_SEVEN_WORDS] = 0
    lab[2, C_TWO_HALVES] = 0
    lab[3, A_ONE_WORD] = 0
    lab[4, A_ONE_WORD] = 1
    lab[5, A_ONE_WORD] = 2
    lab[Z, Z_READS] = 0
    lab[6, Z_READS] = 1
    lab[7, Z_READS] = 2
    for s, t in ((0, "het_snp"), (1, "het_snp"), (3, "snp"), (4, "het_snp"), (5, "het_snp"), (6, "mismatch"),
                 (7, "mismatch"), (Z, "het_snp")):
        types[s] = t
    if extra is not None:
        lab[0, extra] = 0
        lab[4, extra] = 1
        lab[5, extra] = 2
    if not a_het:
        types[0] = "mismatch"                                # only its het partners' pairs are evaluated
    return _unit(rng, lab, types)


def small_batch():
    """Per shape: the unit at the cap, its twins with site 0 at eight in the same word and in another word, and the
    same-word twin with site 0 non-het."""
    eus = []
    for S, R in SMALL_SHAPES:
        eus += [small_unit(S, R), small_unit(S, R, EXTRA_SAME_WORD), small_unit(S, R, EXTRA_OTHER_WORD),
                small_unit(S, R, EXTRA_SAME_WORD, a_het=False)]
    return eus


# (b) the mid-depth tensor path: kTgMaxReads = 65535 (nine u16 counts per pair in k_tile_gram_ws)
K_TG_MAX_READS = 65535


def mid_unit(S, R):
    """Sites S // 3 and S - 1 identical, covered on every read and major on all (T[2][2] = N = R); sites 1, 2 a
    2x2 pair and sites 3, 4 a 3x3 pair covered on every read; the rest background with a few "other" reads."""
    rng = np.random.default_rng(S * 100003 + R)
    lab = _rows(rng, S, R, third=0.002)
    lab[S // 3] = 2
    lab[S - 1] = 2
    _full_pair(rng, lab, 1, 2, 0.0)
    _full_pair(rng, lab, 3, 4, 0.3)
    return _unit(rng, lab)


# (c) the deep four-block form: the list cap max(kDenseOthMin, R / kDenseOthDiv) and k_other_fix's byte counters
def oth_cap(R):
    return max(256, R // 64)


def listed_unit(S, R, s, extra=False, far=()):
    """Site s with exactly oth_cap(R) "other" reads (one more with extra=True), spread evenly over the reads, so
    over many 256-read blocks of k_dense_prep.  Its partners on those reads: s-3 / s+1 major on all, s-2 / s+2
    minor on all, s-1 / s+3 "other" on all (each itself at the cap), s+4 covering none; `far` = three more sites
    (major, minor, "other"), e.g. below the row limit of a piece.  k_other_fix's two parity warps per label each
    count half of the listed reads: more than the 252 its byte counters hold between flushes once the cap is past
    504."""
    n = oth_cap(R)
    rng = np.random.default_rng(S * 7919 + R + s)
    lab = _rows(rng, S, R, third=0.003)
    reads = np.linspace(0, R - 1, n).round().astype(np.int64)
    crafted = [s, s - 1, s + 3] + ([far[2]] if far else [])  # rows that hold exactly these "other" reads
    for t in crafted:
        lab[t][lab[t] == 0] = 2
    for t, v in zip((s - 3, s - 2, s - 1, s, s + 1, s + 2, s + 3, s + 4), (2, 1, 0, 0, 2, 1, 0, 255)):
        lab[t, reads] = v
    for t, v in zip(far, (2, 1, 0)):
        lab[t, reads] = v
    if extra:
        lab[s, reads[0] + 1] = 0
    types = [TYPES[int(k)] for k in rng.integers(0, 3, S)]
    types[s] = "het_snp"
    return _unit(rng, lab, types)


LISTED = [(60, 9000, 30, False), (60, 9000, 30, True), (60, 40000, 30, False), (60, 40000, 30, True)]
SPLIT = dict(S=200, R=40000, s=150, far=(10, 11, 12))
SPLIT_BOUNDS = [0, 128, 200]


# (d) the deep path across kFastMathMaxCount = 2^21 - 1
K_FAST_MATH_MAX_COUNT = (1 << 21) - 1


def big_unit(R):
    """48 sites: 0 and 1 identical, covered on every read, major on all (T[2][2] = R); 2, 3 a 3x3 pair and 4, 5 a
    2x2 pair, both covered on every read; the rest background with a few "other" reads."""
    rng = np.random.default_rng(R)
    lab = _rows(rng, 48, R, third=0.001)
    lab[0] = 2
    lab[1] = 2
    _full_pair(rng, lab, 2, 3, 0.3)
    _full_pair(rng, lab, 4, 5, 0.0)
    return _unit(rng, lab)


BIG_SUB = np.array([0, 1, 2, 3, 4, 5, 9, 17, 23, 31, 40, 47])    # the sub-unit the oracle checks


# (e) MODE_COMPACT_OUTPUT: (i, j) in two bytes while no unit has more than 256 sites
def compact_unit(S, seed):
    """S sites x 120 reads; the last two sites covered on every read, the last one het: pair (S-2, S-1) is kept."""
    rng = np.random.default_rng(seed)
    lab = _rows(rng, S, 120, third=0.01)
    _full_pair(rng, lab, S - 2, S - 1, 0.0)
    types = [TYPES[int(k)] for k in rng.integers(0, 3, S)]
    types[S - 1] = "het_snp"
    return _unit(rng, lab, types)


# --------------------------------------------------------------------------- device runs
@pytest.fixture()
def ctx(lg, gpu_ctx):
    """The shared context; the dense threshold, the dense form and the tile path are set back to their defaults
    afterwards, whatever the test did."""
    yield gpu_ctx
    gpu_ctx.set_dense_threshold(*lg.DENSE_DEFAULT)
    gpu_ctx.set_dense_path(4)
    gpu_ctx.set_tile_path(2)


def _modes(lg):
    return [lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS, lg.MODE_HET_ONLY, lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET]


def _same(a, b):
    """Two results of the same batch, bit for bit."""
    assert a.n_records == b.n_records
    assert np.array_equal(a.records.view(np.uint8), b.records.view(np.uint8))
    assert np.array_equal(a.unit_rec_off, b.unit_rec_off)
    assert (a.counts is None) == (b.counts is None)
    if a.counts is not None:
        assert np.array_equal(a.counts, b.counts)
    assert np.array_equal(a.site_mean.view(np.uint64), b.site_mean.view(np.uint64))
    assert np.array_equal(a.site_cnt, b.site_cnt)


def _has_pair(res, unit, i, j):
    rec = res.unit_records(unit)
    return bool(np.any((rec['i'] == i) & (rec['j'] == j)))


def _check_sub(res, unit, lab, idx, mc):
    """The rows of `res` (ALL_PAIRS | EMIT_COUNTS) between sites of idx (ascending) against the oracle on the
    sub-unit lab[idx]: the same pairs in the same order, the same tables, MI within tolerance."""
    i, j, mi, tab = c_oracle.unit_pairs_from_labels(signed(lab[idx]), None, mc)
    rec, cnt = res.unit_records(unit), res.unit_counts(unit)
    inside = np.isin(rec['i'], idx) & np.isin(rec['j'], idx)
    key = rec['i'][inside].astype(np.int64) * 65536 + rec['j'][inside]
    assert np.array_equal(key, idx[i].astype(np.int64) * 65536 + idx[j]), "pair set of the sub-unit"
    assert np.array_equal(cnt[inside].astype(np.int64), tab), "3x3 counts of the sub-unit"
    assert_mi_close(rec['mi'][inside], mi, 0.9, "sub-unit MI")
    return tab


@pytest.mark.gpu
def test_small_path_seven_and_eight_other_reads(lg, ctx):
    """kOthCap = 7 (lgmi_fast.cuh): k_pairs_fast packs the five "other" cells of a pair into 3-bit fields of ocell
    and lists at most 7 "other" reads per site; a site with 8 sends its unit to k_pairs_generic<0>.  Units at
    exactly 7 in every layout and cell (small_unit), their twins at 8 (same word, another word, and a non-het site
    for HET_ONLY | SKIP_NONHET), at 12 and 64 sites and 200 and 256 reads (the NW = 7 and NW = 8 count paths, both
    128-read halves), at min_common 1, 6, N and N + 1 with N the common reads of the crafted pair (0, 5), "other"
    reads included; then the same batch forced onto the deep path, bit for bit."""
    eus = small_batch()
    lab0 = eus[0].labels
    N = int(np.count_nonzero((lab0[0] != 255) & (lab0[5] != 255)))
    assert N > 20
    for mc in (1, 6, N, N + 1):
        full = check_batch(lg, ctx, eus, mc)
        assert _has_pair(full, 0, 0, 5) == (mc <= N)
    pb = lg.pack_units(eus)
    small = [lg.mi_step_batched(pb, 6, m, ctx=ctx) for m in _modes(lg)]
    assert small[0].n_dense_units == 0
    ctx.set_dense_threshold(2, 1)
    for m, want in zip(_modes(lg), small):
        got = lg.mi_step_batched(pb, 6, m, ctx=ctx)
        assert got.n_dense_units == len(eus)
        _same(got, want)


@pytest.mark.gpu
def test_mid_depth_at_65535_and_65536_reads(lg, ctx):
    """kTgMaxReads = 65535 (lgmi_plan.h): k_tile_gram_ws stores nine u16 counts per pair, so a mid-depth unit with
    65 535 reads is counted there (the last k-block ragged: 511 x 128 + 127 reads) and one with 65 536 by k_tile_mi.
    In each a pair has T[2][2] = N = R, which a u16 would wrap to 0 at 65 536.  47 sites (below the dense
    threshold), then 130 sites x 65 535 reads with the threshold raised: 2 row blocks x 3 column blocks, 512
    k-blocks each.  Against the oracle, and tile path 2 bit for bit against tile path 0."""
    for eus, thr in (([mid_unit(47, K_TG_MAX_READS), mid_unit(47, K_TG_MAX_READS + 1)], None),
                     ([mid_unit(130, K_TG_MAX_READS)], RAISED)):
        if thr:
            ctx.set_dense_threshold(*thr)
        full = check_batch(lg, ctx, eus, 6, min_exact=0.9)
        assert full.n_dense_units == 0
        for u, eu in enumerate(eus):
            S, R = eu.labels.shape
            rec, cnt = full.unit_records(u), full.unit_counts(u)
            k = np.flatnonzero((rec['i'] == S // 3) & (rec['j'] == S - 1))
            assert len(k) == 1 and cnt[k[0], 8] == R and cnt[k[0]].sum() == R
        pb = lg.pack_units(eus)
        out = {}
        for path in (2, 0):
            ctx.set_tile_path(path)
            out[path] = [lg.mi_step_batched(pb, 6, m, ctx=ctx) for m in _modes(lg)]
        ctx.set_tile_path(2)
        for a, b in zip(out[2], out[0]):
            assert a.n_dense_units == 0
            _same(a, b)


@pytest.mark.gpu
def test_deep_four_blocks_list_cap_and_byte_flush(lg, ctx):
    """The four-block form of the deep path (lgmi_dense.cuh).  k_dense_prep lists up to max(kDenseOthMin = 256,
    R / kDenseOthDiv) "other" reads per site (lgmi_plan.h) and sends the unit to nine blocks when a reservation
    passes the cap (idx + n > cap); k_other_fix adds the listed reads' bit rows into byte counters flushed every 18
    rounds of 14 reads (252 per byte).  Units A / B: 9 000 reads (cap 256) with one site at 256 / 257; C / D:
    40 000 reads (cap 625) with one site at 625 / 626 and partners major, minor and "other" on all of them on both
    sides (slots 0-2 and 3 / 6), so that each parity warp counts 313 reads of one partner into one byte.  Against
    the oracle; nine blocks and the popcount path bit for bit."""
    eus = [listed_unit(S, R, s, extra) for S, R, s, extra in LISTED]
    four = check_batch(lg, ctx, eus, 6, min_exact=0.9)
    assert four.n_dense_units == 4 and four.n_dense_four == 2
    pb = lg.pack_units(eus)
    want = [lg.mi_step_batched(pb, 6, m, ctx=ctx) for m in _modes(lg)]
    rec, cnt = want[0].unit_records(2), want[0].unit_counts(2)
    k = np.flatnonzero((rec['i'] == 30) & (rec['j'] == 31))
    assert cnt[k[0], 2] == 625                              # slot 2 of (s, s + 1): "other" at s, major at s + 1
    ctx.set_dense_path(9)
    for m, w in zip(_modes(lg), want):
        got = lg.mi_step_batched(pb, 6, m, ctx=ctx)
        assert got.n_dense_units == 4 and got.n_dense_four == 0
        _same(got, w)
    ctx.set_dense_path(4)
    ctx.set_dense_threshold(*RAISED)
    for m, w in zip(_modes(lg), want):
        got = lg.mi_step_batched(pb, 6, m, ctx=ctx)
        assert got.n_dense_units == 0
        _same(got, w)


@pytest.mark.gpu
def test_deep_four_blocks_at_the_cap_split_by_rows(lg, ctx):
    """k_other_fix's row limit under heavy counts: a 200-site x 40 000-read unit like C of the test above, its
    site 150 at the cap of 625 with partners at 147-149, 151-154 and 10-12 (below the row limit of 128), run whole
    and as the pieces [0, 128) and [128, 200): the pieces' rows and the gathered means equal the whole unit's, bit
    for bit, in every mode, and the crafted sites against the oracle."""
    eu = listed_unit(**SPLIT)
    pb = lg.pack_units([eu])
    for m in _modes(lg):
        whole = _check_split(lg, ctx, pb, SPLIT_BOUNDS, m)
        assert whole.n_dense_units == 1 and whole.n_dense_four == 1
        if m & lg.MODE_EMIT_COUNTS:
            idx = np.array([3, 10, 11, 12, 77, 130, 147, 148, 149, 150, 151, 152, 153, 154, 199])
            tab = _check_sub(whole, 0, eu.labels, idx, 6)
            assert tab.max() >= 625


@pytest.mark.gpu
def test_deep_path_across_two_to_the_21_reads(lg, ctx):
    """kFastMathMaxCount = 2^21 - 1 (lgmi_fast.cuh): k_pairs_generic<2> evaluates MI with the reorganised epilogues
    (mi_2x2 / mi_3x3) for units of up to that many reads and with the straightforward arithmetic of lgmi_math.cuh
    above.  48 sites x 2^21 - 1 and x 2^21 reads, crafted pairs with N = R (2x2 and 3x3 tables): a 12-site sub-unit
    against the oracle, the whole units bit for bit against the popcount path (k_tile_mi).  The context's ln table
    grows to 2^22 entries here, built once on the host (lgmi_build_lntab in binary128: about 5 s on one core of an
    Intel Xeon)."""
    eus = [big_unit(K_FAST_MATH_MAX_COUNT), big_unit(K_FAST_MATH_MAX_COUNT + 1)]
    pb = lg.pack_units(eus)
    modes = [lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS, lg.MODE_HET_ONLY]
    dense = [lg.mi_step_batched(pb, 6, m, ctx=ctx) for m in modes]
    assert dense[0].n_dense_units == 2
    for u, eu in enumerate(eus):
        R = eu.n_reads
        tab = _check_sub(dense[0], u, eu.labels, BIG_SUB, 6)
        assert tab[0].tolist() == [0, 0, 0, 0, 0, 0, 0, 0, R]       # pair (0, 1)
        assert tab.sum(axis=1).max() == R and np.count_nonzero(tab, axis=1).max() == 9
    ctx.set_dense_threshold(*RAISED)
    for m, want in zip(modes, dense):
        got = lg.mi_step_batched(pb, 6, m, ctx=ctx)
        assert got.n_dense_units == 0
        _same(got, want)


@pytest.mark.gpu
def test_compact_rows_at_256_and_257_sites(lg, ctx):
    """MODE_COMPACT_OUTPUT: while no unit has more than 256 sites the pipelined step ships (i, j) as i | j << 8 in
    a uint16 (step_form, k_split_records); a unit of 257 sites makes it uint32.  Pair (254, 255) of a 256-site
    unit is emitted as 0xfffe and decoded; records and means equal the synchronous Batch run, which matches the
    oracle."""
    base = [compact_unit(256, 20261201 + k) for k in range(4)]
    for eus, dtype in ((base, np.uint16), (base[:2] + [compact_unit(257, 20261211)] + base[2:], np.uint32)):
        pb = lg.pack_units(eus)
        b = lg.Batch(ctx, pb)
        pipe = lg.Pipeline(ctx, pb, 3)
        try:
            b.upload()
            b.run(6, lg.MODE_HET_ONLY)
            want = b.download()
            got = pipe.step(6, lg.MODE_HET_ONLY | lg.MODE_COMPACT_OUTPUT, tight=True)
        finally:
            pipe.close()
            b.close()
        assert got.rec_ij.dtype == dtype and got._site_cnt is None
        _same(got, want)
        for u, eu in enumerate(eus):
            S = eu.n_sites
            assert _has_pair(got, u, S - 2, S - 1)
            i, j, mi, tab, mean, cnt = oracle_unit(eu, 6)
            het = np.array([t == "het_snp" for t in eu.types])
            keep = het[i] | het[j]
            rec = want.unit_records(u)
            assert rec['i'].tolist() == i[keep].tolist() and rec['j'].tolist() == j[keep].tolist()
            assert_mi_close(rec['mi'], mi[keep], 0.97)
            off = int(pb.units['site_off'][u])
            assert_mi_close(want.site_mean[off:off + S], mean, 0.97)
        if dtype == np.uint16:
            assert np.count_nonzero(got.rec_ij == (254 | 255 << 8)) == len(eus)


# --------------------------------------------------------------------------- the constructions, on the CPU
def test_constructions_hit_their_limits():
    """Every unit above sits where its docstring says: 7 and 8 "other" reads per site and the crafted cells of 7
    and 8 (a); T[2][2] = R around 65 535 (b); exactly cap and cap + 1 listed reads for both read counts, nobody
    else above the cap, more than 252 reads per k_other_fix parity warp, and the crafted slots (c); and the compact
    units' last pair (e).  (d)'s generator is checked at a small R: the same code as at 2^21."""
    for eu in small_batch():
        lab = eu.labels
        S, R = lab.shape
        Z = S - 1
        oth = n_other(lab)
        eighth = next((r for r in (EXTRA_SAME_WORD, EXTRA_OTHER_WORD) if lab[0, r] == 0), None)
        want = np.zeros(S, np.int64)
        want[[0, 1, 2, 3, Z]] = K_OTH_CAP
        want[0] += eighth is not None
        assert oth.tolist() == want.tolist()
        words = lambda s: sorted(set((np.flatnonzero(lab[s] == 0) // 32).tolist()))
        assert len(words(0)) == (2 if eighth == EXTRA_OTHER_WORD else 1)
        assert words(1) == list(range(7))
        assert (np.flatnonzero(lab[2] == 0) < 128).sum() == 4 and (np.flatnonzero(lab[2] == 0) >= 128).sum() == 3
        cell = K_OTH_CAP + (eighth is not None)
        assert table(lab, 0, 3)[0, 0] == K_OTH_CAP
        assert table(lab, 0, 4)[0, 1] == cell and table(lab, 0, 5)[0, 2] == cell
        assert table(lab, 6, Z)[1, 0] == K_OTH_CAP and table(lab, 7, Z)[2, 0] == K_OTH_CAP
        # partners t of site 0 covered on its "other" reads: pairs (0, t), index t - 1, of both parities (both
        # 16-bit halves of ocell)
        partners = [t for t in range(1, S) if ((lab[0] == 0) & (lab[t] != 255)).any()]
        assert {(t - 1) & 1 for t in partners} == {0, 1}
        if eu.types[0] != "het_snp":
            assert eighth is not None and eu.types[4] == eu.types[5] == "het_snp"
        assert set(np.unique(lab).tolist()) <= {0, 1, 2, 255}
    for S, R in ((47, K_TG_MAX_READS), (47, K_TG_MAX_READS + 1), (130, K_TG_MAX_READS)):
        lab = mid_unit(S, R).labels
        assert table(lab, S // 3, S - 1)[2, 2] == R
        assert table(lab, 1, 2).sum() == R and table(lab, 1, 2)[0].sum() + table(lab, 1, 2)[:, 0].sum() == 0
        assert table(lab, 3, 4).sum() == R and np.count_nonzero(table(lab, 3, 4)) == 9
    assert (K_TG_MAX_READS - 1) // 128 == 511 and K_TG_MAX_READS - 511 * 128 == 127
    for S, R, s, extra in LISTED + [(SPLIT["S"], SPLIT["R"], SPLIT["s"], False)]:
        far = SPLIT["far"] if S == SPLIT["S"] else ()
        lab = listed_unit(S, R, s, extra, far).labels
        cap = oth_cap(R)
        oth = n_other(lab)
        assert cap == (256 if R == 9000 else 625)
        assert oth[s] == cap + extra
        at_cap = [s - 1, s + 3] + ([far[2]] if far else [])
        assert all(oth[t] == cap for t in at_cap)
        rest = np.delete(oth, [s] + at_cap)
        assert rest.max() < cap and rest.max() > 0
        reads = np.flatnonzero(lab[s] == 0)
        assert len(set((reads // 256).tolist())) > 30             # many k_dense_prep blocks
        if R == 40000:
            assert (cap + 1) // 2 > 252                  # a parity warp's reads: the byte flush runs mid-stream
        n = cap
        for t, cell in ((s - 3, (2, 0)), (s - 2, (1, 0)), (s - 1, (0, 0)), (s + 1, (0, 2)), (s + 2, (0, 1)),
                        (s + 3, (0, 0))):
            T = table(lab, min(s, t), max(s, t))
            assert T[cell] - n in ((0, 1) if extra else (0,))      # (a twin's extra read may add one)
        assert not (lab[s + 4][lab[s] == 0] != 255).any()
        for t, cell in zip(far, ((2, 0), (1, 0), (0, 0))):
            assert table(lab, t, s)[cell] == n and t < SPLIT_BOUNDS[1] <= s
    lab = big_unit(5000).labels
    assert table(lab, 0, 1)[2, 2] == 5000 and np.count_nonzero(table(lab, 2, 3)) == 9
    assert table(lab, 4, 5).sum() == 5000 and np.count_nonzero(table(lab, 4, 5)) == 4
    assert K_FAST_MATH_MAX_COUNT + 1 == 1 << 21
    for S in (256, 257):
        eu = compact_unit(S, 1)
        assert table(eu.labels, S - 2, S - 1).sum() == 120 and eu.types[S - 1] == "het_snp"
