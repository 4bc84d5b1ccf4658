"""Deep units split by row blocks of their pair grid (lgmi_batch_create_rows, lgmi_split_means, DevicePool).

A piece of rows [a, b) of a unit is the suffix unit of sites [a, S) with row limit b - a.  The pieces' records, in
row order with i and j shifted by a, must be the whole unit's records, and the means gathered over the pieces the
unsplit run's, bit for bit.  The planner and the merge are host bookkeeping and run without a device."""
import importlib
import types

import numpy as np
import pytest
from numpy.random import PCG64, Generator

lg_mod = importlib.import_module("l-giremi_b200")
api = importlib.import_module("l-giremi_b200.api")
enc = importlib.import_module("l-giremi_b200.encode")
mg = importlib.import_module("l-giremi_b200.multigpu")
synth = importlib.import_module("l-giremi_b200.synth")

from parity import _check_split, _pieces  # noqa: E402


def _descs(shapes):
    u = np.zeros(len(shapes), dtype=lg_mod.UNIT_DESC)
    u['n_sites'] = [s for s, _r in shapes]
    u['n_reads'] = [r for _s, r in shapes]
    u['row_words'] = 4 * ((u['n_reads'] + 127) // 128)
    return u


def _cfg4_descs():
    S, R = synth.heavy_tail_shapes(Generator(PCG64(20261022)), 20000)    # make_heavy_tail(20261022, 20000)'s shapes
    return _descs(list(zip(S.tolist(), R.tolist())))


# --------------------------------------------------------------------------- planner, no device
@pytest.mark.parametrize("n_dev", [2, 4, 8])
def test_cfg4_is_never_split(n_dev):
    assert mg.split_plan(_cfg4_descs(), n_dev) == {}


@pytest.mark.parametrize("n_dev", [2, 4, 8])
def test_cfg4_with_the_cfg3_unit_splits_the_deep_unit(n_dev):
    units = np.concatenate([_cfg4_descs(), _descs([(2000, 100000)])])
    deep = len(units) - 1
    plan = mg.split_plan(units, n_dev)
    assert list(plan) == [deep]
    cost = api.unit_costs(units).astype(np.float64)
    m = min(n_dev, int(np.ceil(cost[deep] * n_dev / cost.sum())), 16)
    b = plan[deep]
    assert len(b) == m + 1 and b[0] == 0 and b[-1] == 2000
    assert all(x % 128 == 0 for x in b[:-1]) and all(x < y for x, y in zip(b, b[1:]))
    pairs = np.diff(mg._rows_pairs(2000, b))
    assert pairs.sum() == 2000 * 1999 // 2
    assert abs(pairs - pairs.sum() / m).max() <= mg._rows_pairs(2000, 128)      # within one (the largest) row block
    shards, pieces, splits = mg.plan_pieces(units, n_dev)
    assert splits == plan
    got = sorted((a, e) for p in pieces for u, a, e in p if u == deep)
    assert got == list(zip(b[:-1], b[1:]))
    assert sorted(np.concatenate(shards).tolist()) == list(range(deep))


def test_small_units_and_one_device_are_never_split():
    units = _descs([(128, 60000), (40, 100), (30, 50)])          # one unit is all the work, but has 128 sites
    assert mg.split_plan(units, 8) == {}
    assert mg.split_plan(_descs([(2000, 100000), (40, 100)]), 1) == {}


def test_split_rows_balances_at_the_largest_piece():
    for S, m in ((2000, 8), (2000, 3), (1000, 2), (300, 3), (4097, 5)):
        b = mg.split_rows(S, m)
        pairs = np.diff(mg._rows_pairs(S, b))
        assert len(b) == m + 1 and pairs.sum() == S * (S - 1) // 2
        # no other choice of boundaries at multiples of 128 has a smaller largest piece (exhaustive for m = 2)
        if m == 2:
            alt = [max(mg._rows_pairs(S, c), S * (S - 1) // 2 - mg._rows_pairs(S, c)) for c in range(128, S, 128)]
            assert pairs.max() == min(alt)


def test_merge_shards_places_pieces():
    units = _descs([(3, 10), (300, 10), (2, 10)])
    units['site_off'] = [0, 3, 303]
    n_sites = 305

    def recs(rows):
        r = np.zeros(len(rows), dtype=lg_mod.PAIR_REC)
        for k, (u, i, j, mi) in enumerate(rows):
            r[k] = (u, i, j, mi)
        return r

    ordinary = (np.array([0, 2]), recs([(0, 0, 1, 0.5), (0, 1, 2, 0.25), (1, 0, 1, 0.125)]),
                np.array([1.0, 2.0, 3.0, 4.0, 5.0]), np.array([1, 2, 3, 4, 5], dtype=np.uint32),
                np.array([0, 2, 3], dtype=np.uint64), np.arange(27, dtype=np.uint32).reshape(3, 9))
    # unit 1 in two pieces: rows [0, 128) (i, j as in the unit) and [128, 300) (i, j counted from 128)
    p0 = recs([(7, 0, 5, 0.75), (7, 127, 299, 0.0625)])
    p1 = recs([(3, 0, 1, 0.375), (3, 2, 171, 0.1875)])
    c0 = np.full((2, 9), 100, dtype=np.uint32)
    c1 = np.full((2, 9), 200, dtype=np.uint32)
    mean = np.linspace(0.0, 1.0, 300)
    cnt = np.arange(300, dtype=np.uint32)
    got = mg.merge_shards(units, n_sites, [ordinary], [(1, [(0, p0, c0), (128, p1, c1)], mean, cnt)])
    assert got.unit_rec_off.tolist() == [0, 2, 6, 7]
    assert got.records['unit'].tolist() == [0, 0, 1, 1, 1, 1, 2]
    assert got.records['i'].tolist() == [0, 1, 0, 127, 128, 130, 0]
    assert got.records['j'].tolist() == [1, 2, 5, 299, 129, 299, 1]
    assert got.records['mi'].tolist() == [0.5, 0.25, 0.75, 0.0625, 0.375, 0.1875, 0.125]
    assert got.counts[2:6, 0].tolist() == [100, 100, 200, 200] and got.counts[6, 0] == 18
    assert np.array_equal(got.site_mean[3:303], mean) and np.array_equal(got.site_cnt[3:303], cnt)
    assert got.site_mean[:3].tolist() == [1.0, 2.0, 3.0] and got.site_mean[303:].tolist() == [4.0, 5.0]


def test_place_pieces_given_in_any_order():
    """Two split units, their pieces from three devices handed over out of row order (place_pieces, then
    merge_shards): the whole units' records, tables and means, and split_units in row order."""
    units = _descs([(20, 10), (300, 10), (5, 10), (400, 10)])
    units['site_off'] = np.concatenate(([0], np.cumsum(units['n_sites'])[:-1]))
    rng = np.random.default_rng(77)
    whole = []                      # per unit: records, tables, site means, site counts
    for u, S in enumerate(units['n_sites'].tolist()):
        i, j = np.triu_indices(S, 1)
        keep = rng.random(len(i)) < 0.2
        rec = np.zeros(int(keep.sum()), dtype=lg_mod.PAIR_REC)
        rec['unit'], rec['i'], rec['j'], rec['mi'] = u, i[keep], j[keep], rng.random(int(keep.sum()))
        whole.append((rec, rng.integers(0, 1000, size=(len(rec), 9)).astype(np.uint32),
                       np.where(rng.random(S) < 0.2, np.nan, rng.random(S)), rng.integers(0, 50, S).astype(np.uint32)))
    device = {(1, 0): 2, (1, 128): 0, (1, 256): 1, (3, 0): 1, (3, 128): 2}
    pieces = []
    for u, a, e in ((1, 0, 128), (1, 128, 256), (1, 256, 300), (3, 0, 128), (3, 128, 400)):
        rec, tab = whole[u][0], whole[u][1]
        sel = (rec['i'] >= a) & (rec['i'] < e)
        r = rec[sel].copy()
        r['unit'], r['i'], r['j'] = 9, r['i'] - a, r['j'] - a     # numbered as in the piece's batch
        pieces.append((device[(u, a)], u, a, e, r, tab[sel]))
    shard = (np.array([0, 2]), np.concatenate([whole[0][0], whole[2][0]]),
             np.concatenate([whole[0][2], whole[2][2]]), np.concatenate([whole[0][3], whole[2][3]]),
             np.array([0, len(whole[0][0]), len(whole[0][0]) + len(whole[2][0])], dtype=np.uint64),
             np.concatenate([whole[0][1], whole[2][1]]))
    shard[1]['unit'][len(whole[0][0]):] = 1                   # a shard numbers its units from 0
    got = mg.merge_shards(units, int(units['n_sites'].sum()), [shard],
                          *mg.place_pieces([pieces[t] for t in (4, 1, 3, 0, 2)], {1: whole[1][2:], 3: whole[3][2:]}))
    assert np.array_equal(got.records, np.concatenate([w[0] for w in whole]))
    assert np.array_equal(got.counts, np.concatenate([w[1] for w in whole]))
    assert np.array_equal(got.site_mean, np.concatenate([w[2] for w in whole]), equal_nan=True)
    assert np.array_equal(got.site_cnt, np.concatenate([w[3] for w in whole]))
    assert got.unit_rec_off.tolist() == np.cumsum([0] + [len(w[0]) for w in whole]).tolist()
    assert got.split_units == {1: [(2, 0, 128), (0, 128, 256), (1, 256, 300)], 3: [(1, 0, 128), (2, 128, 400)]}


class _Words:
    """pb.planes of a plane batch whose word at position p is p, without holding them."""

    def __getitem__(self, s):
        return np.arange(s.start, s.stop, dtype=np.int64)


class _HostPieces:
    """A device's batch of pieces as numpy words: what upload_piece_rows and the copies write, and how often."""

    def __init__(self, units, pieces):
        self.pb = types.SimpleNamespace(units=mg.piece_units(units, pieces))
        n = int((3 * self.pb.units['n_sites'].astype(np.int64) * self.pb.units['row_words']).sum())
        self.words, self.writes, self.uploaded = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, bool)

    def upload_rows(self, word_begin, words):
        self.words[word_begin:word_begin + len(words)] = words
        self.writes[word_begin:word_begin + len(words)] += 1
        self.uploaded[word_begin:word_begin + len(words)] = True


def _with_planes(units):
    words = 3 * units['n_sites'].astype(np.int64) * units['row_words']
    units['plane_off'] = np.concatenate(([0], np.cumsum(words)[:-1]))
    return units


def _plans():
    """(units, pieces) of the cfg4 + cfg3 plan at 2, 4 and 8 devices, of two split units, and of two pieces of one
    unit on one device."""
    cfg = np.concatenate([_cfg4_descs(), _descs([(2000, 100000)])])
    plans = [mg.plan_pieces(cfg, n)[1] for n in (2, 4, 8)]
    cfg['row_words'] = 3               # (after planning: keeps the stand-in planes of the 2 000-site unit small)
    hand = _with_planes(_descs([(300, 500), (40, 100), (520, 1000)]))
    return [(_with_planes(cfg), p) for p in plans] + [
        (hand, [[(2, 256, 520), (0, 0, 128)], [(2, 0, 256)], [(0, 128, 300)]]),
        (hand, [[(0, 0, 128), (0, 256, 300)], [(0, 128, 256)]])]


def test_plane_copies_assemble_every_piece():
    """Each device's own rows (upload_piece_rows), then plane_copies in order: every piece holds its unit's suffix
    planes [3aW, 3SW), every word written once, and a copy reads only rows its source uploaded itself."""
    for units, pieces in _plans():
        pb = types.SimpleNamespace(units=units, planes=_Words())
        host = [_HostPieces(units, mine) for mine in pieces]
        for b, mine in zip(host, pieces):
            mg.upload_piece_rows(b, pb, mine)
        for b, copies in zip(host, mg.plane_copies(units, pieces)):
            for dst, ks, _qs, src, n in copies:
                assert host[ks].uploaded[src:src + n].all()
                b.words[dst:dst + n] = host[ks].words[src:src + n]
                b.writes[dst:dst + n] += 1
        off, S, W = units['plane_off'].astype(np.int64), units['n_sites'], units['row_words']
        for b, mine in zip(host, pieces):
            want = [np.arange(off[u] + 3 * a * W[u], off[u] + 3 * S[u] * W[u]) for u, a, _e in mine]
            assert np.array_equal(b.words, np.concatenate(want) if want else np.zeros(0, np.int64))
            assert (b.writes == 1).all()
        for u in {u for mine in pieces for u, _a, _e in mine}:
            order = mg.row_order(pieces, u)
            assert [a for a, _e, _k, _q in order] == [0] + [e for _a, e, _k, _q in order[:-1]]
            assert order[-1][1] == units['n_sites'][u] and all(pieces[k][q] == (u, a, e) for a, e, k, q in order)


def test_plane_copies_read_what_the_export_reports():
    """src_word is the source piece's plane_off in its device's batch and n_words its own rows' words: the
    plane_word and plane_words of lgmi_piece_export, which the copies between processes use."""
    for units, pieces in _plans():
        for copies in mg.plane_copies(units, pieces):
            for _dst, ks, qs, src, n in copies:
                u, a, e = pieces[ks][qs]
                assert src == mg.piece_units(units, pieces[ks])['plane_off'][qs]
                assert n == 3 * int(units['row_words'][u]) * (e - a)


# --------------------------------------------------------------------------- on the device
def _unit(rng, S, R, cov, third=0.0):
    a, k = synth.draw_alleles(rng, 1, S, R, cov)
    al = a[0]
    if third:
        al[(rng.random(al.shape) < third) & (al != synth.NOCOV)] = synth.THIRD
    return enc.EncodedUnit(list(range(S)), [("mismatch", "snp", "het_snp")[int(x)] for x in k[0]],
                           synth.labels_from_alleles(al))


MODES = [api.MODE_HET_ONLY | api.MODE_SKIP_NONHET, api.MODE_HET_ONLY, api.MODE_ALL_PAIRS | api.MODE_EMIT_COUNTS]


BOUNDS = ([0, 128, 512, None], [0, 256, None], [0, None])


def _all_bounds(S):
    return [[S if x is None else x for x in b] for b in BOUNDS]


@pytest.mark.gpu
@pytest.mark.parametrize("blocks", [4, 9])
def test_deep_unit_piece_by_piece_equals_whole(lg, gpu_ctx, blocks):
    """Tensor-core path, both forms; the last piece of [0, 128, 512, 550) has 38 sites and takes the mid-depth path."""
    rng = np.random.default_rng(401)
    pb = lg.pack_units([_unit(rng, 550, 9000, 0.6)])
    gpu_ctx.set_dense_path(blocks)
    try:
        for mode in MODES:
            for bounds in _all_bounds(550):
                whole = _check_split(lg, gpu_ctx, pb, bounds, mode)
                assert whole.n_dense_units == 1 and whole.n_dense_four == (1 if blocks == 4 else 0)
    finally:
        gpu_ctx.set_dense_path(4)


@pytest.mark.gpu
def test_deep_unit_falling_back_to_nine_blocks_piece_by_piece(lg, gpu_ctx):
    rng = np.random.default_rng(402)
    pb = lg.pack_units([_unit(rng, 600, 9000, 0.7, third=0.4)])
    for mode in MODES:
        for bounds in _all_bounds(600):
            whole = _check_split(lg, gpu_ctx, pb, bounds, mode)
            assert whole.n_dense_units == 1 and whole.n_dense_four == 0


@pytest.mark.gpu
@pytest.mark.parametrize("tile_path", [2, 0])
def test_mid_depth_unit_piece_by_piece_equals_whole(lg, gpu_ctx, tile_path):
    rng = np.random.default_rng(403)
    pb = lg.pack_units([_unit(rng, 540, 2000, 0.5)])
    gpu_ctx.set_tile_path(tile_path)
    try:
        for mode in MODES:
            for bounds in _all_bounds(540):
                assert _check_split(lg, gpu_ctx, pb, bounds, mode).n_dense_units == 0
    finally:
        gpu_ctx.set_tile_path(2)


@pytest.mark.gpu
def test_mixed_batch_leaves_ordinary_units_as_they_were(lg, gpu_ctx):
    rng = np.random.default_rng(404)
    eus = [_unit(rng, 40, 150, 0.5), _unit(rng, 550, 9000, 0.6), _unit(rng, 200, 1500, 0.5), _unit(rng, 60, 9000, 0.5)]
    pb = lg.pack_units(eus)
    sub, lim = _pieces(pb, [0, 128, 550], unit=1)
    mixed = enc.PlaneBatch(np.concatenate([pb.units, sub.units]), pb.planes, pb.site_flags)
    limits = [0] * pb.n_units + lim
    mode = api.MODE_ALL_PAIRS | api.MODE_EMIT_COUNTS
    want = lg.mi_step_batched(pb, 6, mode, ctx=gpu_ctx, n_chunks=1)
    b = lg.Batch(gpu_ctx, mixed, row_limit=limits)
    try:
        b.upload()
        b.run(6, mode)
        got = b.download()
    finally:
        b.close()
    for u in range(pb.n_units):
        assert np.array_equal(got.unit_records(u), want.unit_records(u))
        assert np.array_equal(got.unit_counts(u), want.unit_counts(u))
    assert np.array_equal(got.site_mean, want.site_mean, equal_nan=True)
    assert np.array_equal(got.site_cnt, want.site_cnt)
    assert got.n_candidates == want.n_candidates + 128 * 550 - 128 * 129 // 2 + 422 * 421 // 2
    rec = np.concatenate([got.unit_records(pb.n_units), got.unit_records(pb.n_units + 1)])
    assert len(rec) == len(want.unit_records(1))


@pytest.mark.gpu
def test_planes_assembled_from_row_ranges_and_copies(lg, gpu_ctx):
    """Piece 0 uploads its own 256 rows from the host and copies the rest from piece 1's batch on another context;
    the results equal those of a piece uploaded whole, and split_means gathers over the two contexts."""
    rng = np.random.default_rng(405)
    pb = lg.pack_units([_unit(rng, 550, 9000, 0.6)])
    W = int(pb.units['row_words'][0])
    mode = api.MODE_HET_ONLY
    whole = lg.mi_step_batched(pb, 6, mode, ctx=gpu_ctx, n_chunks=1)
    other = lg.Context(0)
    p0, l0 = _pieces(pb, [0, 256, 550])
    b0 = lg.Batch(gpu_ctx, enc.PlaneBatch(p0.units[:1].copy(), pb.planes, pb.site_flags), row_limit=l0[:1])
    d1 = p0.units[1:].copy()
    d1['plane_off'] = 0
    d1['site_off'] = 0
    b1 = lg.Batch(other, enc.PlaneBatch(d1, pb.planes[3 * 256 * W:], pb.site_flags[256:]), row_limit=l0[1:])
    ref = lg.Batch(gpu_ctx, enc.PlaneBatch(p0.units[:1].copy(), pb.planes, pb.site_flags), row_limit=l0[:1])
    try:
        b0.upload_rows(0, pb.planes[:3 * 256 * W])
        b1.upload_rows(0, pb.planes[3 * 256 * W:])
        b0.copy_planes_from(3 * 256 * W, b1, 0, 3 * 294 * W)
        ref.upload()
        for b in (b0, b1, ref):
            b.run(6, mode)
        got0, want0 = b0.download(), ref.download()
        assert np.array_equal(got0.records, want0.records) and got0.n_records > 0
        got1 = b1.download()
        mean, cnt = lg.split_means(other, pb.site_flags, [(b0, 0), (b1, 0)])
        rec = np.concatenate([got0.records, got1.records.copy()])
        rec['i'][len(got0.records):] += 256
        rec['j'][len(got0.records):] += 256
        assert np.array_equal(rec, whole.records)
        assert np.array_equal(mean, whole.site_mean, equal_nan=True) and np.array_equal(cnt, whole.site_cnt)
    finally:
        for b in (b0, b1, ref):
            b.close()
        other.close()


@pytest.mark.gpu
def test_argument_errors(lg, gpu_ctx):
    rng = np.random.default_rng(406)
    pb = lg.pack_units([_unit(rng, 300, 500, 0.6)])
    for limit in (100, 301):                       # neither a multiple of 128 nor S; above S
        with pytest.raises(lg.LgmiError) as e:
            lg.Batch(gpu_ctx, pb, row_limit=[limit])
        assert e.value.code == -2
    sub, lim = _pieces(pb, [0, 128, 256, 300])
    b = lg.Batch(gpu_ctx, sub, row_limit=lim)
    try:
        b.upload()
        with pytest.raises(lg.LgmiError) as e:    # not run yet
            lg.split_means(gpu_ctx, pb.site_flags, [(b, 0), (b, 1), (b, 2)])
        assert e.value.code == -4
        b.run(6, api.MODE_HET_ONLY)
        b.sync()
        with pytest.raises(lg.LgmiError) as e:    # a piece missing
            lg.split_means(gpu_ctx, pb.site_flags, [(b, 0), (b, 2)])
        assert e.value.code == -2
        with pytest.raises(lg.LgmiError) as e:    # the whole unit is not covered
            lg.split_means(gpu_ctx, pb.site_flags, [(b, 0), (b, 1)])
        assert e.value.code == -2
        mean, _cnt = lg.split_means(gpu_ctx, pb.site_flags, [(b, 0), (b, 1), (b, 2)])
        assert mean.shape == (300,)
    finally:
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("deep", [(1000, 20000), (2000, 100000)])
def test_device_pool_splits_a_deep_unit(lg, gpu_ctx, deep):
    n = lg.device_count()
    devices = list(range(n)) if n >= 2 else [0, 0]
    S, R = deep
    if deep == (2000, 100000):
        pb, _ = synth.make_deep_unit(20261021, S, R, 0.6)            # cfg3 alone
    else:
        unit, _ = synth.make_deep_unit(20261041, S, R, 0.6)
        tail, _ = synth.make_heavy_tail(20261042, 300)
        pb = enc.concat_plane_batches([tail, unit])
    pool = lg.DevicePool(devices)
    try:
        for mode in (lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET, lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS):
            want = lg.mi_step_batched(pb, 6, mode, ctx=gpu_ctx)
            got = pool.run(pb, 6, mode)
            deep_unit = pb.n_units - 1
            assert list(got.split_units) == [deep_unit] and len(got.split_units[deep_unit]) >= 2
            assert sum(got.shard_units) == pb.n_units
            assert np.array_equal(got.records, want.records)
            assert np.array_equal(got.site_mean, want.site_mean, equal_nan=True)
            assert np.array_equal(got.site_cnt, want.site_cnt)
            assert np.array_equal(got.unit_rec_off, want.unit_rec_off)
            if mode & lg.MODE_EMIT_COUNTS:
                assert np.array_equal(got.counts, want.counts)
    finally:
        pool.close()
