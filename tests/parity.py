"""Helpers shared by the GPU parity tests: the C oracle on an EncodedUnit, one batch checked against it in every
mode, synthetic units, and the pieces of a split deep unit checked against the whole unit."""
import importlib
import os
import sys

import numpy as np

from conftest import ROOT, assert_mi_close

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import c_oracle  # noqa: E402

api = importlib.import_module("l-giremi_b200.api")
enc = importlib.import_module("l-giremi_b200.encode")
lg_mod = importlib.import_module("l-giremi_b200")
synth = importlib.import_module("l-giremi_b200.synth")


def signed(labels):
    out = labels.astype(np.int16)
    out[out == 255] = -1
    return out.astype(np.int8)


def oracle_unit(eu, min_common):
    """Oracle on an EncodedUnit: (i, j, mi, tables, mean, cnt)."""
    S = eu.n_sites
    if S < 2:
        z = np.zeros(0, np.int32)
        return z, z, np.zeros(0), np.zeros((0, 9), np.int64), np.full(S, np.nan), np.zeros(S, np.int32)
    i, j, mi, tab = c_oracle.unit_pairs_from_labels(signed(eu.labels), None, min_common)
    is_het = np.array([t == 'het_snp' for t in eu.types], dtype=np.uint8)
    mean, cnt = c_oracle.site_means(S, is_het, i, j, mi)
    return i, j, mi, tab, mean, cnt


def check_batch(lg, ctx, eus, min_common, min_exact=0.97):
    """Runs one batch in ALL_PAIRS|EMIT_COUNTS and HET_ONLY modes and checks
    every output against the oracle."""
    pb = lg.pack_units(eus)
    full = lg.mi_step_batched(pb, min_common, lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS, ctx=ctx)
    het = lg.mi_step_batched(pb, min_common, lg.MODE_HET_ONLY, ctx=ctx)
    skip = lg.mi_step_batched(pb, min_common, lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET, ctx=ctx)
    assert full.n_candidates == pb.n_candidates == het.n_candidates
    assert full.unit_rec_off[0] == 0 and full.unit_rec_off[-1] == full.n_records
    got_mi, want_mi, got_mean, want_mean = [], [], [], []
    for u, eu in enumerate(eus):
        i, j, mi, tab, mean, cnt = oracle_unit(eu, min_common)
        rec = full.unit_records(u)
        assert np.all(rec['unit'] == u)
        assert rec['i'].tolist() == i.tolist() and rec['j'].tolist() == j.tolist(), "pair set of unit %d" % u
        assert np.array_equal(full.unit_counts(u).astype(np.int64), tab), "3x3 counts of unit %d" % u
        got_mi.append(rec['mi'])
        want_mi.append(mi)
        is_het = np.array([t == 'het_snp' for t in eu.types], dtype=bool)
        keep = is_het[i] | is_het[j] if len(i) else np.zeros(0, bool)
        for res in (het, skip):
            hrec = res.unit_records(u)
            assert hrec['i'].tolist() == i[keep].tolist() and hrec['j'].tolist() == j[keep].tolist()
            assert np.array_equal(hrec['mi'], rec['mi'][keep])          # same bits in every mode
        off = int(pb.units['site_off'][u])
        for res in (full, het, skip):
            assert res.site_cnt[off:off + eu.n_sites].tolist() == cnt.tolist()
            assert np.array_equal(res.site_mean[off:off + eu.n_sites], full.site_mean[off:off + eu.n_sites],
                                  equal_nan=True)
        got_mean.append(full.site_mean[off:off + eu.n_sites])
        want_mean.append(mean)
    cat = lambda v: np.concatenate(v) if v else np.zeros(0)
    assert_mi_close(cat(got_mi), cat(want_mi), min_exact, "pair MI")
    assert_mi_close(cat(got_mean), cat(want_mean), min_exact, "mean MI")
    return full


def _synth_unit(rng, S, R, cov):
    a, k = synth.draw_alleles(rng, 1, S, R, cov)
    return enc.EncodedUnit([1000 + 37 * s for s in range(S)],
                           [("mismatch", "snp", "het_snp")[int(x)] for x in k[0]], synth.labels_from_alleles(a[0]))


def _other_heavy_unit(rng, S, R, cov, third):
    """Like _synth_unit with a chosen rate of third alleles (label "other")."""
    a, k = synth.draw_alleles(rng, 1, S, R, cov)
    al = a[0]
    extra = (rng.random(al.shape) < third) & (al != synth.NOCOV)
    al[extra] = synth.THIRD
    return enc.EncodedUnit([1000 + 37 * s for s in range(S)],
                           [("mismatch", "snp", "het_snp")[int(x)] for x in k[0]], synth.labels_from_alleles(al))


# --------------------------------------------------------------------------- pieces of a split deep unit
def _pieces(pb, bounds, unit=0):
    """A PlaneBatch whose units are the pieces of pb's unit `unit` (suffix units into the same planes) + row limits."""
    g = pb.units[unit]
    W = int(g['row_words'])
    desc = np.zeros(len(bounds) - 1, dtype=lg_mod.UNIT_DESC)
    for q, a in enumerate(bounds[:-1]):
        desc[q] = (int(g['plane_off']) + 3 * a * W, int(g['n_sites']) - a, int(g['n_reads']), W, int(g['site_off']) + a)
    return enc.PlaneBatch(desc, pb.planes, pb.site_flags), [e - a for a, e in zip(bounds[:-1], bounds[1:])]


def _joined(res, bounds):
    rec = np.concatenate([res.unit_records(q).copy() for q in range(len(bounds) - 1)])
    shift = np.concatenate([np.full(len(res.unit_records(q)), a) for q, a in enumerate(bounds[:-1])])
    rec['i'] += shift.astype(np.uint16)
    rec['j'] += shift.astype(np.uint16)
    rec['unit'] = 0
    return rec


def _check_split(lg, ctx, pb, bounds, mode, mc=6):
    whole = lg.mi_step_batched(pb, mc, mode, ctx=ctx, n_chunks=1)
    sub, lim = _pieces(pb, bounds)
    b = lg.Batch(ctx, sub, row_limit=lim)
    try:
        b.upload()
        b.run(mc, mode)
        got = b.download()
        mean, cnt = lg.split_means(ctx, pb.site_flags, [(b, q) for q in range(len(lim))])
    finally:
        b.close()
    rec = _joined(got, bounds)
    assert np.array_equal(rec.view(np.uint8), whole.records.view(np.uint8))      # bit for bit, MI included
    if mode & api.MODE_EMIT_COUNTS:
        assert np.array_equal(got.counts, whole.counts)
    assert got.n_candidates == whole.n_candidates and got.n_evaluated == whole.n_evaluated
    assert np.isnan(got.site_mean).all() and not got.site_cnt.any()                # a piece's means would be partial
    assert np.array_equal(mean.view(np.uint64), whole.site_mean.view(np.uint64))
    assert np.array_equal(cnt, whole.site_cnt)
    return whole
