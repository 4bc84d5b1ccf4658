#!/usr/bin/env python
"""Small run through every kernel path (small popcount, tiled, deep tensor, generic fallback,
pipeline, ecdf) for compute-sanitizer memcheck.  No timing, no assertions beyond agreement of
the paths."""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
lg = importlib.import_module("l-giremi_b200")
synth = importlib.import_module("l-giremi_b200.synth")
enc = importlib.import_module("l-giremi_b200.encode")

rng = np.random.default_rng(3)


def unit(S, R, cov=0.6):
    a, k = synth.draw_alleles(rng, 1, S, R, cov)
    return enc.EncodedUnit(list(range(S)), [("mismatch", "snp", "het_snp")[int(x)] for x in k[0]],
                           synth.labels_from_alleles(a[0]))


ctx = lg.Context(0)
eus = [unit(S, R) for S, R in [(2, 6), (7, 33), (50, 200), (60, 256), (64, 256), (65, 40), (70, 300), (33, 1000),
                               (130, 17), (20, 2100)]]
eus.append(enc.EncodedUnit([], [], np.zeros((0, 0), np.uint8)))
eus.append(enc.EncodedUnit([5], ['het_snp'], np.full((1, 9), 2, np.uint8)))
lab = rng.choice(np.array([0, 1, 2, 255], np.uint8), size=(12, 150), p=[0.3, 0.3, 0.3, 0.1])
eus.append(enc.EncodedUnit(list(range(12)), ['het_snp', 'mismatch'] * 6, lab))
pb = lg.pack_units(eus)
mode = lg.MODE_ALL_PAIRS | lg.MODE_EMIT_COUNTS
out = lg.mi_step_batched(pb, 6, mode, ctx=ctx, n_chunks=1)
for m in (lg.MODE_HET_ONLY, lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET):
    lg.mi_step_batched(pb, 3, m, ctx=ctx, n_chunks=1)
ctx.set_dense_threshold(2, 1)                     # everything with a pair through k_dense_x + k_gram_i8
d = lg.mi_step_batched(pb, 6, mode, ctx=ctx, n_chunks=1)
assert d.n_dense_units >= 10
p = lg.Pipeline(ctx, pb, 3)                       # ... also inside the groups of a pipelined step, packed input
r = p.step(6, mode | lg.MODE_SPLIT_RECORDS, packed=True)
assert r.n_dense_units == d.n_dense_units and np.array_equal(r.records, d.records) and np.array_equal(r.counts, d.counts)
p.close()
ctx.set_dense_threshold(*lg.DENSE_DEFAULT)
assert np.array_equal(d.records, out.records) and np.array_equal(d.counts, out.counts)
for chunks in (2, 5, 40):
    p = lg.Pipeline(ctx, pb, chunks)
    r = p.step(6, mode)
    assert np.array_equal(r.records, out.records)
    p.close()
empty = lg.pack_units([])
assert lg.mi_step_batched(empty, 6, mode, ctx=ctx).n_records == 0
p = lg.Pipeline(ctx, empty, 3)
assert p.step(6, lg.MODE_HET_ONLY).n_records == 0
p.close()
mip, call = lg.mip_and_calls(out.site_mean, pb.site_flags & 3, 0.05, ctx=ctx)
print("sanitize run ok:", out.n_records, "records,", ctx.launch_count, "launches")
