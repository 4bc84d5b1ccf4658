"""The site x splice-site MI on the device (lgmi_site_splice_mi) at every edge of its count pass.

Each case checks the integer 2x2 tables exactly against a numpy count over the same arrays, MI against the oracle
(calculate_site_splice_mi.py:106-125 restated) with test_site_splice.py's thresholds, and MI bit for bit against the
former construction: every site a unit of pseudo-sites (one per requested allele, one per requested splice site) run
through the all-pairs step.  Same integers and the same epilogue give the same bits."""
import importlib
import os
import sys

import numpy as np
import pandas as pd
import pytest

from conftest import ROOT, assert_mi_close, unhex
from test_site_splice import golden_tables, random_case

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import oracle  # noqa: E402

api = importlib.import_module("l-giremi_b200.api")
enc = importlib.import_module("l-giremi_b200.encode")
ss = importlib.import_module("l-giremi_b200.site_splice")

FAST_MAX = (1 << 21) - 1          # kFastMathMaxCount: entries up to here take the reorganised epilogue
TILE_COLS = 128                   # kSsTileCols


def numpy_tables(a):
    """[N-x-y+xy, y-xy, x-xy, xy] of every triple, counted on the host from the arrays."""
    owner = np.repeat(np.arange(a.n_reads), np.diff(a.splice_off.astype(np.int64)))
    spliced = {}
    out = np.zeros((a.tri_site.size, 4), np.int64)
    for t in range(a.tri_site.size):
        s, al, sp = int(a.tri_site[t]), int(a.tri_allele[t]), int(a.tri_splice[t])
        if sp not in spliced:
            spliced[sp] = np.zeros(a.n_reads, bool)
            spliced[sp][owner[a.splice_id == sp]] = True
        lo, hi = int(a.entry_off[s]), int(a.entry_off[s + 1])
        reads, alleles = a.entry_read[lo:hi], a.entry_allele[lo:hi]
        with_x = np.isin(reads, reads[alleles == al])
        with_y = spliced[sp][reads]
        x, y, xy = int(with_x.sum()), int(with_y.sum()), int((with_x & with_y).sum())
        out[t] = (hi - lo - x - y + xy, y - xy, x - xy, xy)
    return out


def pseudo_site_mi(sites, splices, pairs, ctx):
    """The former path: per site a unit whose sites are the requested alleles and splice sites, every list entry a
    read, label 2 ("with") or 1; the pair (allele, splice) of the all-pairs step is the triple's table."""
    by_site = {}
    for k, (site_label, seq, splice_label) in enumerate(pairs):
        by_site.setdefault(site_label, []).append((k, seq, splice_label))
    units, lookup = [], []
    for site_label, wanted in by_site.items():
        alleles = sites[site_label]
        entries = sorted(name for allele in alleles for name in alleles[allele])
        seqs = list(dict.fromkeys(seq for _k, seq, _s in wanted))
        spl = list(dict.fromkeys(s for _k, _seq, s in wanted))
        members = [set(alleles[seq]) for seq in seqs] + [set(splices.get(s, ())) for s in spl]
        labels = np.empty((len(members), len(entries)), dtype=np.uint8)
        for row, names in enumerate(members):
            labels[row] = [2 if name in names else 1 for name in entries]
        units.append(enc.EncodedUnit(list(range(len(members))), ['mismatch'] * len(members), labels))
        lookup.append([(k, seqs.index(seq), len(seqs) + spl.index(s)) for k, seq, s in wanted])
    out = np.zeros(len(pairs))
    res = api.mi_step_batched(enc.pack_units(units), 0, api.MODE_ALL_PAIRS, ctx=ctx)
    for u, want in enumerate(lookup):
        rec = res.unit_records(u)
        S = units[u].n_sites
        for k, i, j in want:
            out[k] = rec['mi'][i * (2 * S - i - 1) // 2 + (j - i - 1)]
    return out


def check(sites, splices, pairs, ctx, with_oracle=True):
    a = api.site_splice_arrays(sites, splices, pairs)
    mi, tab = api.site_splice_mi_arrays(a, ctx=ctx, tables=True)
    assert np.array_equal(tab.astype(np.int64), numpy_tables(a))
    if with_oracle:
        assert_mi_close(mi, oracle.site_splice_mutual_info(sites, splices, pairs), 0.9, "site x splice MI")
    old = pseudo_site_mi(sites, splices, pairs, ctx)
    assert np.array_equal(mi.view(np.int64), old.view(np.int64)), "not the former path's bits"
    assert api.site_splice_mutual_info(sites, splices, pairs, ctx=ctx) == mi.tolist()
    return mi, tab


@pytest.mark.gpu
def test_golden_tables_end_to_end(gpu_ctx, golden, tmp_path):
    g, sf, pf = golden_tables(golden, tmp_path)
    prefix = str(tmp_path / "out")
    ss.main(["-m", sf, "-s", pf, "-o", prefix])
    table = pd.read_table(prefix + ".site_splice_pair", dtype={"chromosome": str, "seq": str},
                          float_precision="round_trip")
    want = g["pairs"]
    assert [[str(r.chromosome), int(r.site_pos), str(r.seq), int(r.splice_pos), int(r["count"])]
            for _, r in table.iterrows()] == [p[:5] for p in want]
    assert_mi_close(table["mi"].to_numpy(), [unhex(p[5]) for p in want], 0.9, "site x splice MI")
    rows, sites, splices = ss.read_tables(sf, pf)
    by_text = {label: {str(seq): seq for seq in alleles} for label, alleles in sites.items()}
    pairs = [(r[0] + ":" + r[1], by_text[r[0] + ":" + r[1]][r[2]], r[0] + ":" + r[3]) for r in rows]
    mi, _tab = check(sites, splices, pairs, gpu_ctx)
    assert np.array_equal(table["mi"].to_numpy().view(np.int64), mi.view(np.int64))


@pytest.mark.gpu
def test_random_cases(gpu_ctx):
    for seed in range(3):
        sites, splices, pairs = random_case(np.random.default_rng(300 + seed))
        mi, _tab = check(sites, splices, pairs, gpu_ctx)
        assert mi[-1] == 0.0


@pytest.mark.gpu
def test_duplicates_missing_labels_one_class_and_unspliced_sites(gpu_ctx):
    """A read under two alleles (counts as "with" both), a read twice under one allele (two entries), a splice
    record repeated for one read (one membership), the header line's list, a splice label nobody has, an allele every
    entry carries (one class: 0.0) and a site none of whose reads is spliced."""
    reads = ["r%03d" % k for k in range(120)]
    sites = {
        "chr1:100": {"A": reads[0:40] + reads[0:5], "G": reads[30:60], "read_name": ["read_name"]},
        "chr1:200": {"T": reads[10:50]},                                     # one allele: every entry carries it
        "chr1:300": {"C": reads[60:90], "T": reads[85:100]},                 # nobody spliced
    }
    splices = {"chr1:500": reads[0:20] + reads[0:3] + reads[35:45], "chr1:600": reads[50:58],
               "chromosome:corrected_pos": ["read_name"]}
    pairs = [("chr1:100", "A", "chr1:500"), ("chr1:100", "G", "chr1:500"), ("chr1:100", "G", "chr1:600"),
             ("chr1:100", "read_name", "chromosome:corrected_pos"), ("chr1:100", "A", "chr1:999"),
             ("chr1:200", "T", "chr1:500"), ("chr1:300", "C", "chr1:500"), ("chr1:300", "T", "chr1:600"),
             ("chr1:100", "A", "chr1:500")]
    mi, tab = check(sites, splices, pairs, gpu_ctx)
    assert mi[0] > 0 and mi[0] == mi[8]
    assert tab[0].sum() == 45 + 30 + 1                                       # every list entry of the site
    assert mi[4] == 0.0 and tab[4][1] == tab[4][3] == 0                      # splice label nobody has
    assert mi[5] == 0.0 and tab[5][0] == tab[5][1] == 0                      # one class
    assert mi[6] == mi[7] == 0.0 and tab[6][1] == tab[6][3] == tab[7][1] == tab[7][3] == 0
    assert tab[3].tolist() == [75, 0, 0, 1]


def deep_site(n, seed):
    """One site of n entries (two alleles, a few reads listed twice) and two splice sites."""
    rng = np.random.default_rng(seed)
    n_reads = n - 1000
    names = np.array(["d%07d" % k for k in range(n_reads)], dtype=object)
    pick = np.concatenate([np.arange(n_reads), rng.integers(0, n_reads, 1000)])
    allele = rng.integers(0, 2, n) == 1
    sites = {"chr2:1": {"A": names[pick[~allele]].tolist(), "G": names[pick[allele]].tolist()}}
    hap = rng.integers(0, 2, n_reads) == 1
    splices = {"chr2:50": names[hap].tolist(), "chr2:60": names[rng.integers(0, 4, n_reads) == 0].tolist()}
    pairs = [("chr2:1", "A", "chr2:50"), ("chr2:1", "G", "chr2:50"), ("chr2:1", "A", "chr2:60")]
    return sites, splices, pairs


@pytest.mark.gpu
@pytest.mark.parametrize("n", [FAST_MAX, FAST_MAX + 1])
def test_deep_site_either_side_of_the_fast_epilogue(gpu_ctx, n):
    sites, splices, pairs = deep_site(n, n)
    _mi, tab = check(sites, splices, pairs, gpu_ctx)
    assert (tab.sum(axis=1) == n).all()


@pytest.mark.gpu
def test_64_alleles_at_a_site_and_65(gpu_ctx):
    reads = ["q%04d" % k for k in range(2000)]
    splices = {"chr3:9": reads[::3]}
    sites = {"chr3:1": {"a%02d" % k: reads[30 * k:30 * k + 40] for k in range(64)}}
    pairs = [("chr3:1", "a%02d" % k, "chr3:9") for k in (0, 1, 31, 32, 62, 63)]
    check(sites, splices, pairs, gpu_ctx)
    sites["chr3:1"]["a64"] = reads[1950:2000]
    with pytest.raises(api.LgmiError) as e:
        api.site_splice_mutual_info(sites, splices, pairs, ctx=gpu_ctx)
    assert e.value.code == -6 and "64 distinct alleles" in str(e.value)


@pytest.mark.gpu
def test_more_requested_columns_than_one_tile(gpu_ctx):
    rng = np.random.default_rng(7)
    reads = ["t%05d" % k for k in range(6000)]
    n_cols = 2 * TILE_COLS + 37
    splices = {"chr4:%d" % (1000 + c): rng.choice(reads, int(rng.integers(1, 900)), replace=False).tolist()
               for c in range(n_cols)}
    cover = rng.choice(reads, 5000, replace=False).tolist()
    sites = {"chr4:10": {"A": cover[:3000], "C": cover[2500:], "G": cover[:100]}}
    pairs = [("chr4:10", seq, label) for label in splices for seq in ("A", "C", "G")][::-1]
    a = api.site_splice_arrays(sites, splices, pairs)
    assert len(a.splice_labels) > 2 * TILE_COLS
    check(sites, splices, pairs, gpu_ctx)


def small_sites(n_sites, seed):
    rng = np.random.default_rng(seed)
    reads = ["s%06d" % k for k in range(20000)]
    splices = {"chr5:%d" % (10 ** 7 + s): rng.choice(reads, 300, replace=False).tolist() for s in range(50)}
    labels = list(splices)
    sites, pairs = {}, []
    for k in range(n_sites):
        label = "chr5:%d" % (1000 + 3 * k)
        names = rng.choice(reads, int(rng.integers(1, 9)), replace=False).tolist()
        sites[label] = {"A": names[::2], "T": names[1::2] + names[:1]}
        pairs += [(label, "A", labels[int(rng.integers(0, 50))]), (label, "T", labels[int(rng.integers(0, 50))])]
    return sites, splices, pairs


@pytest.mark.gpu
def test_many_small_sites_in_a_constant_number_of_launches(gpu_ctx):
    launches = []
    for n_sites in (10, 100000):
        sites, splices, pairs = small_sites(n_sites, n_sites)
        a = api.site_splice_arrays(sites, splices, pairs)
        before = gpu_ctx.launch_count
        mi, tab = api.site_splice_mi_arrays(a, ctx=gpu_ctx, tables=True)
        launches.append(gpu_ctx.launch_count - before)
    assert launches[0] == launches[1] <= 4
    assert np.array_equal(tab.astype(np.int64), numpy_tables(a))
    assert_mi_close(mi, oracle.site_splice_mutual_info(sites, splices, pairs), 0.9, "site x splice MI")
    assert np.array_equal(mi.view(np.int64), pseudo_site_mi(sites, splices, pairs, gpu_ctx).view(np.int64))


@pytest.mark.gpu
def test_argument_errors(gpu_ctx):
    lib, h = gpu_ctx._lib, gpu_ctx.handle
    P = api.ptr

    def call(entry_off=(0, 2, 3), read=(0, 1, 1), allele=(0, 1, 0), splice_off=(0, 1, 3), splice_id=(4, 4, 2),
             tri=((0, 0, 4), (1, 0, 2)), out=True, n_reads=2):
        a = [np.ascontiguousarray(v, dtype=np.uint64 if k in (0, 3) else np.uint32)
             for k, v in enumerate((entry_off, read, allele, splice_off, splice_id))]
        t = np.ascontiguousarray(tri, dtype=np.uint32).reshape(-1, 3).T.copy()
        mi = np.empty(t.shape[1]) if out else None
        return lib.lgmi_site_splice_mi(h, a[0].size - 1, P(a[0]), P(a[1]), P(a[2]), n_reads, P(a[3]), P(a[4]),
                                       t.shape[1], P(t[0]), P(t[1]), P(t[2]), P(mi), None), mi

    assert call(splice_id=(4, 2, 5))[0] == 0
    assert call()[0] == -2                                   # read 1's splice ids not ascending and unique
    ok = dict(splice_id=(4, 2, 5))
    assert call(entry_off=(1, 2, 3), **ok)[0] == -2          # offsets do not start at 0
    assert call(entry_off=(0, 3, 2), **ok)[0] == -2          # decreasing
    assert call(read=(0, 2, 1), **ok)[0] == -2               # read id out of range
    assert call(tri=((2, 0, 4),), **ok)[0] == -2             # site out of range
    assert call(out=False, **ok)[0] == -2                    # NULL output
    assert call(allele=(0, 64, 0), **ok)[0] == -6            # 65th allele
    assert "lgmi_site_splice_mi" in lib.lgmi_last_error(h).decode()
    rc, mi = call(tri=(), **ok)
    assert rc == 0 and mi.size == 0
