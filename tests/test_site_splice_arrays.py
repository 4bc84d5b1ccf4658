"""The integer arrays of the site x splice-site MI (api.SiteSpliceArrays) describe the same sets as the reference's
dicts (calculate_site_splice_mi.py:88-102): built from the two tables (site_splice.site_splice_arrays) and from the
dicts (api.site_splice_arrays).  No device needed."""
import importlib
from collections import Counter

import numpy as np
import pandas as pd

from test_site_splice import golden_tables, random_case

api = importlib.import_module("l-giremi_b200.api")
ss = importlib.import_module("l-giremi_b200.site_splice")


def decoded(a):
    """({site label: Counter of (read name, allele text)}, {splice label: set of read names}) from the arrays."""
    sites = {}
    for k, label in enumerate(a.site_labels):
        lo, hi = int(a.entry_off[k]), int(a.entry_off[k + 1])
        sites[label] = Counter((a.read_names[r], str(a.allele_names[k][al]))
                               for r, al in zip(a.entry_read[lo:hi].tolist(), a.entry_allele[lo:hi].tolist()))
    splices = {label: set() for label in a.splice_labels}
    for r in range(a.n_reads):
        ids = a.splice_id[int(a.splice_off[r]):int(a.splice_off[r + 1])]
        assert np.all(np.diff(ids.astype(np.int64)) > 0)          # ascending, each once
        for i in ids.tolist():
            splices[a.splice_labels[i]].add(a.read_names[r])
    return sites, splices


def check_against_dicts(a, sites, splices, pairs):
    got_sites, got_splices = decoded(a)
    assert a.site_labels == list(dict.fromkeys(p[0] for p in pairs))
    for label in a.site_labels:
        assert got_sites[label] == Counter((name, str(seq)) for seq, names in sites[label].items() for name in names)
    reads = set(a.read_names)
    assert set(a.splice_labels) == {p[2] for p in pairs}
    for label in a.splice_labels:
        assert got_splices[label] == set(splices.get(label, ())) & reads
    for t, (site_label, seq, splice_label) in enumerate(pairs):
        k = int(a.tri_site[t])
        assert a.site_labels[k] == site_label
        assert str(a.allele_names[k][a.tri_allele[t]]) == str(seq)
        assert a.splice_labels[a.tri_splice[t]] == splice_label


def tables_arrays(sf, pf):
    rsite = pd.read_table(sf, header=0, sep="\t")
    rows = ss.pair_rows(rsite, pf)
    return rows, ss.site_splice_arrays(rsite, ss.read_splice_lines(pf), rows)


def write_tables(tmp_path, site_rows, splice_rows):
    sf, pf = str(tmp_path / "site.tsv"), str(tmp_path / "splice.tsv")
    pd.DataFrame(site_rows, columns=["read_name", "chromosome", "pos", "seq"]).to_csv(sf, sep="\t", index=False)
    pd.DataFrame(splice_rows, columns=["read_name", "chromosome", "pos", "type", "corrected_pos", "annotation"]
                 ).to_csv(pf, sep="\t", index=False)
    return sf, pf


def test_arrays_from_tables_and_dicts_describe_the_golden_sets(golden, tmp_path):
    _g, sf, pf = golden_tables(golden, tmp_path)
    rows, a = tables_arrays(sf, pf)
    rows_d, sites, splices = ss.read_tables(sf, pf)
    assert rows == rows_d
    pairs = [(r[0] + ":" + r[1], r[2], r[0] + ":" + r[3]) for r in rows]
    check_against_dicts(a, sites, splices, pairs)
    by_text = {label: {str(seq): seq for seq in alleles} for label, alleles in sites.items()}
    dict_pairs = [(s, by_text[s][seq], sp) for s, seq, sp in pairs]
    check_against_dicts(api.site_splice_arrays(sites, splices, dict_pairs), sites, splices, dict_pairs)


def test_arrays_from_dicts_random_cases():
    for seed in range(4):
        sites, splices, pairs = random_case(np.random.default_rng(100 + seed), 20, 8)
        check_against_dicts(api.site_splice_arrays(sites, splices, pairs), sites, splices, pairs)


def test_arrays_from_tables_random_cases(tmp_path):
    """random_case's dicts written out as the two tables, a read listed twice under two alleles among them."""
    for seed in range(3):
        sites, splices, _pairs = random_case(np.random.default_rng(200 + seed), 15, 6)
        site_rows = [(name, "chr1", int(label.split(":")[1]), seq)
                     for label, alleles in sites.items() for seq, names in alleles.items() for name in names]
        splice_rows = [(name, "chr1", 0, "x", int(label.split(":")[1]), "a")
                       for label, names in splices.items() for name in names]
        sf, pf = write_tables(tmp_path, site_rows, splice_rows)
        rows, a = tables_arrays(sf, pf)
        assert rows
        _rows, d_sites, d_splices = ss.read_tables(sf, pf)
        check_against_dicts(a, d_sites, d_splices, [(r[0] + ":" + r[1], r[2], r[0] + ":" + r[3]) for r in rows])


def test_duplicates_and_the_header_line(tmp_path):
    """A read under two alleles and a read twice under one allele stay two entries each; a splice record repeated
    for one read is one membership; the header line of the splice file is a list of its own ('read_name' under
    'chromosome:corrected_pos'), as in the script."""
    site_rows = [("r1", "chr1", 100, "A"), ("r1", "chr1", 100, "G"),       # two alleles
                 ("r2", "chr1", 100, "A"), ("r2", "chr1", 100, "A"),       # twice under one
                 ("r3", "chr1", 100, "G"), ("read_name", "chr1", 100, "A"),
                 ("r4", "chr1", 200, "T")]
    splice_rows = [("r1", "chr1", 0, "x", 500, "a"), ("r1", "chr1", 0, "x", 500, "a"),   # repeated record
                   ("r2", "chr1", 0, "x", 500, "a"), ("r3", "chr1", 0, "x", 600, "a"),
                   ("r4", "chr1", 0, "x", 600, "a")]
    sf, pf = write_tables(tmp_path, site_rows, splice_rows)
    rows, a = tables_arrays(sf, pf)
    _rows, sites, splices = ss.read_tables(sf, pf)
    pairs = [(r[0] + ":" + r[1], r[2], r[0] + ":" + r[3]) for r in rows]
    check_against_dicts(a, sites, splices, pairs)
    got_sites, got_splices = decoded(a)
    assert got_sites["chr1:100"][("r1", "A")] == 1 and got_sites["chr1:100"][("r1", "G")] == 1
    assert got_sites["chr1:100"][("r2", "A")] == 2
    assert got_splices["chr1:500"] == {"r1", "r2"}
    assert int(a.splice_off[-1]) == 4                                    # r1:500, r2:500, r3:600, r4:600
    header = ss.read_splice_lines(pf)
    assert header.iloc[0].tolist() == ["read_name", "chromosome", "corrected_pos"]
    # the header's list, asked for through the dicts
    pairs = [("chr1:100", "A", "chromosome:corrected_pos"), ("chr1:100", "G", "chr1:500")]
    a = api.site_splice_arrays(sites, splices, pairs)
    check_against_dicts(a, sites, splices, pairs)
    assert decoded(a)[1]["chromosome:corrected_pos"] == {"read_name"}


def test_read_splice_csr_sorts_and_deduplicates():
    off, ids = api.read_splice_csr([2, 0, 2, 2, 0], [7, 3, 1, 7, 3], 4)
    assert off.tolist() == [0, 1, 1, 3, 3] and ids.tolist() == [3, 1, 7]
