"""Drop-in for the reference's `calculate_site_splice_mi` console script
(giremi/script/calculate_site_splice_mi.py:34-130): same two input tables, same output table
`<prefix>.site_splice_pair` (columns chromosome, site_pos, seq, splice_pos, count, mi), with the
mutual information of every (site allele, splice site) pair computed in ONE GPU submit
(api.site_splice_mutual_info) instead of a Python loop with `a in list` scans per pair (:106-125).

    python -m l-giremi_b200.site_splice -m READ_SITE.tsv -s READ_SPLICE.tsv -o PREFIX   (via importlib / runpy)

The table bookkeeping around the MI (which pairs exist, how many reads cover each) is host work
either way and follows the script's own procedure, including its row order: the splice table is
consumed in chunks of 10 000 rows, each chunk contributes its (chromosome, site_pos, seq,
splice_pos) groups in sorted order, a pair keeps the place of its first appearance."""
from __future__ import annotations

import argparse
import csv
from collections import defaultdict

import numpy as np
import pandas as pd

from . import api

SPLICE_CHUNK_ROWS = 10000          # calculate_site_splice_mi.py:45-48


def parse_args(argv=None):
    parser = argparse.ArgumentParser(
        description='calculate the mutual information of mismatch site and splice site pairs')
    parser.add_argument("-m", "--read_site", type=str,
                        help="read-site file: [read_name, chromosome, pos, seq]")
    parser.add_argument("-s", "--read_splice", type=str,
                        help="corrected read-splice file: [read_name, chromosome, pos, type, corrected_pos, annotation]")
    parser.add_argument("-o", "--output_prefix", type=str, default='out', help="prefix of output file")
    return parser.parse_args(argv)


def pair_rows(rsite, splice_file):
    """Pair rows [(chromosome, site_pos, seq, splice_pos, count)] in the script's order (:40-86)."""
    count_of = {}                                   # insertion order = first appearance, as the script's Counter
    for chunk in pd.read_table(splice_file, header=0, sep='\t', chunksize=SPLICE_CHUNK_ROWS):
        merged = pd.merge(rsite, chunk[['read_name', 'chromosome', 'corrected_pos']], how='inner',
                          on=['read_name', 'chromosome'])
        if not len(merged):
            continue
        groups = merged.groupby(['chromosome', 'pos', 'seq', 'corrected_pos'])['read_name'].count()
        for key, n in zip(groups.index.tolist(), groups.tolist()):
            key = tuple(str(k) for k in key)        # the script joins the key as text and splits it again (:63-85)
            count_of[key] = count_of.get(key, 0) + int(n)
    return [key + (n,) for key, n in count_of.items()]


def read_tables(site_file, splice_file):
    """(pair rows [(chromosome, site_pos, seq, splice_pos, count)] in the script's order,
    sites {label: {allele: [read names]}}, splices {label: [read names]})  -- :40-102."""
    rsite = pd.read_table(site_file, header=0, sep='\t')
    rows = pair_rows(rsite, splice_file)
    sites = defaultdict(lambda: defaultdict(list))
    for chrom, pos, seq, name in zip(rsite['chromosome'].tolist(), rsite['pos'].tolist(), rsite['seq'].tolist(),
                                     rsite['read_name'].tolist()):
        sites['{}:{}'.format(chrom, pos)][seq].append(name)
    splices = defaultdict(list)
    with open(splice_file, 'r') as fh:              # every line, the header included (:97-102)
        for line in fh:
            cols = line.strip().split('\t')
            splices[':'.join([cols[1], cols[4]])].append(cols[0])
    return rows, sites, splices


def read_splice_lines(splice_file) -> pd.DataFrame:
    """Every line of the splice file, the header included, as text: the columns read name (0), chromosome (1) and
    corrected_pos (4) that the script's membership lists are built from (:97-102)."""
    return pd.read_csv(splice_file, sep='\t', header=None, usecols=[0, 1, 4], dtype=str, keep_default_na=False,
                       quoting=csv.QUOTE_NONE)


def _labels(left, right):
    """Codes of the text labels '<left>:<right>' of rows, and the labels, formatted once per distinct pair."""
    lc, lu = pd.factorize(left, use_na_sentinel=False)
    rc, ru = pd.factorize(right, use_na_sentinel=False)
    code, pair = pd.factorize(lc.astype(np.int64) * max(len(ru), 1) + rc)
    lu, ru = list(lu), list(ru)
    return code, ['{}:{}'.format(lu[k // max(len(ru), 1)], ru[k % max(len(ru), 1)]) for k in pair.tolist()]


def site_splice_arrays(rsite: pd.DataFrame, splice_lines: pd.DataFrame, rows) -> api.SiteSpliceArrays:
    """The arrays of lgmi_site_splice_mi straight from the two tables (the sets read_tables' dicts describe, for
    the sites and splice sites the pair rows ask for).  Alleles and splice sites are looked up as the script does:
    by the text of the pair row (:107-116)."""
    code, labels = _labels(rsite['chromosome'], rsite['pos'])
    label_ids = {}
    for k, label in enumerate(labels):              # two sites printing alike are one label, as in the dict
        label_ids.setdefault(label, []).append(k)
    site_labels = list(dict.fromkeys(r[0] + ':' + r[1] for r in rows))
    req = np.full(len(labels), -1, dtype=np.int64)
    for k, label in enumerate(site_labels):
        req[label_ids[label]] = k
    site = req[code]
    order = np.flatnonzero(site >= 0)
    order = order[np.argsort(site[order], kind='stable')]   # by requested site, rows in file order within one
    site = site[order]
    entry_off = np.zeros(len(site_labels) + 1, dtype=np.uint64)
    entry_off[1:] = np.cumsum(np.bincount(site, minlength=len(site_labels)))
    entry_read, read_names = pd.factorize(rsite['read_name'].to_numpy()[order], use_na_sentinel=False)
    seq_code, seq_u = pd.factorize(rsite['seq'].to_numpy()[order], use_na_sentinel=False)
    n_seq = max(len(seq_u), 1)
    combo_code, combo = pd.factorize(site * n_seq + seq_code)
    combo_site = combo // n_seq
    local = np.arange(combo.size) - np.searchsorted(combo_site, combo_site)   # alleles by first appearance
    allele_names = [[] for _ in site_labels]
    allele_of = {}
    for k, s, c in zip(local.tolist(), combo_site.tolist(), (combo % n_seq).tolist()):
        allele_names[s].append(seq_u[c])
        allele_of[(s, str(seq_u[c]))] = k
    scode, slabels = _labels(splice_lines[1], splice_lines[4])
    splice_labels = list(dict.fromkeys(r[0] + ':' + r[3] for r in rows))
    spl_of = {label: k for k, label in enumerate(splice_labels)}
    sid = np.array([spl_of.get(label, -1) for label in slabels], dtype=np.int64)[scode]
    sread = pd.Index(read_names).get_indexer(splice_lines[0].to_numpy())
    keep = (sid >= 0) & (sread >= 0)
    splice_off, splice_id = api.read_splice_csr(sread[keep], sid[keep], len(read_names))
    site_of = {label: k for k, label in enumerate(site_labels)}
    tri_site = [site_of[r[0] + ':' + r[1]] for r in rows]
    tri_allele = [allele_of[(s, r[2])] for s, r in zip(tri_site, rows)]
    tri_splice = [spl_of[r[0] + ':' + r[3]] for r in rows]
    return api.SiteSpliceArrays(entry_off, entry_read, local[combo_code], splice_off, splice_id, tri_site,
                                tri_allele, tri_splice, list(read_names), site_labels, allele_names, splice_labels)


def site_splice_table(site_file, splice_file, ctx=None) -> pd.DataFrame:
    """The script's output table, MI from the GPU."""
    rsite = pd.read_table(site_file, header=0, sep='\t')
    rows = pair_rows(rsite, splice_file)
    out = pd.DataFrame([list(r[:4]) for r in rows], columns=['chromosome', 'site_pos', 'seq', 'splice_pos'])
    out.loc[:, 'count'] = [r[4] for r in rows]
    out.loc[:, 'mi'] = (api.site_splice_mi_arrays(site_splice_arrays(rsite, read_splice_lines(splice_file), rows),
                                                  ctx=ctx) if rows else [])
    return out


def main(argv=None):
    args = parse_args(argv)
    table = site_splice_table(args.read_site, args.read_splice)
    table.to_csv(args.output_prefix + '.site_splice_pair', sep='\t', index=False)


if __name__ == '__main__':
    main()
