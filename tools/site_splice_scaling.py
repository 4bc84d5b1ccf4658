"""Site x splice-site MI at several sizes: the device path (lgmi_site_splice_mi) against the former pseudo-site
construction (every site a unit of pseudo-sites, one per requested allele and splice site, through the all-pairs
step), on the same seeded synthetic tables.

Per size: rows of the two tables, requested pairs, and the candidate pairs the all-pairs step would evaluate;
host time of interning + CSR (site_splice.site_splice_arrays), device time of the call (CUDA events around it on
the launching stream), end-to-end time of site_splice.site_splice_table (the new path) and of read_tables + the
pseudo-site construction + table (the former path, up to --old-max-rows site rows, else "not measured"), and a
sha256 of each output table as CSV text, which must agree.  The pair-row bookkeeping (pair_rows, shared by both
paths) is timed on its own.  The GPU's name and power limit are read in the same run.

    python tools/site_splice_scaling.py [--out-dir profiles] [--old-max-rows 500000]
Writes <out-dir>/site_splice_scaling.json."""
import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import pandas as pd

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

lg = importlib.import_module("l-giremi_b200")
api = importlib.import_module("l-giremi_b200.api")
enc = importlib.import_module("l-giremi_b200.encode")
ss = importlib.import_module("l-giremi_b200.site_splice")

# (sites, entries per site, reads, splice records per read, splice sites)
SIZES = [(100, 500, 20000, 2, 200), (400, 1000, 100000, 4, 400), (2000, 1000, 100000, 2, 400)]


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return [dict(zip(("name", "power_limit"), [x.strip() for x in line.split(",")])) for line in out]


def write_tables(tmp, n_sites, per_site, n_reads, per_read, n_splice, seed):
    rng = np.random.default_rng(seed)
    names = np.array(["read%07d" % k for k in range(n_reads)], dtype=object)
    site = np.repeat(np.arange(n_sites), per_site)
    rows = pd.DataFrame({"read_name": names[rng.integers(0, n_reads, site.size)], "chromosome": "chr1",
                         "pos": 10000 + 50 * site,
                         "seq": np.array(list("ACGT"))[rng.choice(4, site.size, p=[0.55, 0.3, 0.1, 0.05])]})
    sf, pf = os.path.join(tmp, "site.tsv"), os.path.join(tmp, "splice.tsv")
    rows.to_csv(sf, sep="\t", index=False)
    r = np.repeat(np.arange(n_reads), per_read)
    spl = pd.DataFrame({"read_name": names[r], "chromosome": "chr1", "pos": 0, "type": "intron",
                        "corrected_pos": 500000 + 100 * rng.integers(0, n_splice, r.size), "annotation": "known"})
    spl.to_csv(pf, sep="\t", index=False)
    return sf, pf, len(rows), len(spl)


def pseudo_site_mutual_info(sites, splices, pairs, ctx):
    """The former api.site_splice_mutual_info: per site a unit whose pseudo-sites are the requested alleles and
    splice sites over every list entry, labels 2 ("with") / 1, all pairs evaluated."""
    by_site = {}
    for k, (site_label, seq, splice_label) in enumerate(pairs):
        by_site.setdefault(site_label, []).append((k, seq, splice_label))
    units, lookup, candidates = [], [], 0
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
        candidates += len(members) * (len(members) - 1) // 2
    out = [0.0] * len(pairs)
    res = api.mi_step_batched(enc.pack_units(units), 0, api.MODE_ALL_PAIRS, ctx=ctx)
    for u, want in enumerate(lookup):
        rec = res.unit_records(u)
        S = units[u].n_sites
        for k, i, j in want:
            out[k] = float(rec['mi'][i * (2 * S - i - 1) // 2 + (j - i - 1)])
    return out, candidates


def old_table(sf, pf, ctx):
    rows, sites, splices = ss.read_tables(sf, pf)
    by_text = {label: {str(seq): seq for seq in alleles} for label, alleles in sites.items()}
    triples = [(c + ':' + p, by_text[c + ':' + p][seq], c + ':' + sp) for c, p, seq, sp, _n in rows]
    mi, candidates = pseudo_site_mutual_info(sites, splices, triples, ctx)
    out = pd.DataFrame([list(r[:4]) for r in rows], columns=['chromosome', 'site_pos', 'seq', 'splice_pos'])
    out.loc[:, 'count'] = [r[4] for r in rows]
    out.loc[:, 'mi'] = mi
    return out, candidates


def table_hash(df):
    return hashlib.sha256(df.to_csv(sep="\t", index=False).encode()).hexdigest()


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", default="profiles")
    ap.add_argument("--old-max-rows", type=int, default=500000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    ctx = lg.get_context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    results = []
    for k, (n_sites, per_site, n_reads, per_read, n_splice) in enumerate(SIZES):
        with tempfile.TemporaryDirectory() as tmp:
            sf, pf, n_site_rows, n_splice_rows = write_tables(tmp, n_sites, per_site, n_reads, per_read, n_splice, k)
            rsite = pd.read_table(sf, header=0, sep="\t")
            t0 = time.perf_counter()
            rows = ss.pair_rows(rsite, pf)
            t_rows = time.perf_counter() - t0
            lines = ss.read_splice_lines(pf)
            t0 = time.perf_counter()
            arrays = ss.site_splice_arrays(rsite, lines, rows)
            t_host = time.perf_counter() - t0
            api.site_splice_mi_arrays(arrays, ctx=ctx)                 # warm-up: ln table, pool blocks
            dev = []
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                api.site_splice_mi_arrays(arrays, ctx=ctx)
                e1.record(stream)
                e1.synchronize()
                dev.append(e0.elapsed_time(e1))
            t0 = time.perf_counter()
            new = ss.site_splice_table(sf, pf, ctx=ctx)
            t_new = time.perf_counter() - t0
            rec = {"sites": n_sites, "entries_per_site": per_site, "reads": n_reads, "site_rows": n_site_rows,
                   "splice_rows": n_splice_rows, "pairs_requested": len(rows),
                   "pair_rows_s": round(t_rows, 3), "host_intern_csr_s": round(t_host, 3),
                   "device_ms": [round(x, 3) for x in dev], "device_ms_median": round(float(np.median(dev)), 3),
                   "new_end_to_end_s": round(t_new, 3), "new_table_sha256": table_hash(new)}
            if n_site_rows <= args.old_max_rows:
                t0 = time.perf_counter()
                old, candidates = old_table(sf, pf, ctx)
                rec["old_end_to_end_s"] = round(time.perf_counter() - t0, 3)
                rec["old_candidate_pairs"] = candidates
                rec["old_table_sha256"] = table_hash(old)
                rec["tables_identical"] = rec["old_table_sha256"] == rec["new_table_sha256"]
            else:
                rec["old_end_to_end_s"] = "not measured"
            print(json.dumps(rec), flush=True)
            results.append(rec)
    ctx.set_stream(0)
    out = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0), "sizes": results}
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "site_splice_scaling.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
