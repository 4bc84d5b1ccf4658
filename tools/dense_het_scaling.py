"""The deep-unit step in HET_ONLY against HET_ONLY | SKIP_NONHET (the het-anchored form) as the share of het sites grows.

The cfg3 unit (2 000 sites x 100 000 reads, the bench's seed) with its flag bytes rewritten so that 1, 5, 10, 25 and
50 % of the sites are het SNPs (seeded choice; the planes are unchanged).  For each share and mode: the step on
device events (kernel_ms), dense_kernel_ms and gram_kernel_ms, best and median of --reps timed runs after warm-up
(the two modes alternate), the issued multiply-accumulates, per-kernel times of the tensor-core path from one
torch.profiler pass of its own, and the sha256 of the rows and means of both modes, which must be equal.  The card's
name and power limit are read in the same run.

    python tools/dense_het_scaling.py --out profiles/r4_dense_het_n1.json
"""
import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
lg = importlib.import_module("l-giremi_b200")
synth = importlib.import_module("l-giremi_b200.synth")

CFG3 = dict(sites=2000, reads=100000, cov=0.6, min_common=6, seed=20261021)
SHARES = (0.01, 0.05, 0.10, 0.25, 0.50)
TYPE_MASK, SNP, HET_SNP = 3, 1, 2
DENSE_KERNELS = ("k_dense_prep", "k_other_fix", "k_dense_x", "k_zero_partial_tiles", "k_gram_i8")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in q.split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def with_het_share(pb, share, seed):
    S = int(pb.units["n_sites"][0])
    rng = np.random.default_rng(seed)
    het = np.sort(rng.choice(S, max(1, int(round(share * S))), replace=False))
    flags = (pb.site_flags & ~np.uint8(TYPE_MASK)) | np.uint8(SNP)
    flags[het] = (flags[het] & ~np.uint8(TYPE_MASK)) | np.uint8(HET_SNP)
    return flags, len(het)


def digest(res):
    h = hashlib.sha256()
    h.update(res.records.tobytes())
    h.update(res.site_mean.tobytes())
    h.update(res.site_cnt.tobytes())
    return h.hexdigest()


def stats(v):
    return dict(best=float(np.min(v)), median=float(np.median(v)))


def kernel_times(b, mc, mode, runs=3):
    """Mean device time per kernel of the tensor-core path over `runs` runs, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(runs):
            b.run(mc, mode)
            b.sync()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for k in DENSE_KERNELS:
            if k in ev.key:
                out[k] = out.get(k, 0.0) + ev.device_time_total / 1e3 / runs  # (us -> ms)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-profile", action="store_true")
    a = ap.parse_args()
    ctx = lg.get_context()
    pb, _ = synth.make_deep_unit(CFG3["seed"], CFG3["sites"], CFG3["reads"], CFG3["cov"])
    mc = CFG3["min_common"]
    modes = {"het_only": lg.MODE_HET_ONLY, "skip_nonhet": lg.MODE_HET_ONLY | lg.MODE_SKIP_NONHET}
    out = dict(tool="tools/dense_het_scaling.py", card=card(),
               workload="cfg3: 1 unit x %d sites x %d reads, cov %g, min_common %d, seed %d; flag bytes rewritten"
                        % (CFG3["sites"], CFG3["reads"], CFG3["cov"], mc, CFG3["seed"]),
               timing="device events of one non-graph run (kernel_ms: whole step; dense_kernel_ms: tensor-core path; "
                      "gram_kernel_ms: k_gram_i8 alone), best and median of %d runs after %d warm-up runs per mode, "
                      "modes alternating; kernels: torch.profiler, mean of 3 runs in a pass of its own"
                      % (a.reps, a.warmup),
               cases=[])
    b = lg.Batch(ctx, pb)
    try:
        for k, share in enumerate(SHARES):
            flags, H = with_het_share(pb, share, 1000 + k)
            b.upload(site_flags=flags)
            case = dict(het_share=share, H=H)
            for m in modes.values():
                for _ in range(a.warmup):
                    b.run(mc, m)
                    b.sync()
            t = {name: dict(kernel_ms=[], dense_kernel_ms=[], gram_kernel_ms=[]) for name in modes}
            res = {}
            for _ in range(a.reps):
                for name, m in modes.items():
                    b.run(mc, m)
                    r = b.download()
                    res[name] = r
                    for f in t[name]:
                        t[name][f].append(getattr(r, f))
            for name in modes:
                r = res[name]
                case[name] = dict({f: stats(v) for f, v in t[name].items()}, dense_macs=r.dense_macs,
                                  gram_macs=r.gram_macs, n_records=r.n_records, n_evaluated=r.n_evaluated,
                                  n_dense_four=r.n_dense_four, sha256=digest(r))
                if not a.no_profile:
                    case[name]["kernels_ms"] = kernel_times(b, mc, modes[name])
            case["same_rows_and_means"] = case["het_only"]["sha256"] == case["skip_nonhet"]["sha256"]
            case["step_speedup_median"] = case["het_only"]["kernel_ms"]["median"] / case["skip_nonhet"]["kernel_ms"]["median"]
            out["cases"].append(case)
            print(json.dumps({kk: case[kk] for kk in ("het_share", "H", "same_rows_and_means", "step_speedup_median")}),
                  flush=True)
    finally:
        b.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    if not all(c["same_rows_and_means"] for c in out["cases"]):
        sys.exit("rows or means differ between the two forms")


if __name__ == "__main__":
    main()
