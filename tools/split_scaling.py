#!/usr/bin/env python
"""Host-to-host time of DevicePool.run over the first N = 1, 2, 4, 8 GPUs of the box, in one process, on
  (a) the cfg3 unit alone (2 000 sites x 100 000 reads), which the pool splits by rows of its pair grid, and
  (b) cfg4 (20 000 heavy-tailed units) plus that unit: a transcriptome with one deep gene.
Per N: best and median of --reps calls after a warm-up call (each call ends with the results on the host), the
kernel time of each device's batch of pieces, the time of the split unit's per-site pass (split_means, host
clock), the number of pieces, and a sha256 of records + means + counts, which must be the same for every N.
The GPU's name and power limit are read in the same run.  Writes <out-dir>/r3_split_scaling_n{N}.json.
--one-device N: the pool over N contexts on GPU 0 instead (r3_split_scaling_n{N}_one_device.json): the same
split, piece batches, copies and gather, but no device-level parallelism -- what the split itself costs.

    python tools/split_scaling.py [--reps 10] [--out-dir profiles] [--one-device N ...]"""
import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
lg = importlib.import_module("l-giremi_b200")
synth = importlib.import_module("l-giremi_b200.synth")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return [dict(zip(("name", "power_limit"), [x.strip() for x in line.split(",")])) for line in out]


def digest(res):
    h = hashlib.sha256()
    for a in (res.records, res.site_mean, res.site_cnt):
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def measure(pool, pb, reps, mode):
    res = pool.run(pb, 6, mode)                                  # warm-up: modules, pools, peer access
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        res = pool.run(pb, 6, mode)
        times.append(1e3 * (time.perf_counter() - t0))
    split = getattr(res, "split_units", {})
    return {
        "host_to_host_ms_best": min(times), "host_to_host_ms_median": float(np.median(times)),
        "host_to_host_ms_all": times,
        "piece_kernel_ms": [x for x in pool.last_piece_ms if x is not None],
        "split_means_ms": pool.last_split_means_ms,
        "n_pieces": sum(len(v) for v in split.values()),
        "pieces": {str(u): v for u, v in split.items()},
        "n_records": int(res.n_records),
        "sha256": digest(res),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out-dir", default="profiles")
    ap.add_argument("--one-device", type=int, nargs="*", default=None, metavar="N")
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    mode = lg.MODE_HET_ONLY
    n_gpus = lg.device_count()
    if n_gpus < 1:
        raise SystemExit("no GPU")
    cfg3, _ = synth.make_deep_unit(20261021, 2000, 100000, 0.6)
    cfg4, _ = synth.make_heavy_tail(20261022, 20000)
    mixed = lg.concat_plane_batches([cfg4, cfg3])
    info = gpu_info()
    hashes = {}
    one = args.one_device is not None
    for n in ([1] + args.one_device if one else (1, 2, 4, 8)):
        if not one and n > n_gpus:
            break
        pool = lg.DevicePool([0] * n if one else list(range(n)))
        try:
            out = {"n_gpus": 1 if one else n, "n_contexts": n, "gpus": info[:1 if one else n], "mode": "HET_ONLY",
                   "min_common": 6, "reps": args.reps}
            for name, pb in (("cfg3", cfg3), ("cfg4_plus_cfg3", mixed)):
                out[name] = measure(pool, pb, args.reps, mode)
                hashes.setdefault(name, out[name]["sha256"])
                out[name]["same_as_n1"] = out[name]["sha256"] == hashes[name]
        finally:
            pool.close()
        path = os.path.join(args.out_dir, "r3_split_scaling_n%d%s.json" % (n, "_one_device" if one and n > 1 else ""))
        with open(path, "w") as f:
            json.dump(out, f, indent=1)
        print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items()
                                                                if kk not in ("host_to_host_ms_all", "pieces")})
                          for k, v in out.items()}))


if __name__ == "__main__":
    main()
