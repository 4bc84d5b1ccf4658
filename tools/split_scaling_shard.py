#!/usr/bin/env python
"""The split of a deep unit in the one-process-per-GPU launch (shard.local_run + shard.gather_run_to_rank0), timed
under torch.distributed.run on
  (a) the cfg3 unit alone (2 000 sites x 100 000 reads), and
  (b) cfg4 (20 000 heavy-tailed units) plus that unit.
Rank r drives GPU r, or GPU 0 when the box has fewer GPUs than ranks (then the pieces' copies and MI slices go
between processes on one device: the run shows correctness and the split's overhead, not a speed-up).  Per case:
best and median end-to-end step time over --reps calls after a warm-up call (local_run on every rank, then the
gather, merged rows on rank 0's host), each rank's piece-batch host time and kernel time, the split_means_ipc time
on the unit's owner, and a sha256 of records + means + counts of the merged result against one GPU's
mi_step_batched of the whole batch.  The GPUs' name and power limit are read in the same run.  Handles and rows go
through the gloo backend: no NCCL.  Rank 0 writes <out-dir>/r3_shard_split_n{N}[_one_device].json.

    python -m torch.distributed.run --nproc_per_node N tools/split_scaling_shard.py [--reps 5] [--out-dir profiles]"""
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
shard = importlib.import_module("l-giremi_b200.shard")
synth = importlib.import_module("l-giremi_b200.synth")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return [dict(zip(("name", "power_limit"), [x.strip() for x in line.split(",")])) for line in out]


def digest(res):
    h = hashlib.sha256()
    for a in (res.records, res.site_mean, res.site_cnt):
        h.update(np.ascontiguousarray(a).tobytes())
    if res.counts is not None:
        h.update(np.ascontiguousarray(res.counts).tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out-dir", default="profiles")
    args = ap.parse_args()
    import torch.distributed as dist
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    n_gpus = lg.device_count()
    if n_gpus < 1:
        raise SystemExit("no GPU")
    one_device = n_gpus < world
    ctx = lg.Context(0 if one_device else int(os.environ.get("LOCAL_RANK", rank)))
    mode = lg.MODE_HET_ONLY
    cfg3, _ = synth.make_deep_unit(20261021, 2000, 100000, 0.6)
    cfg4, _ = synth.make_heavy_tail(20261022, 20000)
    cases = (("cfg3", cfg3), ("cfg4_plus_cfg3", lg.concat_plane_batches([cfg4, cfg3])))
    out = {"world": world, "n_gpus_used": 1 if one_device else world, "one_device": one_device,
           "gpus": gpu_info()[:1 if one_device else world], "mode": "HET_ONLY", "min_common": 6, "reps": args.reps,
           "backend": "gloo (handles and rows); pieces' planes and MI slices over CUDA IPC"}
    for name, pb in cases:
        times, per_rank = [], []
        merged = None
        for rep in range(args.reps + 1):                      # the first call warms up modules and pools
            dist.barrier()
            t0 = time.perf_counter()
            run = shard.local_run(pb, rank, world, 6, mode, ctx)
            merged = shard.gather_run_to_rank0(pb, run)
            ms = 1e3 * (time.perf_counter() - t0)
            if rep:
                times.append(ms)
                per_rank.append({"shard_ms": run.shard_ms, "pieces_ms": run.pieces_ms,
                                 "piece_kernel_ms": run.piece_kernel_ms,
                                 "split_means_ipc_ms": run.split_means_ms if run.means else None})
        ranks = [None] * world
        dist.all_gather_object(ranks, per_rank)
        if rank == 0:
            single = lg.mi_step_batched(pb, 6, mode, ctx=ctx)
            want, got = digest(single), digest(merged)
            out[name] = {
                "step_ms_best": min(times), "step_ms_median": float(np.median(times)), "step_ms_all": times,
                "per_rank": [{k: [r[k] for r in ranks[q]] for k in ranks[q][0]} for q in range(world)],
                "pieces": {str(u): v for u, v in merged.split_units.items()},
                "n_records": int(merged.n_records), "sha256": got, "single_gpu_sha256": want,
                "identical_to_single_gpu": got == want,
            }
    ctx.close()
    if rank == 0:
        os.makedirs(args.out_dir, exist_ok=True)
        path = os.path.join(args.out_dir, "r3_shard_split_n%d%s.json" % (world, "_one_device" if one_device else ""))
        with open(path, "w") as f:
            json.dump(out, f, indent=1)
        print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items()
                                                                if kk not in ("step_ms_all", "per_rank")})
                          for k, v in out.items()}))
    dist.destroy_process_group()
    if rank == 0 and not all(out[name]["identical_to_single_gpu"] for name, _pb in cases):
        raise SystemExit("merged result differs from one GPU's")


if __name__ == "__main__":
    main()
