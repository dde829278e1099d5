#!/usr/bin/env python
"""Batched RANSAC on problems too large for one thread block (one thread-block cluster per problem), measured against the
loop a user runs without it: one lsqr_compute per problem over the same host arrays.  Workloads: 512 3-D plane problems x
50 000 points (40 % outliers) with fp64 and with fp32 scoring, 2 048 2-D line problems x 15 000 points, 64 spheres x 150 000
points with fp32 scoring (150 000 3-D points exceed the fp64 capacity) and the geometric (Levenberg-Marquardt) refit.  The arms alternate: one lsqr_ransac_batch call from pageable memory,
the same call from page-locked memory, the loop.  Per arm: wall time, problems/s, device_ms (batch) and the mean consensus
size.  One JSON object per line:

  python tools/batch_cluster_probe.py [--reps 2] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lsqrrecipes_b200 import FP32, FP64, Engine, synth  # noqa: E402

WORKLOADS = [("plane3", 512, 50_000, FP64, 1), ("plane3", 512, 50_000, FP32, 1), ("line2d", 2048, 15_000, FP64, 1),
             ("sphere3", 64, 150_000, FP32, 1)]
PROB, TRIES, SEED = 0.999, 1024, 7


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    name, power = (c.strip() for c in out.strip().split(","))
    return {"gpu": name, "power_limit": power}


def cluster_size(n, dim, precision):
    """the cluster lsqr_ransac_batch picks: the smallest whose 200 KiB slices hold the problem (fp64 rows, or fp32 rows)"""
    width = 4 if precision == FP32 else 8
    slice_ = (200 * 1024 // (dim * width)) & ~1
    for c in (2, 4, 8, 16):
        if (((n + c - 1) // c + 1) & ~1) <= slice_:
            return c
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    out_file = open(args.out, "w") if args.out else None

    def emit(**kw):
        line = json.dumps(kw)
        print(line, flush=True)
        if out_file:
            out_file.write(line + "\n")
            out_file.flush()

    info = gpu_info()
    emit(kind="device", **info)
    for name, count, n, precision, ls_type in WORKLOADS:
        eng = Engine(name, synth.DELTAS[name], ls_type=ls_type)
        one, most = eng.batch_capacity(precision)
        gen = synth.GENERATORS[name]
        data = np.concatenate([gen(n, seed=100 + i)[0] for i in range(count)])
        offsets = (np.arange(count + 1, dtype=np.uint64) * n).astype(np.uint64)
        pinned_t = torch.empty(data.shape, dtype=torch.float64, pin_memory=True)
        pinned = pinned_t.numpy()
        pinned[...] = data
        common = dict(workload=name, problems=count, points=n, precision="fp32" if precision == FP32 else "fp64", ls_type=ls_type,
                      one_block=one, max_records=most, cluster=cluster_size(n, data.shape[1], precision), **info)
        eng.ransac_batch(data[: 4 * n], offsets[:5], prob=PROB, max_tries=TRIES, seed=SEED, precision=precision)   # warm-up
        eng.compute(data[:n], PROB, precision=precision, seed=SEED)
        for rep in range(args.reps):
            for arm, src in (("batch_pageable", data), ("batch_pinned", pinned)):
                t0 = time.perf_counter()
                out = eng.ransac_batch(src, offsets, prob=PROB, max_tries=TRIES, seed=SEED, precision=precision)
                wall = time.perf_counter() - t0
                emit(kind="arm", arm=arm, rep=rep, wall_s=wall, problems_per_s=count / wall, device_ms=out["device_ms"],
                     mean_consensus=float(out["counts"].mean()), **common)
            counts = np.zeros(count)
            t0 = time.perf_counter()
            for i in range(count):
                r = eng.compute(data[i * n:(i + 1) * n], PROB, precision=precision, seed=SEED + i, want_mask=False)
                counts[i] = r["best_count"]
            wall = time.perf_counter() - t0
            emit(kind="arm", arm="compute_loop", rep=rep, wall_s=wall, problems_per_s=count / wall, mean_consensus=float(counts.mean()), **common)
        eng.close()
        del pinned, pinned_t
    if out_file:
        out_file.close()


if __name__ == "__main__":
    main()
