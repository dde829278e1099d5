#!/usr/bin/env python
"""Batched RANSAC on data that already live in a CUDA tensor (Engine.ransac_batch_device, lsqr_ransac_batch_device) against
the host entry point on the same problems.  Workloads: 65 536 problems x 256 points (plane3 and line2d, fp32 and fp64 scoring,
the data of bench.py's configs[4] entries and its 2048-hypothesis cap), 512 plane3 problems x 50 000 points (one thread-block
cluster per problem, both precisions) and 64 spheres x 150 000 points (fp32 scoring, Levenberg-Marquardt refit), the last two
as in tools/batch_cluster_probe.py.  The arms alternate, --reps times each:

  (a) host_pinned    ransac_batch from page-locked memory
  (b) host_pageable  ransac_batch from pageable memory
  (c) cpu_then_host  what a CUDA-tensor user does without the device entry point: tensor.cpu(), then (b)
  (d) device         ransac_batch_device on the tensor: wall time from the call to torch.cuda.synchronize(), and device time
                     from CUDA events recorded around the call on the stream it runs on

Every line carries (a)'s device_ms (kernel time of the host path); each (d) line says whether its outputs are bitwise equal to
(a)'s of the same repetition.  The last line of a workload holds each arm's median.  One JSON object per line:

  python tools/batch_device_probe.py [--reps 3] [--out FILE]
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

# (model, problems, points per problem, scoring precision, least-squares type, cap on hypotheses per problem)
WORKLOADS = [("plane3", 65536, 256, FP32, 1, 2048), ("plane3", 65536, 256, FP64, 1, 2048),
             ("line2d", 65536, 256, FP32, 1, 2048), ("line2d", 65536, 256, FP64, 1, 2048),
             ("plane3", 512, 50_000, FP64, 1, 1024), ("plane3", 512, 50_000, FP32, 1, 1024),
             ("sphere3", 64, 150_000, FP32, 1, 1024)]
PROB, SEED = 0.999, 7
ARMS = ("host_pinned", "host_pageable", "cpu_then_host", "device")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    name, power = (c.strip() for c in out.strip().split(","))
    return {"gpu": name, "power_limit": power}


def make_data(name, count, n):
    """65 536 x 256: bench.py's configs[4] data (64 base problems, each copy shifted); larger problems: one draw each"""
    if count == 65536:
        rng = np.random.default_rng(17)
        D = synth.GENERATORS[name](8, seed=1)[0].shape[1]
        bases = [synth.GENERATORS[name](n, seed=300 + i)[0] for i in range(64)]
        data = np.concatenate([bases[i % 64] for i in range(count)]) + np.repeat(rng.uniform(-50, 50, (count, D)), n, axis=0)
    else:
        data = np.concatenate([synth.GENERATORS[name](n, seed=100 + i)[0][:n] for i in range(count)])
    return np.ascontiguousarray(data), (np.arange(count + 1, dtype=np.uint64) * np.uint64(n))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("batch_device_probe: no CUDA device")

    out_file = open(args.out, "w") if args.out else None

    def emit(**kw):
        line = json.dumps(kw)
        print(line, flush=True)
        if out_file:
            out_file.write(line + "\n")
            out_file.flush()

    info = gpu_info()
    emit(kind="device", **info)
    for name, count, n, precision, ls_type, tries in WORKLOADS:
        eng = Engine(name, synth.DELTAS[name], ls_type=ls_type)
        data, offsets = make_data(name, count, n)
        pinned_t = torch.from_numpy(data).pin_memory()
        pinned = pinned_t.numpy()
        dev = torch.from_numpy(data).cuda()
        torch.cuda.synchronize()
        kw = dict(prob=PROB, max_tries=tries, seed=SEED, precision=precision)
        common = dict(workload=name, problems=count, points=n, precision="fp32" if precision == FP32 else "fp64", ls_type=ls_type,
                      max_tries=tries, host_bytes=int(data.nbytes), **info)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def run(arm):
            """(wall ms, device ms, outputs as numpy)"""
            if arm == "device":
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                e0.record()
                o = eng.ransac_batch_device(dev, offsets, **kw)
                e1.record()
                torch.cuda.synchronize()
                wall = 1e3 * (time.perf_counter() - t0)
                return wall, e0.elapsed_time(e1), {"params": o["params"].cpu().numpy(), "counts": o["counts"].cpu().numpy().astype(np.uint32)}
            t0 = time.perf_counter()
            src = dev.cpu().numpy() if arm == "cpu_then_host" else (pinned if arm == "host_pinned" else data)
            o = eng.ransac_batch(src, offsets, **kw)
            return 1e3 * (time.perf_counter() - t0), o["device_ms"], o

        for arm in ARMS:   # warm-up: modules, buffers at this size, both staging slots of the device path
            run(arm)
        run("device")
        walls = {a: [] for a in ARMS}
        dms = {a: [] for a in ARMS}
        equal_all = True
        for rep in range(args.reps):
            res = {arm: run(arm) for arm in ARMS}
            a_ms, a_out = res["host_pinned"][1], res["host_pinned"][2]
            for arm in ARMS:
                wall, dm, o = res[arm]
                walls[arm].append(wall)
                dms[arm].append(dm)
                line = dict(kind="arm", arm=arm, rep=rep, wall_ms=wall, device_ms=dm, host_pinned_device_ms=a_ms, problems_per_s=count / (wall * 1e-3))
                if arm == "device":
                    eq = o["params"].tobytes() == a_out["params"].tobytes() and np.array_equal(o["counts"], a_out["counts"])
                    equal_all &= eq
                    line["bitwise_equal_to_host_pinned"] = bool(eq)
                    line["mean_consensus"] = float(o["counts"].mean())
                emit(**line, **common)
        emit(kind="summary", equal=equal_all, **{f"wall_ms_{a}": float(np.median(walls[a])) for a in ARMS},
             **{f"device_ms_{a}": float(np.median(dms[a])) for a in ARMS},
             speedup_device_vs_host_pinned=float(np.median(walls["host_pinned"]) / np.median(walls["device"])),
             speedup_device_vs_cpu_then_host=float(np.median(walls["cpu_then_host"]) / np.median(walls["device"])), **common)
        eng.close()
        del dev, pinned, pinned_t
        torch.cuda.empty_cache()
    if out_file:
        out_file.close()


if __name__ == "__main__":
    main()
