#!/usr/bin/env python
"""Batched least squares on device-resident data (Engine.least_squares_batch_device, lsqr_least_squares_batch_device).
Workloads a user runs: 65 536 planes x 256 points, 65 536 weighted absolute orientations x 256 pairs, 512 planes x 50 000
points and 64 spheres x 150 000 points with the geometric (Levenberg-Marquardt) fit; every input is larger than the L2 cache.

Per workload: device time of one call from CUDA events, median of --reps runs after a warm-up; the algorithmic bytes of one
pass (records x dim x 8, plus 8 per weight); for the one-pass workloads their rate against a device-to-device copy measured in
the same run (read + write bytes over time) and against the data sheet's 7.7 TB/s.  For comparison on the same data: the
plane fit in torch (per-problem scatter by einsum, then torch.linalg.eigh), and a Python loop of Engine.least_squares over
1 024 problems, per problem.  One JSON object per line:

  python tools/ls_batch_probe.py [--reps 7] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from batch_device_probe import gpu_info, make_data  # noqa: E402
from lsqrrecipes_b200 import Engine, synth  # noqa: E402

# (name, model, problems, records per problem, least-squares type, weighted)
WORKLOADS = [("plane3_65536x256", "plane3", 65536, 256, 1, False), ("absor_weighted_65536x256", "absor", 65536, 256, 1, True),
             ("plane3_512x50000", "plane3", 512, 50_000, 1, False), ("sphere3_geometric_64x150000", "sphere3", 64, 150_000, 1, False)]
DATASHEET_BPS = 7.7e12
LOOP_PROBLEMS = 1024


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return statistics.median(ms), ms


def copy_bandwidth(reps):
    import torch
    src = torch.empty(1 << 28, dtype=torch.float64, device="cuda")   # 2 GiB
    dst = torch.empty_like(src)
    ms, _ = timed(lambda: dst.copy_(src), reps)
    return 2 * src.numel() * 8 / (ms * 1e-3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ls_batch_probe: no CUDA device")
    out_file = open(args.out, "w") if args.out else None

    def emit(**kw):
        line = json.dumps(kw)
        print(line, flush=True)
        if out_file:
            out_file.write(line + "\n")
            out_file.flush()

    copy_bps = copy_bandwidth(args.reps)
    emit(kind="device", **gpu_info(), d2d_copy_bytes_per_s=copy_bps)
    for label, name, count, n, ls_type, weighted in WORKLOADS:
        eng = Engine(name, synth.DELTAS[name], ls_type=ls_type)
        data, offsets = make_data(name, count, n)
        x = torch.from_numpy(data).cuda().reshape(count, n, eng.dim)
        w = torch.from_numpy(np.random.default_rng(3).uniform(0.1, 2.0, (count, n))).cuda() if weighted else None
        ms, runs = timed(lambda: eng.least_squares_batch_device(x, weights=w), args.reps)
        nbytes = count * n * eng.dim * 8 + (count * n * 8 if weighted else 0)
        rec = dict(kind="workload", workload=label, problems=count, records=n, device_ms=ms, runs_ms=runs, algorithmic_bytes=nbytes)
        if name != "sphere3":   # one pass over the data; the geometric fit takes one pass per LM evaluation
            bps = nbytes / (ms * 1e-3)
            rec.update(bytes_per_s=bps, share_of_d2d_copy=bps / copy_bps, share_of_datasheet_7_7TBps=bps / DATASHEET_BPS)
        if name == "plane3":
            # cuSOLVER's batched eigh refuses 65 536 matrices in one call (CUSOLVER_STATUS_INVALID_VALUE on one B200, torch 2.11):
            # the largest chunk it takes is used, and reported
            for chunk in (count, 16384, 4096, 1024):
                def torch_plane():
                    mean = x.mean(dim=1, keepdim=True)
                    xc = x - mean
                    cov = torch.einsum("bni,bnj->bij", xc, xc)
                    return [torch.linalg.eigh(cov[i:i + chunk]) for i in range(0, count, chunk)]
                try:
                    rec["torch_einsum_eigh_ms"], _ = timed(torch_plane, args.reps)
                    rec["torch_eigh_chunk"] = chunk
                    break
                except RuntimeError as e:
                    rec.setdefault("torch_eigh_refused", []).append([chunk, str(e).split(",")[0]])
        lp = min(LOOP_PROBLEMS, count)
        host = data.reshape(count, n, eng.dim)
        ww = w.cpu().numpy() if weighted else None
        t0 = time.perf_counter()
        for i in range(lp):
            if weighted:
                eng.weighted_least_squares(host[i], ww[i])
            else:
                eng.least_squares(host[i])
        rec["loop_least_squares_ms_per_problem"] = (time.perf_counter() - t0) * 1e3 / lp
        rec["device_ms_per_problem"] = ms / count
        emit(**rec)
        eng.close()
        del x, w
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
