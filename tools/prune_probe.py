#!/usr/bin/env python
"""Early exit of fp32 scoring, measured: the bench workload (plane3, 10 M points, 1 M Philox hypotheses, fp32, a 256 MB L2 flush
before every call) scored with per-hypothesis counts (the full pass) and without them (the early exit), alternated, same seeds.
Per arm: consensus_ms, executed evaluations over H x N, executed evaluations per second over the live FFMA2 peak, and
whether the winners agree.  A separate profiled call counts the compactions and the seed and sums their device time.  Then
plane3, sphere3 and line2d at 1 M points x 2^20 hypotheses.  One JSON object per line:

  python tools/prune_probe.py [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import FLOP_PER_EVAL  # noqa: E402
from lsqrrecipes_b200 import FP32, Engine, synth  # noqa: E402

WINNER = ("best_index", "best_count", "n_valid", "best_subset", "best_params")


def emit(**kw):
    print(json.dumps(kw), flush=True)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    name, power = (c.strip() for c in out.strip().split(","))
    return {"gpu": name, "power_limit": power}


def same_winner(a, b):
    return all(np.array_equal(np.atleast_1d(a[k]).view(np.uint8), np.atleast_1d(b[k]).view(np.uint8)) for k in WINNER)


def profile_prune(eng, H, seed, flush):
    """Device time of the early exit's own kernels in one call, from torch.profiler (a run of its own: tracing slows the host)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    flush.zero_()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.score(count=H, precision=FP32, seed=seed)
        torch.cuda.synchronize()
    ms, calls = {}, {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        t = getattr(e, "cuda_time_total", 0.0) if t is None else t
        for tag in ("prune_tally_kernel", "prune_move_kernel", "prune_scatter_kernel", "prune_seed_kernel", "consensus32_kernel", "argmax_kernel",
                    "consensus_cb_kernel"):
            if tag in e.key:
                ms[tag] = ms.get(tag, 0.0) + t / 1e3
                calls[tag] = calls.get(tag, 0) + e.count
    compact_ms = ms.get("prune_tally_kernel", 0.0) + ms.get("prune_move_kernel", 0.0) + ms.get("prune_scatter_kernel", 0.0)
    seed_ms = ms.get("prune_seed_kernel", 0.0) + ms.get("consensus32_kernel", 0.0)
    return {"compactions": calls.get("prune_tally_kernel", 0), "compaction_kernels_ms": compact_ms, "seed_kernels_ms": seed_ms,
            "consensus_cb_kernel_ms": ms.get("consensus_cb_kernel", 0.0), "consensus_cb_launches": calls.get("consensus_cb_kernel", 0),
            "kernel_ms": ms, "kernel_calls": calls}


def arms(name, n, H, reps, peak, flush, label):
    import torch
    data, _ = synth.GENERATORS[name](n)
    eng = Engine(name, synth.DELTAS[name])
    eng.upload(data)
    del data
    eng.score(count=H, precision=FP32, seed=999, want_counts=True)      # warm-up, both paths
    eng.score(count=H, precision=FP32, seed=999)
    res = {"full": [], "early_exit": []}
    agree = True
    for i in range(reps):
        out = {}
        for arm, want in (("full", True), ("early_exit", False)):
            flush.zero_()
            torch.cuda.synchronize()
            out[arm] = eng.score(count=H, precision=FP32, seed=i, want_counts=want)
            res[arm].append(out[arm])
        agree = agree and same_winner(out["full"], out["early_exit"])
    rec = {"config": label, "model": name, "points": n, "hypotheses": H, "reps": reps, "winners_equal": bool(agree)}
    for arm, rs in res.items():
        ms = [r["consensus_ms"] for r in rs]
        ev = [r["evals"] for r in rs]
        rec[arm] = {"consensus_ms": ms, "consensus_ms_median": float(np.median(ms)), "evals_over_HN": [e / (H * n) for e in ev],
                    "executed_frac_of_ffma_peak": [e * FLOP_PER_EVAL[name] / (m * 1e-3) / peak for e, m in zip(ev, ms)],
                    "best_count": [r["best_count"] for r in rs]}
    rec["speedup_consensus_median"] = rec["full"]["consensus_ms_median"] / rec["early_exit"]["consensus_ms_median"]
    rec["profiled_early_exit_call"] = profile_prune(eng, H, 0, flush)
    eng.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-models", action="store_true", help="the bench workload only")
    args = ap.parse_args()
    import torch
    info = gpu_info()
    probe = Engine("plane3", 0.5)
    ffma, _ = probe.microbench_fma(0, 8192)
    ffma2, _ = probe.microbench_fma(1, 8192)
    probe.close()
    peak = max(ffma, ffma2) * 2                  # FLOP/s, the better of the measured FFMA and FFMA2 chains (as bench.py)
    emit(**info, ffma_tflops=ffma * 2 / 1e12, ffma2_tflops=ffma2 * 2 / 1e12)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    emit(**info, **arms("plane3", 10_000_000, 1_000_000, args.reps, peak, flush, "bench workload: plane3, 10M points, 1M Philox hypotheses, fp32"))
    if not args.no_models:
        for name in ("plane3", "sphere3", "line2d"):
            emit(**info, **arms(name, 1_000_000, 1 << 20, 2, peak, flush, f"{name}, 1M points x 2^20 hypotheses, fp32"))


if __name__ == "__main__":
    main()
