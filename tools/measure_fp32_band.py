#!/usr/bin/env python
"""Evidence for the fp32 band of tests/test_parity_gpu.py: how far from the threshold can a datum be and still be decided
differently by the fp32 fast mode?

For every estimator H Philox hypotheses are scored in fp32 and in fp64 (same parameter vectors).  For the hypotheses with the
largest count differences the residuals are recomputed in float64 numpy; a difference of k decisions needs the k data closest to
the threshold, so the k-th smallest | |residual| - delta | is the band that hypothesis needs.  Reported per model: the largest
needed band, absolute and as a fraction of the band the test allows (oracle/fast32.py fp32_band); the test's constants are set so that this
fraction stays below one half.   python tools/measure_fp32_band.py [n] [H] [model ...]"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lsqrrecipes_b200 import FP32, FP64, MODELS, SAMPLE_PARAMS, Engine, synth  # noqa: E402
from oracle.fast32 import fp32_band as _fp32_band  # noqa: E402
from oracle.fast32 import residual64 as _residual64  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 200_000
H = int(sys.argv[2]) if len(sys.argv) > 2 else 20_000
only = sys.argv[3:]
for name in MODELS:
    if only and name not in only:
        continue
    data, _ = synth.GENERATORS[name](n, seed=4711)
    delta = synth.DELTAS[name]
    eng = Engine(name, delta)
    eng.upload(data)
    r32 = eng.score(count=H, seed=5, precision=FP32, want_counts=True, want_params=True)
    prm = r32["params"]
    ok = ~np.isnan(prm[:, 0])
    c32 = r32["counts"].astype(np.int64)
    c64 = eng.score(sampler=SAMPLE_PARAMS, params=prm, precision=FP64, want_counts=True)["counts"].astype(np.int64)
    eng.close()
    diff = np.where(ok, np.abs(c32 - c64), 0)
    worst = np.argsort(-diff)[:256]
    need_abs, need_frac, at = 0.0, 0.0, None
    for h in worst:
        if diff[h] == 0:
            break
        res, thr = _residual64(name, prm[h], data, delta)
        gap = np.partition(np.abs(res - thr), int(diff[h]) - 1)[int(diff[h]) - 1]      # k-th smallest distance to the threshold
        allowed = _fp32_band(name, data, prm[h], delta)
        need_abs = max(need_abs, float(gap))
        if gap / allowed > need_frac:
            need_frac, at = float(gap / allowed), int(h)
    print(json.dumps({"model": name, "points": n, "hypotheses": int(ok.sum()), "max_count_diff": int(diff.max()), "sum_count_diff": int(diff.sum()),
                      "sum_counts": int(c64[ok].sum()), "needed_band_abs_max": need_abs, "needed_over_allowed_max": need_frac, "worst_hypothesis": at,
                      "allowed_band_of_worst": float(_fp32_band(name, data, prm[at], delta)) if at is not None else None, "delta": delta}), flush=True)
