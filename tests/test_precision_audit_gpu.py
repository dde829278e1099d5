"""SURVEY.md 8d, config 2, at its full size: the precision audit of the two scoring modes on 10 M points.

  * fp64 validation mode: 10^4 hypotheses x 10 M points (10^11 agree() evaluations) recounted by the CPU oracle -- every count
    bit-exact, the arg-max the oracle's;
  * fp32 fast mode against the fp64 mode over 131 072 hypotheses x 10 M points (1.3 * 10^12 evaluations each): every count
    difference of every hypothesis is explained by data whose fp64 residual lies inside the fp32 rounding band of the
    threshold (the band of oracle/fast32.py::fp32_band, whose constants are twice what tools/measure_fp32_band.py
    measured); the band is counted on the GPU by scoring the same hypotheses in fp64 at delta + band and delta - band.
"""
import numpy as np
import pytest

from lsqrrecipes_b200 import FP32, FP64, SAMPLE_LIST, SAMPLE_PARAMS, Engine, synth
from oracle.pyoracle import MODELS
from oracle.fast32 import fp32_band as _fp32_band

pytestmark = pytest.mark.gpu

N_POINTS = 10_000_000


@pytest.fixture(scope="module")
def plane10m():
    return synth.GENERATORS["plane3"](N_POINTS)


def test_fp64_mode_10k_hypotheses_x_10m_points_bit_exact(port, plane10m):
    data, _ = plane10m
    m, delta = MODELS["plane3"], synth.DELTAS["plane3"]
    subs = synth.random_subsets(N_POINTS, 3, 10_000, seed=2031)
    c_ref, p_ref = port.score_subsets(m, delta, data, subs)          # ~25 s on the GPU box's host cores
    eng = Engine("plane3", delta)
    eng.upload(data)
    r = eng.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP64, want_counts=True, want_params=True)
    assert np.array_equal(r["counts"], c_ref)
    assert np.array_equal(r["params"], p_ref)
    assert r["best_index"] == int(np.argmax(c_ref)) and r["best_count"] == int(c_ref.max())
    eng.close()


def test_fp32_mode_vs_fp64_mode_131072_hypotheses_x_10m_points(plane10m):
    data, _ = plane10m
    delta = synth.DELTAS["plane3"]
    H = 131_072
    eng = Engine("plane3", delta)
    eng.upload(data)
    r32 = eng.score(count=H, seed=2032, precision=FP32, want_counts=True, want_params=True)      # constant-bank kernel
    prm = r32["params"]
    ok = ~np.isnan(prm[:, 0])
    c32 = r32["counts"].astype(np.int64)
    c64 = eng.score(sampler=SAMPLE_PARAMS, params=prm, precision=FP64, want_counts=True)["counts"].astype(np.int64)
    # one band for all: the widest the per-hypothesis formula gives (plane parameters are a unit normal and a data point)
    band = max(_fp32_band("plane3", data, prm[h], delta) for h in np.flatnonzero(ok)[:: max(1, H // 512)])
    band = max(band, _fp32_band("plane3", data, prm[np.flatnonzero(ok)[np.argmax(np.abs(prm[ok]).max(axis=1))]], delta))
    eng.set_estimator(delta + band)
    hi = eng.score(sampler=SAMPLE_PARAMS, params=prm, precision=FP64, want_counts=True)["counts"].astype(np.int64)
    eng.set_estimator(delta - band)
    lo = eng.score(sampler=SAMPLE_PARAMS, params=prm, precision=FP64, want_counts=True)["counts"].astype(np.int64)
    eng.close()
    diff = np.abs(c32 - c64)
    assert np.all(diff[ok] <= (hi - lo)[ok]), "an fp32 decision differs outside the rounding band of the threshold"
    assert np.all(c32[~ok] == 0) and np.all(c64[~ok] == 0)
    # ... and the band is narrow: it holds a vanishing share of the data, so do the differences
    # (data spread evenly over the slab of half-width delta put 2 band / delta of the count inside the band; the synthetic
    # inliers are denser near the plane than at the threshold, so that is an upper estimate -- allow it once over)
    assert band <= 1e-6 * np.abs(data).max(), "the band must stay within the north star's 1e-6 of the coordinate scale"
    assert (hi - lo)[ok].sum() <= 4 * band / delta * c64[ok].sum()
    assert diff[ok].sum() <= 2e-5 * c64[ok].sum()
    assert int(np.argmax(c32)) == int(np.argmax(c64)) or abs(int(c32.max()) - int(c64.max())) <= int((hi - lo)[int(np.argmax(c64))])
