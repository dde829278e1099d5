"""BASELINE.json's configurations at their FULL sizes (10 M points, 1 M hypotheses, 1 M correspondences, 65 536 small
problems) on the GPU, checked through properties that do not need the CPU to redo 10^13 evaluations:

  * a slice of hypotheses is still compared with the oracle directly on all 10 M points (fp64, bit-exact);
  * partition additivity: counts over the data = counts over its two halves added (fp64, bit-exact);
  * sampler partition independence: scoring hypotheses [0, H) in one request or in two gives the same winner;
  * fp32 counts differ from fp64 counts by no more than the number of points inside the fp32 rounding band;
  * the consensus mask of the winner is bit-exact against the oracle and the refit of that mask agrees to 1e-6;
  * compute(): the returned fraction, mask and parameters are mutually consistent when re-derived by the oracle;
  * batched mode: popcount(mask) = count and the oracle's refit of each sampled mask reproduces the parameters.
"""
import numpy as np
import pytest

from conftest import SIGN_IDX, same_up_to_sign
from lsqrrecipes_b200 import FP32, FP64, SAMPLE_LIST, SAMPLE_PARAMS, Engine, synth
from oracle.pyoracle import MODELS
from oracle.fast32 import fp32_band as _fp32_band

pytestmark = pytest.mark.gpu

N_POINTS = 10_000_000
N_HYPS = 1_000_000
REFINE_TOL = 1e-6


@pytest.fixture(scope="module")
def plane10m():
    data, true = synth.GENERATORS["plane3"](N_POINTS)
    return data, true


def test_plane_10m_fp64_counts_vs_oracle_and_partition_additivity(port, plane10m):
    """configs[1], fp64 validation: 48 hypotheses x 10 M points recounted by the oracle, bit-exact; the same counts as
    the sum over two uneven parts of the data."""
    data, _ = plane10m
    m, delta = MODELS["plane3"], synth.DELTAS["plane3"]
    subs = synth.random_subsets(N_POINTS, 3, 48, seed=2026)
    c_ref, p_ref = port.score_subsets(m, delta, data, subs)
    eng = Engine("plane3", delta)
    eng.upload(data)
    r = eng.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP64, want_counts=True, want_params=True)
    assert np.array_equal(r["counts"], c_ref)
    assert np.array_equal(r["params"], p_ref), "estimate() is plain double arithmetic: bit-exact"
    assert r["best_index"] == int(np.argmax(c_ref)) and r["best_count"] == int(c_ref.max())
    eng.close()
    cut = 3_333_337
    parts = []
    for part in (data[:cut], data[cut:]):
        e = Engine("plane3", delta)
        e.upload(part)
        parts.append(e.score(sampler=SAMPLE_PARAMS, params=p_ref, precision=FP64, want_counts=True)["counts"].astype(np.int64))
        e.close()
    assert np.array_equal(parts[0] + parts[1], c_ref.astype(np.int64))


def test_plane_10m_x_1m_fp32_winner_is_independent_of_the_request_split(port, plane10m):
    """configs[1] as benchmarked: 10 M points x 1 M Philox hypotheses in fp32 (10^13 evaluations).  The winner of one
    request equals the better of two half requests (ties to the smaller index, RANSAC.hxx:100), its fp32 count is within
    the rounding band of the oracle's fp64 count, and its consensus mask / refit match the oracle."""
    data, true = plane10m
    m, delta = MODELS["plane3"], synth.DELTAS["plane3"]
    eng = Engine("plane3", delta)
    eng.upload(data)
    whole = eng.score(count=N_HYPS, seed=7, precision=FP32)
    lo = eng.score(count=N_HYPS // 2, first=0, seed=7, precision=FP32)
    hi = eng.score(count=N_HYPS - N_HYPS // 2, first=N_HYPS // 2, seed=7, precision=FP32)
    best = lo if (lo["best_count"], -lo["best_index"]) >= (hi["best_count"], -hi["best_index"]) else hi
    assert whole["n_valid"] == lo["n_valid"] + hi["n_valid"]
    assert (whole["best_count"], whole["best_index"]) == (best["best_count"], best["best_index"])
    assert np.array_equal(whole["best_subset"], best["best_subset"]) and np.array_equal(whole["best_params"], best["best_params"])
    # the winning hypothesis is what the oracle computes from the winning subset
    want = port.estimate(m, delta, data[whole["best_subset"]])
    assert np.array_equal(whole["best_params"], want)
    # fp32 count vs the oracle's fp64 count of the same hypothesis
    cnt64, mask64 = port.agree(m, delta, want, data)
    res = np.abs((data - want[3:]) @ want[:3])
    band = _fp32_band("plane3", data, want, delta)     # measured band (tests/test_parity_gpu.py), 5e-4 here
    assert abs(int(whole["best_count"]) - int(cnt64)) <= int(np.sum(np.abs(res - delta) <= band))
    assert cnt64 > 0.45 * N_POINTS   # 60 % inliers with sigma 0.4 against delta 0.5: the true plane collects ~47 %
    # consensus set and refit (fp64 path)
    assert eng.consensus(want) == cnt64
    assert np.array_equal(eng.get_mask(), mask64)
    prm = eng.refine()
    assert same_up_to_sign(prm, port.least_squares(m, delta, data[mask64.astype(bool)]), SIGN_IDX["plane3"], REFINE_TOL)
    assert abs(abs(np.dot(prm[:3], true[:3])) - 1.0) < 1e-8
    eng.close()


def test_plane_10m_compute_is_self_consistent(port, plane10m):
    """RANSAC<T,S>::compute on 10 M points: fraction = popcount(mask) / N, the mask is the oracle's agree() set of some
    hypothesis whose refit gives the returned parameters."""
    data, true = plane10m
    m, delta = MODELS["plane3"], synth.DELTAS["plane3"]
    eng = Engine("plane3", delta)
    eng.upload(data)
    for precision in (FP64, FP32):
        out = eng.ransac(0.999, precision=precision, seed=3)
        prm, mask, frac = out["params"], out["mask"], out["fraction"]
        assert len(prm) == 6 and int(mask.sum()) == round(frac * N_POINTS) and frac > 0.45
        tol = 1e-6 if precision == FP64 else 1e-4
        assert same_up_to_sign(prm, port.least_squares(m, delta, data[mask.astype(bool)]), SIGN_IDX["plane3"], tol)
        assert abs(abs(np.dot(prm[:3], true[:3])) - 1.0) < 1e-7
    eng.close()


def test_sphere_10m_counts_and_levenberg_marquardt_refit(port):
    """configs[2]: 10 M points, 4-point minimal solver, geometric (Levenberg-Marquardt) refit of ~4.7 M inliers."""
    data, true = synth.GENERATORS["sphere3"](N_POINTS)
    m, delta = MODELS["sphere3"], synth.DELTAS["sphere3"]
    subs = synth.random_subsets(N_POINTS, 4, 32, seed=2027)
    c_ref, p_ref = port.score_subsets(m, delta, data, subs)
    eng = Engine("sphere3", delta, ls_type=1)
    eng.upload(data)
    r = eng.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP64, want_counts=True, want_params=True)
    assert np.array_equal(r["counts"], c_ref) and np.array_equal(np.nan_to_num(r["params"]), np.nan_to_num(p_ref))
    r32 = eng.score(sampler=SAMPLE_PARAMS, params=p_ref, precision=FP32, want_counts=True)
    d = np.abs(r32["counts"].astype(np.int64) - c_ref.astype(np.int64))
    assert d.sum() <= 1e-3 * c_ref.sum() + 64
    cnt, mask = port.agree(m, delta, true, data)
    assert eng.consensus(true) == cnt and np.array_equal(eng.get_mask(), mask)
    prm = eng.refine()
    want = port.least_squares(m, delta, data[mask.astype(bool)], 1)
    assert same_up_to_sign(prm, want, [], REFINE_TOL), (prm, want)
    assert np.abs(prm - true).max() < 0.05
    eng.close()


def test_absolute_orientation_1m_pairs(port):
    """configs[3]: 1 M 3D-3D correspondences, 30 % gross outliers; triad hypotheses, Horn refit."""
    n = 1_000_000
    data, true = synth.GENERATORS["absor"](n)
    m, delta = MODELS["absor"], synth.DELTAS["absor"]
    subs = synth.random_subsets(n, 3, 256, seed=2028)
    c_ref, p_ref = port.score_subsets(m, delta, data, subs)
    eng = Engine("absor", delta)
    eng.upload(data)
    r = eng.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP64, want_counts=True, want_params=True)
    assert np.array_equal(r["counts"], c_ref) and np.array_equal(np.nan_to_num(r["params"]), np.nan_to_num(p_ref))
    b = int(np.argmax(c_ref))
    cnt, mask = port.agree(m, delta, p_ref[b], data)
    assert eng.consensus(p_ref[b]) == cnt and np.array_equal(eng.get_mask(), mask)
    assert same_up_to_sign(eng.refine(), port.least_squares(m, delta, data[mask.astype(bool)]), SIGN_IDX["absor"], REFINE_TOL)
    out = eng.ransac(0.999, precision=FP32, seed=5)
    prm, cmask, frac = out["params"], out["mask"], out["fraction"]
    assert frac > 0.4 and int(cmask.sum()) == round(frac * n)   # 70 % inliers, sigma 1 per coordinate against delta 2: ~52 % at best
    assert same_up_to_sign(prm, true, SIGN_IDX["absor"], 1e-2)
    eng.close()


@pytest.mark.parametrize("name", ["line2d", "plane3"])
def test_65536_small_problems_in_one_batch(port, name):
    """configs[4]: 65 536 independent problems of 256 points, one thread block each.  Deterministic for a seed; for a
    sample of problems popcount(mask) = count and the oracle's refit of the mask reproduces the parameters."""
    m, delta = MODELS[name], synth.DELTAS[name]
    nprob, npts = 65_536, 256
    D = synth.GENERATORS[name](8, seed=1)[0].shape[1]
    rng = np.random.default_rng(17)
    bases = [synth.GENERATORS[name](npts, seed=300 + i)[0] for i in range(64)]
    data = np.empty((nprob * npts, D))
    for i in range(nprob):
        data[i * npts:(i + 1) * npts] = bases[i % 64] + rng.uniform(-50, 50, D)
    offsets = (np.arange(nprob + 1) * npts).astype(np.uint64)
    eng = Engine(name, delta, ls_type=1)
    out = eng.ransac_batch(data, offsets, exhaustive=False, prob=0.999, max_tries=2048, seed=11, want_masks=True)
    again = eng.ransac_batch(data, offsets, exhaustive=False, prob=0.999, max_tries=2048, seed=11, want_masks=True)
    assert np.array_equal(out["counts"], again["counts"]) and np.array_equal(out["masks"], again["masks"])
    assert np.array_equal(np.nan_to_num(out["params"]), np.nan_to_num(again["params"]))
    assert np.array_equal(out["masks"].reshape(nprob, npts).sum(axis=1), out["counts"])
    assert out["counts"].min() >= 0.3 * npts and out["counts"].mean() >= 0.4 * npts   # 60-70 % inliers generated, sigma 0.4 against delta 0.5
    for i in rng.choice(nprob, 48, replace=False):
        chunk = data[i * npts:(i + 1) * npts]
        mask = out["masks"][i * npts:(i + 1) * npts].astype(bool)
        assert same_up_to_sign(out["params"][i], port.least_squares(m, delta, chunk[mask]), SIGN_IDX[name], REFINE_TOL)
    eng.close()
