"""Parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle on the
same seeded inputs and the same ordered subset lists, and against the committed golden fixtures
minted by the reference.  Bars (BASELINE.json north_star):
  * fp64 validation mode: per-hypothesis inlier counts, the chosen best subset and the consensus
    mask are BIT-EXACT; estimate() parameters bit-exact where the reference's arithmetic is plain
    double (all models but pivot, whose 9x6 pseudo-inverse goes through an SVD stand-in);
  * fp32 fast mode: per-point decisions may differ only within the fp32 rounding band of the
    threshold (stated below), refined parameters within 1e-4 relative;
  * refined parameters: 1e-6 relative (fp64), modulo the sign of eigenvector-derived entries.
"""
import numpy as np
import pytest

from conftest import SIGN_IDX, golden, is_sphere, lm_case_is_clear, ls_types, model_family, pinv_tol, same_up_to_sign
from lsqrrecipes_b200 import FP32, FP64, SAMPLE_EXHAUSTIVE, SAMPLE_LIST, SAMPLE_PARAMS, Engine, synth
from oracle.fast32 import fp32_band as _fp32_band
from oracle.fast32 import residual64 as _residual64
from oracle.pyoracle import INFO, MODELS

pytestmark = pytest.mark.gpu
from lsqrrecipes_b200 import MODELS as ENGINE_MODELS

ALL = [(n, m) for n, m in MODELS.items() if n in ENGINE_MODELS]   # every estimator the engine implements
REFINE_TOL = 1e-6




@pytest.mark.parametrize("name,m", ALL)
def test_fp64_counts_bit_exact_vs_reference_fixture(name, m):
    """Subset list from the fixture -> device minimal solve + fp64 consensus == what the reference returned."""
    g = golden(name)
    eng = Engine(name, float(g["delta"]))
    eng.upload(g["data"])
    r = eng.score(sampler=SAMPLE_LIST, subsets=g["subsets"], precision=FP64, want_counts=True, want_params=True)
    assert np.array_equal(r["counts"], g["counts"])
    assert np.array_equal(np.isnan(r["params"]), np.isnan(g["params"]))
    if pinv_tol(name):
        assert np.allclose(np.nan_to_num(r["params"]), np.nan_to_num(g["params"]), rtol=pinv_tol(name), atol=pinv_tol(name))
    else:
        assert np.array_equal(np.nan_to_num(r["params"]), np.nan_to_num(g["params"])), "device estimate() must round like the reference"
    b = int(np.argmax(g["counts"]))  # first maximum: strict '>' of RANSAC.hxx:245
    assert r["best_index"] == b and r["best_count"] == g["counts"][b]
    assert np.array_equal(r["best_subset"], g["subsets"][b])
    eng.close()


@pytest.mark.parametrize("name,m", ALL)
def test_fp64_counts_bit_exact_vs_oracle_large(port, name, m):
    """Same, at a size where tiles, chunks and atomics are all exercised, against the oracle."""
    D, P, k = INFO[m]
    n, H = 20011, 3000
    data, _ = synth.GENERATORS[name](n, seed=777 + m)
    delta = synth.DELTAS[name]
    subs = synth.random_subsets(n, k, H, seed=31 + m)
    c_ref, p_ref = port.score_subsets(m, delta, data, subs)
    eng = Engine(name, delta)
    eng.upload(data)
    r = eng.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP64, want_counts=True, want_params=True)
    assert np.array_equal(r["counts"], c_ref)
    # agree() alone, on the oracle's own hypotheses (covers pivot bit-exactly as well)
    r2 = eng.score(sampler=SAMPLE_PARAMS, params=p_ref, precision=FP64, want_counts=True)
    assert np.array_equal(r2["counts"], c_ref)
    assert r2["best_index"] == int(np.argmax(c_ref))
    eng.close()


@pytest.mark.parametrize("name,m", ALL)
def test_degenerate_subsets_are_rejected_like_the_oracle(port, name, m):
    """Minimal subsets with repeated, collinear, scaled and all-zero records (synth.degenerate_pool; the oracle is pinned to the
    reference on the same pools in tests/test_oracle.py): the device solvers reject exactly the subsets the oracle rejects
    (a rejected hypothesis counts as a try and scores nothing, RANSAC.hxx:87-88), agree on the rest, and the arg-max ignores the
    rejected ones."""
    D, P, k = INFO[m]
    data = synth.degenerate_pool(name, seed=31 + m)
    subs = synth.random_subsets(len(data), k, 600, seed=7 + m)
    delta = synth.DELTAS[name]
    c_ref, p_ref = port.score_subsets(m, delta, data, subs)
    eng = Engine(name, delta)
    eng.upload(data)
    r = eng.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP64, want_counts=True, want_params=True)
    bad = np.isnan(p_ref[:, 0])
    assert bad.any() and not bad.all()
    assert np.array_equal(np.isnan(r["params"][:, 0]), bad), "same subsets rejected"
    # (n_valid counts non-empty parameter vectors, as the reference's `parameters.size() > 0` does: the triad solver of the absolute
    # orientation can return a vector whose quaternion is NaN for a numerically collinear triple -- valid, and agreeing with nothing)
    assert r["n_valid"] >= int((~bad).sum()) and (name == "absor" or r["n_valid"] == int((~bad).sum())) and np.all(r["counts"][bad] == 0)
    if pinv_tol(name) is None:
        assert np.array_equal(np.nan_to_num(r["params"]), np.nan_to_num(p_ref)) and np.array_equal(r["counts"], c_ref)
        assert r["best_index"] == int(np.argmax(c_ref))
    # the fp32 fast mode rejects the same subsets (the minimal solve is fp64 in both modes)
    r32 = eng.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP32, want_counts=True)
    assert np.all(r32["counts"][bad] == 0) and r32["n_valid"] == r["n_valid"]
    eng.close()


@pytest.mark.parametrize("name,m", ALL)
def test_exhaustive_compute_vs_reference_fixture(name, m):
    """RANSAC<T,S>::compute, brute-force overload (RANSAC.hxx:150-249), on the fixture's small problem."""
    g = golden(name)
    for ls in ls_types(name):
        eng = Engine(name, float(g["delta"]), ls_type=ls)
        eng.upload(g["small"])
        r = eng.ransac_exhaustive(precision=FP64)
        assert np.array_equal(r["mask"], g[f"ex_mask_ls{ls}"]), "consensus set must be bit-exact"
        assert r["fraction"] == float(g[f"ex_fraction_ls{ls}"])
        tol = REFINE_TOL
        assert same_up_to_sign(r["params"], g[f"ex_params_ls{ls}"], SIGN_IDX[name], tol)
        eng.close()


def test_config1_plane23_exhaustive(port):
    """BASELINE.json configs[0] restated (SURVEY.md 8d 1a)."""
    g = golden("config1_plane23")
    eng = Engine("plane3", 0.5)
    eng.upload(g["data"])
    s = eng.score(count=1771, sampler=SAMPLE_EXHAUSTIVE, precision=FP64, want_counts=True, want_params=True)
    assert np.array_equal(s["counts"], g["all_counts"])
    assert np.array_equal(s["params"], g["all_params"])
    assert s["best_index"] == int(np.argmax(g["all_counts"]))
    r = eng.ransac_exhaustive(precision=FP64)
    assert np.array_equal(r["mask"], g["mask"]) and r["fraction"] == float(g["fraction"])
    assert same_up_to_sign(r["params"], g["params"], [0, 1, 2], REFINE_TOL)
    # the on-device unranking follows the reference's enumeration order
    for rank in (0, 5, 1014, 1770):
        s1 = eng.score(count=1, first=rank, sampler=SAMPLE_EXHAUSTIVE, precision=FP64)
        assert np.array_equal(s1["best_subset"], port.unrank_lex(rank, 23, 3)) or s1["best_count"] == 0
    eng.close()


def test_pivot_file_known_answers():
    """The reference's one file-based known-answer test (PivotCalibrationParametersEstimatorTest.cxx)."""
    g = golden("pivot_file")
    frames = g["frames"]
    n = len(frames)
    eng = Engine("pivot", 1.0)
    exact = eng.estimate(frames[[0, int(n / 2.0), n - 1]])
    assert len(exact) == 6 and np.all(np.abs(exact - g["known_exact"]) < 1.0)
    assert np.allclose(exact, g["exact"], rtol=1e-9, atol=1e-9)
    assert eng.agree(exact, frames[[0, int(n / 2.0), n - 1]]).sum() == 3
    ls = eng.least_squares(frames)
    assert len(ls) == 6 and np.all(np.abs(ls - g["known_ls"]) < 1.0)
    assert np.allclose(ls, g["ls"], rtol=1e-8, atol=1e-8)
    eng.close()


def test_dense_file_known_answer():
    """DenseLinearEquationSystemParametersEstimatorTest.cxx:153-213: least squares over
    testing/Data/augmentedMatrix.txt (1443 rows x 7) against the 17-digit solution, tolerance 0.5 there."""
    g = golden("dense_file")
    eng = Engine("dense6", 0.5)
    ls = eng.least_squares(g["rows"])
    assert np.all(np.abs(ls - g["known_ls"]) < 0.5)          # the reference's own criterion
    assert np.allclose(ls, g["ls"], rtol=1e-9, atol=1e-9)    # and what the reference itself returns
    eng.upload(g["rows"])
    assert eng.consensus(g["known_ls"]) == int(np.sum(np.abs(g["rows"][:, :6] @ g["known_ls"] - g["rows"][:, 6]) < 0.5))
    eng.close()


def test_weighted_horn_vs_oracle(port):
    """lsqr_weighted_least_squares == AbsoluteOrientationParametersEstimator::weightedLeastSquaresEstimate (.cxx:208-297)."""
    data, true = synth.absolute_orientation(20000, seed=91)
    rng = np.random.default_rng(6)
    w = rng.uniform(0.0, 2.0, 20000)
    eng = Engine("absor", 2.0)
    got = eng.weighted_least_squares(data, w)
    assert same_up_to_sign(got, port.weighted_absor(data, w), SIGN_IDX["absor"], REFINE_TOL)
    assert same_up_to_sign(eng.weighted_least_squares(data, np.ones(20000)), eng.least_squares(data), SIGN_IDX["absor"], 1e-9)
    assert len(eng.weighted_least_squares(data[:2], np.ones(2))) == 0
    eng.close()
    from lsqrrecipes_b200 import AbsoluteOrientationParametersEstimator
    est = AbsoluteOrientationParametersEstimator(2.0)
    prm = []
    est.weightedLeastSquaresEstimate(data, w, prm)
    assert same_up_to_sign(prm, port.weighted_absor(data, w), SIGN_IDX["absor"], REFINE_TOL)


def test_direct_least_squares_ignore_the_shard():
    """lsqr_least_squares / lsqr_weighted_least_squares fit all the data they are given on one device: on rank 0 of 2 (caller
    hooks, lsqr_set_shard) they return exactly what an unsharded context returns and never call the all-reduce hooks."""
    calls = []

    def max_fn(user, dev, stream):
        calls.append("max")
        return 0

    def sum_fn(user, dev, count, stream):
        calls.append("sum")
        return 0

    w = np.random.default_rng(8).uniform(0.0, 2.0, 20000)
    for name in ("plane3", "sphere3", "absor"):   # sphere3: the geometric fit's Levenberg-Marquardt passes reduce too
        data, _ = synth.GENERATORS[name](20000, seed=17)
        one, sharded = Engine(name, synth.DELTAS[name]), Engine(name, synth.DELTAS[name])
        sharded.set_shard(0, 2, max_fn, sum_fn)
        want = one.least_squares(data)
        assert len(want) and np.array_equal(sharded.least_squares(data), want), name
        if name == "absor":
            want = one.weighted_least_squares(data, w)
            assert len(want) and np.array_equal(sharded.weighted_least_squares(data, w), want)
        one.close()
        sharded.close()
    assert calls == []


def test_crosswire_operator_interface(port):
    """SingleUnknownPointTargetUSCalibrationParametersEstimator through the Python mirror of the reference API:
    estimate() wants exactly four data (.cxx:21-22), ANALYTIC / ITERATIVE least squares, RANSAC::compute."""
    from lsqrrecipes_b200 import RANSAC, SingleUnknownPointTargetUSCalibrationParametersEstimator as Est
    m = MODELS["usxw"]
    for attempt in range(12):      # a case whose iterative fit ends well inside the reference's evaluation cap (conftest.lm_case_is_clear)
        data, true = synth.crosswire(400, seed=12 + attempt)
        cnt, flags = port.agree(m, 1.0, true, data)
        port.least_squares(m, 1.0, data[flags.astype(bool)], 1)
        if lm_case_is_clear(port, "usxw", 1):
            break
    est = Est(1.0)
    p4, p5 = [], [1.0]
    est.estimate(data[:4], p4)
    est.estimate(data[:5], p5)
    assert len(p4) == 20 and p5 == []
    assert np.allclose(p4, port.estimate(m, 1.0, data[:4]), rtol=1e-6, atol=1e-6)
    cnt, flags = port.agree(m, 1.0, true, data)
    inl = data[flags.astype(bool)]
    for ls_type in (Est.ANALYTIC, Est.ITERATIVE):
        est.setLeastSquaresType(ls_type)
        prm = []
        est.leastSquaresEstimate(inl, prm)
        assert same_up_to_sign(prm, port.least_squares(m, 1.0, inl, ls_type), [], REFINE_TOL)
    assert est.agree(list(true), data[flags.astype(bool)][0]) and not est.agree(list(true), data[~flags.astype(bool)][0])
    prm, cs = [], []
    est.setLeastSquaresType(Est.ANALYTIC)   # (compute() with the iterative refit: test_randomized_compute_end_to_end)
    frac = RANSAC.compute(prm, est, data, 0.999, cs)
    assert frac > 0.6 and len(prm) == 20 and sum(cs) == round(frac * len(data))
    assert np.abs(np.array(prm[:6]) - true[:6]).max() < 0.5 and abs(prm[9] - 0.143) < 1e-3 and abs(prm[10] - 0.139) < 1e-3


def test_hypersphere_4d_as_the_reference_tests_it(port):
    """testing/SphereParametersEstimatorTest.cxx:379-428 (testnD<4>, "covers all the code for dimensionality greater than
    3"): 50 points on a random 4-D sphere, coordinates up to 1000, unit noise; the minimal estimate from clean data and
    both least-squares fits must land within 3 sigma of the known [c, r]."""
    from lsqrrecipes_b200 import SphereParametersEstimator as Est
    rng = np.random.default_rng(404)
    c, r = rng.uniform(-1000, 1000, 4), rng.uniform(0, 1000)
    u = rng.uniform(-1, 1, (50, 4))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    clean = c + r * u
    noisy = clean + rng.normal(0, 1.0, (50, 4))
    true = np.append(c, r)
    est = Est(0.5, dimension=4)
    prm = []
    est.estimate(clean[:5], prm)
    assert len(prm) == 5 and np.abs(np.array(prm) - true).max() < 3.0
    assert np.allclose(prm, port.estimate(MODELS["sphere4"], 0.5, clean[:5]), rtol=1e-9, atol=1e-7)
    for ls_type in (Est.ALGEBRAIC, Est.GEOMETRIC):
        est.setLeastSquaresType(ls_type)
        prm = []
        est.leastSquaresEstimate(noisy, prm)
        assert len(prm) == 5 and np.abs(np.array(prm) - true).max() < 3.0
        assert np.allclose(prm, port.least_squares(MODELS["sphere4"], 0.5, noisy, ls_type), rtol=REFINE_TOL, atol=REFINE_TOL)
    # five points in a hyperplane: rank < 4, no sphere (SphereParametersEstimator.hxx:190-191)
    flat = clean[:5].copy()
    flat[:, 3] = 7.0
    prm = [1.0]
    est.estimate(flat, prm)
    assert prm == []


def test_hyperplane_4d_operator_interface(port):
    """PlaneParametersEstimator<4> goes through the null-space branch (PlaneParametersEstimator.hxx:70-108) that the
    reference's own test leaves to "any dimension" (testing/PlaneParametersEstimatorTest.cxx:37): same checks as its
    3-D test -- exact estimate from k points, least squares on noisy inliers, agree(), and RANSAC::compute."""
    from lsqrrecipes_b200 import RANSAC, PlaneParametersEstimator as Est
    data, true = synth.plane(5000, seed=31, dim=4)
    m = MODELS["plane4"]
    est = Est(0.5, dimension=4)
    prm = []
    est.estimate(data[:4], prm)
    assert len(prm) == 8 and same_up_to_sign(prm, port.estimate(m, 0.5, data[:4]), SIGN_IDX["plane4"], 1e-9)
    assert abs(np.linalg.norm(prm[:4]) - 1.0) < 1e-12 and prm[4:] == data[0].tolist()
    assert np.abs((data[:4] - np.array(prm[4:])) @ np.array(prm[:4])).max() < 1e-9    # the four points lie on it
    dup = data[[0, 1, 2, 2]]                                                         # linearly dependent rows: rank 3
    prm = [1.0]
    est.estimate(dup, prm)
    assert prm == []
    cnt, flags = port.agree(m, 0.5, true, data)
    inl = data[flags.astype(bool)]
    prm = []
    est.leastSquaresEstimate(inl, prm)
    assert same_up_to_sign(prm, port.least_squares(m, 0.5, inl), SIGN_IDX["plane4"], REFINE_TOL)
    assert est.agree(list(true), inl[0]) and not est.agree(list(true), data[~flags.astype(bool)][0])
    out, cs = [], []
    frac = RANSAC.compute(out, est, data, 0.999, cs)
    assert frac > 0.9 * cnt / len(data) and sum(cs) == round(frac * len(data))
    n_est, n_true = np.array(out[:4]), true[:4]
    assert abs(abs(n_est @ n_true) - 1.0) < 1e-6 and abs((np.array(out[4:]) - true[4:]) @ n_true) < 0.1


def test_sign_of_delta_is_immaterial_where_the_reference_squares_it(port):
    """PlaneParametersEstimator.hxx:16 stores delta*delta, so -0.5 and 0.5 are the same estimator (also in fp32 fast mode, whose
    kernels compare an unsquared residual); SphereParametersEstimator.hxx:20 keeps delta itself: a negative one admits nothing."""
    data, _ = synth.plane(20011, seed=3)
    subs = synth.random_subsets(len(data), 3, 256, seed=4)
    want, _ = port.score_subsets(MODELS["plane3"], -0.5, data, subs)
    assert np.array_equal(want, port.score_subsets(MODELS["plane3"], 0.5, data, subs)[0])
    pos, neg = Engine("plane3", 0.5), Engine("plane3", -0.5)
    for eng in (pos, neg):
        eng.upload(data)
    for precision in (FP64, FP32):
        a = pos.score(sampler=SAMPLE_LIST, subsets=subs, precision=precision, want_counts=True)["counts"]
        b = neg.score(sampler=SAMPLE_LIST, subsets=subs, precision=precision, want_counts=True)["counts"]
        assert np.array_equal(a, b)
        if precision == FP64:
            assert np.array_equal(a, want)
    pos.close(); neg.close()
    # delta = 0 admits nothing (|s| < 0), in both fp32 kernels and in fp64
    zero = Engine("plane3", 0.0)
    zero.upload(data)
    assert zero.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP32, want_counts=True)["counts"].max() == 0
    assert zero.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP64, want_counts=True)["counts"].max() == 0
    assert zero.score(count=98304 + 64, seed=1, precision=FP32)["best_count"] == 0
    zero.close()
    sdata, strue = synth.sphere(5000, 3, seed=5)
    eng = Engine("sphere3", -0.5)
    eng.upload(sdata)
    for precision in (FP64, FP32):
        assert eng.score(sampler=SAMPLE_PARAMS, params=strue[None, :], precision=precision, want_counts=True)["counts"][0] == 0
    eng.close()


def test_circle_agree_literals():
    """testing/SphereParametersEstimatorTest.cxx:280-296"""
    eng = Engine("circle2", 0.5)
    out = eng.agree([0.0, 0.0, 2.0], np.array([[0, 0], [1.75, 0], [2.25, 0], [4, 0.]]))
    assert out.tolist() == [0, 1, 1, 0]
    eng.close()


@pytest.mark.parametrize("name,m", ALL)
def test_consensus_mask_and_refine_vs_oracle(port, name, m):
    D, P, k = INFO[m]
    delta = synth.DELTAS[name]
    for ls in ls_types(name):
        for attempt in range(12):
            n = 301 if (name == "usxw" and ls == 1) else 50021     # see conftest.lm_case_is_clear
            data, _ = synth.GENERATORS[name](n, seed=1234 + m + 1000 * attempt)
            subs = synth.random_subsets(n, k, 64, seed=5 + m)
            c_ref, p_ref = port.score_subsets(m, delta, data, subs)
            b = int(np.argmax(c_ref))
            cnt_ref, mask_ref = port.agree(m, delta, p_ref[b], data)
            want = port.least_squares(m, delta, data[mask_ref.astype(bool)], ls)
            if lm_case_is_clear(port, name, ls):
                break
        else:
            raise AssertionError("no clear Levenberg-Marquardt case found")
        eng = Engine(name, delta, ls_type=ls)
        eng.upload(data)
        cnt = eng.consensus(p_ref[b])
        assert cnt == cnt_ref
        assert np.array_equal(eng.get_mask(), mask_ref), "agree() mask must be bit-exact in fp64"
        prm = eng.refine()
        assert same_up_to_sign(prm, want, SIGN_IDX[name], REFINE_TOL), (prm, want)
        if is_sphere(name) and ls == 1:
            # same MINPACK run: the number of function evaluations is the oracle's (a stopping test that sits on its threshold may
            # fire one evaluation earlier or later: the moments are summed in a different order)
            assert abs(eng.last_refine_stats()["lm_iterations"] - port.last_lm()[1]) <= 1
        # leastSquaresEstimate() called directly on the inliers gives the same answer
        direct = eng.least_squares(data[mask_ref.astype(bool)])
        assert same_up_to_sign(direct, want, SIGN_IDX[name], REFINE_TOL)
        eng.close()


@pytest.mark.parametrize("name,m", ALL)
def test_fp32_fast_mode_differs_only_near_threshold(port, name, m):
    D, P, k = INFO[m]
    n, H = 30011, 512
    data, _ = synth.GENERATORS[name](n, seed=900 + m)
    delta = synth.DELTAS[name]
    subs = synth.random_subsets(n, k, H, seed=77 + m)
    c64, p64 = port.score_subsets(m, delta, data, subs)
    eng = Engine(name, delta)
    eng.upload(data)
    r = eng.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP32, want_counts=True)
    c32 = r["counts"].astype(np.int64)
    diff = np.abs(c32 - c64.astype(np.int64))
    # every count difference must be explained by points inside the rounding band of the threshold
    worst = np.argsort(-diff)[:8]
    for h in worst:
        if np.isnan(p64[h, 0]):
            assert c32[h] == 0
            continue
        res, thr = _residual64(name, p64[h], data, delta)
        band = _fp32_band(name, data, p64[h], delta)
        near = int(np.sum(np.abs(res - thr) <= band))
        assert diff[h] <= near, (name, h, diff[h], near)
    assert diff.sum() <= 1e-3 * c64.sum() + 16
    eng.close()


@pytest.mark.parametrize("name,m", ALL)
def test_fp32_constant_bank_kernel_matches_shared_memory_kernel(name, m):
    """Requests of >= 98304 hypotheses take the constant-bank kernel (k_fast.cu), smaller ones the
    shared-memory kernel.  Both evaluate the same fp32 expressions, so one large request and the same
    hypotheses scored in small pieces must give identical counts; the data size is chosen so that the
    last constant-bank launch is partial and the last sub-chunk ragged."""
    n, H, piece = 7001, 100352, 25088
    data, _ = synth.GENERATORS[name](n, seed=4100 + m)
    eng = Engine(name, synth.DELTAS[name])
    eng.upload(data)
    whole = eng.score(count=H, seed=9, precision=FP32, want_counts=True)
    parts = [eng.score(count=piece, first=f, seed=9, precision=FP32, want_counts=True) for f in range(0, H, piece)]
    c_parts = np.concatenate([p["counts"] for p in parts])
    assert np.array_equal(whole["counts"], c_parts)
    b = int(np.argmax(c_parts))
    assert whole["best_index"] == b and whole["best_count"] == c_parts[b]
    # and the fp32 counts stay within a whisker of the bit-exact fp64 ones
    c64 = eng.score(count=4096, seed=9, precision=FP64, want_counts=True)["counts"].astype(np.int64)
    assert np.abs(whole["counts"][:4096].astype(np.int64) - c64).sum() <= 1e-3 * c64.sum() + 16
    eng.close()


@pytest.mark.parametrize("name,m", ALL)
@pytest.mark.parametrize("precision", [FP64, FP32])
def test_randomized_compute_end_to_end(port, name, m, precision):
    """RANSAC<T,S>::compute(parameters, estimator, data, 0.999, &consensusSet): the result must be the
    least-squares fit of a consensus set that the oracle reproduces from the chosen hypothesis."""
    D, P, k = INFO[m]
    delta = synth.DELTAS[name]
    for attempt in range(12):
        n = 300 if name == "usxw" else 20000     # see conftest.lm_case_is_clear
        data, true = synth.GENERATORS[name](n, seed=2024 + m + 1000 * attempt)
        eng = Engine(name, delta)
        eng.upload(data)
        r = eng.ransac(0.999, precision=precision, seed=11)
        mask = r["mask"].astype(bool)
        want = port.least_squares(m, delta, data[mask], 1)
        if lm_case_is_clear(port, name, 1):
            break
        eng.close()
    else:
        raise AssertionError("no clear Levenberg-Marquardt case found")
    assert r["fraction"] > 0.3 and r["tries"] >= 1
    assert mask.sum() == r["best_count"] and abs(r["fraction"] - mask.sum() / n) < 1e-15
    assert same_up_to_sign(r["params"], want, SIGN_IDX[name], REFINE_TOL if precision == FP64 else 1e-4)
    # and the refined model explains the generating model's inliers
    cnt, _ = port.agree(m, delta, r["params"], data)
    assert cnt >= 0.9 * mask.sum()
    eng.close()


def test_philox_sampler_is_partition_independent():
    """Hypothesis h depends only on (seed, h): scoring [0,H) in one request or in pieces gives the same counts."""
    data, _ = synth.plane(5000, seed=3)
    eng = Engine("plane3", 0.5)
    eng.upload(data)
    whole = eng.score(count=4096, seed=5, precision=FP64, want_counts=True)
    parts = [eng.score(count=1024, first=f, seed=5, precision=FP64, want_counts=True)["counts"] for f in (0, 1024, 2048, 3072)]
    assert np.array_equal(whole["counts"], np.concatenate(parts))
    assert whole["n_valid"] == 4096
    other = eng.score(count=4096, seed=6, precision=FP64, want_counts=True)
    assert not np.array_equal(whole["counts"], other["counts"])
    # subsets are distinct, in range
    s = eng.score(count=1, first=123, seed=5, precision=FP64)
    assert len(set(s["best_subset"].tolist())) == 3 and s["best_subset"].min() >= 0 and s["best_subset"].max() < 5000
    eng.close()


def test_edge_cases_match_reference_conventions():
    eng = Engine("plane3", 0.5)
    # fewer data than the minimal subset (RANSAC.hxx:16-19 / :168-169)
    eng.upload(np.zeros((2, 3)))
    r = eng.ransac(0.99)
    assert r["fraction"] == 0.0 and len(r["params"]) == 0
    r = eng.ransac_exhaustive()
    assert r["fraction"] == 0.0 and len(r["params"]) == 0
    # all subsets degenerate -> empty parameters, return 0
    eng.upload(np.ones((8, 3)))
    r = eng.ransac_exhaustive()
    assert r["fraction"] == 0.0 and len(r["params"]) == 0 and r["best_count"] == 0
    # probability outside (0,1)
    data, _ = synth.plane(100, seed=1)
    eng.upload(data)
    assert eng.ransac(1.0)["fraction"] == 0.0 and eng.ransac(0.0)["fraction"] == 0.0
    # all inliers: terminates on the first perfect hypothesis (RANSAC.hxx:104-105)
    flat = np.random.default_rng(0).uniform(-10, 10, (1000, 3))
    flat[:, 2] = 0.0
    eng.upload(flat)
    r = eng.ransac(0.99, precision=FP64)
    assert r["fraction"] == 1.0 and r["best_count"] == 1000
    # estimate(): degenerate -> empty
    assert len(eng.estimate(np.array([[0, 0, 0], [1, 1, 1], [2, 2, 2.]]))) == 0
    eng.close()


@pytest.mark.parametrize("name", ["line2d", "plane3", "plane4", "sphere3", "sphere4", "dense5", "plane2", "line5", "dense3"])
def test_batched_small_problems_vs_oracle(port, name):
    """BASELINE.json configs[4]: many independent small problems, one thread block each.  Exhaustive mode is
    bit-comparable with the reference's brute-force driver run per problem."""
    m = MODELS[name]
    D, P, k = INFO[m]
    delta = synth.DELTAS[name]
    nprob = 24
    sizes = [20 + (7 * i) % 13 for i in range(nprob)]
    sizes[3] = 1   # ragged: fewer points than the minimal subset
    sizes[5] = k
    chunks = [synth.GENERATORS[name](max(s, k + 1), seed=50 + i)[0][:s] for i, s in enumerate(sizes)]
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    eng = Engine(name, delta, ls_type=1)
    out = eng.ransac_batch(np.concatenate(chunks), offsets, exhaustive=True, want_masks=True)
    for i, ch in enumerate(chunks):
        prm, mask, frac, cnt, rank = port.ransac_exhaustive(m, delta, ch, ls_type=1)
        assert out["counts"][i] == cnt
        got_mask = out["masks"][int(offsets[i]):int(offsets[i + 1])]
        assert np.array_equal(got_mask, mask)
        if len(prm) == 0:
            assert np.isnan(out["params"][i]).all()
        else:
            assert same_up_to_sign(out["params"][i], prm, SIGN_IDX[name], REFINE_TOL)
    # randomized mode: consensus at least as large as the generating inlier set minus noise tail
    out2 = eng.ransac_batch(np.concatenate(chunks), offsets, exhaustive=False, prob=0.999, max_tries=4096, seed=9)
    ok = [i for i, s in enumerate(sizes) if s > 2 * k]
    # (five noisy points pin a 4-D sphere loosely, so the stopping rule of RANSAC.hxx:121-126 ends further from the optimum)
    assert np.mean(out2["counts"][ok] >= (0.7 if name == "sphere4" else 0.8) * out["counts"][ok]) > 0.9
    eng.close()


@pytest.mark.parametrize("name", ["line2d", "plane3", "sphere3", "line3", "absor", "dense5", "plane6", "sphere5"])
def test_batched_small_problems_fp32_scoring(port, name):
    """Randomized batched mode with fp32 scoring (what the large-problem path does): the fast forms choose the hypothesis, everything
    returned is fp64 -- the consensus set is agree() of the winner in reference arithmetic, the count is its size, the parameters
    its least-squares fit -- and the consensus reached is what fp64 scoring reaches (same sampler, same stop rule)."""
    m = MODELS[name]
    D, P, k = INFO[m]
    delta = synth.DELTAS[name]
    nprob = 48
    sizes = [150 + (37 * i) % 107 for i in range(nprob)]      # odd and even sizes: the fp32 copy is padded to a pair
    sizes[3] = 1
    sizes[5] = k
    chunks = [synth.GENERATORS[name](max(s, k + 1), seed=700 + i)[0][:s] + (0.0 if name.startswith("dense") else 40.0 * i) for i, s in enumerate(sizes)]
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    data = np.concatenate(chunks)
    eng = Engine(name, delta, ls_type=1)
    o32 = eng.ransac_batch(data, offsets, prob=0.999, max_tries=2048, seed=5, want_masks=True, precision=FP32)
    again = eng.ransac_batch(data, offsets, prob=0.999, max_tries=2048, seed=5, want_masks=True, precision=FP32)
    o64 = eng.ransac_batch(data, offsets, prob=0.999, max_tries=2048, seed=5, want_masks=True, precision=FP64)
    eng.close()
    assert np.array_equal(o32["counts"], again["counts"]) and np.array_equal(o32["masks"], again["masks"])
    assert np.array_equal(np.nan_to_num(o32["params"]), np.nan_to_num(again["params"]))
    for i, ch in enumerate(chunks):
        mask = o32["masks"][int(offsets[i]):int(offsets[i + 1])].astype(bool)
        assert mask.sum() == o32["counts"][i], "the count is the fp64 size of the returned consensus set"
        if sizes[i] < k or o32["counts"][i] == 0:
            assert np.isnan(o32["params"][i]).all() or o32["counts"][i] >= k
            continue
        want = port.least_squares(m, delta, ch[mask], 1)
        if len(want) == 0:
            assert np.isnan(o32["params"][i]).all()
        else:
            assert same_up_to_sign(o32["params"][i], want, SIGN_IDX[name], REFINE_TOL), (i, o32["params"][i], want)
    big = [i for i, s in enumerate(sizes) if s > 4 * k]
    # same hypotheses, same stop rule: the two precisions agree on the winner except where fp32 rounding reorders near-ties
    close = np.abs(o32["counts"][big].astype(np.int64) - o64["counts"][big].astype(np.int64)) <= np.maximum(2, 0.02 * o64["counts"][big])
    assert close.mean() > 0.9, (o32["counts"][big], o64["counts"][big])


def test_batched_problems_cross_copy_pieces_and_launches(port):
    """lsqr_ransac_batch uploads in pieces (4 MB from pageable memory) and launches per ~32 MB of problems: 100 000 copies of one
    16-point problem (38 MB) in exhaustive mode must all return the oracle's answer for that problem, whichever piece and launch
    they travelled in; the same from page-locked memory (16 MB pieces)."""
    import torch
    per, nprob = 16, 100_000
    one, _ = synth.GENERATORS["plane3"](per, seed=9)
    prm, mask, frac, cnt, rank = port.ransac_exhaustive(MODELS["plane3"], 0.5, one, ls_type=1)
    data = np.tile(one, (nprob, 1))
    offsets = (np.arange(nprob + 1) * per).astype(np.uint64)
    eng = Engine("plane3", 0.5)
    for src in (data, torch.from_numpy(data).pin_memory().numpy()):
        out = eng.ransac_batch(src, offsets, exhaustive=True, want_masks=True)
        assert np.all(out["counts"] == cnt)
        assert np.array_equal(out["masks"].reshape(nprob, per), np.tile(mask, (nprob, 1)))
        assert np.all(np.abs(out["params"] - out["params"][0]) == 0) and same_up_to_sign(out["params"][0], prm, SIGN_IDX["plane3"], REFINE_TOL)
    eng.close()


def test_python_operator_interface_mirrors_reference():
    """Reads like examples/planeEstimation.cxx:112-118."""
    from lsqrrecipes_b200 import PlaneParametersEstimator, RANSAC
    data, true = synth.plane(1000, outlier_frac=0.1, seed=8)
    est = PlaneParametersEstimator(0.5)
    params, consensus = [], []
    frac = RANSAC.compute(params, est, data.tolist(), 0.999, consensus)
    assert len(params) == 6 and len(consensus) == 1000 and abs(frac - sum(consensus) / 1000) < 1e-12
    assert abs(abs(np.dot(params[:3], true[:3])) - 1) < 1e-3
    assert est.agree(params, data[consensus.index(True)])
    ls = []
    est.leastSquaresEstimate(data[np.array(consensus)], ls)
    assert same_up_to_sign(ls, params, [0, 1, 2], 1e-9)


@pytest.mark.parametrize("name", ["plane3", "line2d", "sphere3", "absor", "pivot", "uscp"])
@pytest.mark.parametrize("precision", [FP64, FP32])
def test_pipelined_compute_equals_upload_then_ransac(name, precision):
    """lsqr_compute (data still on the host: first-round subsets drawn by the host copy of the Philox sampler, their records
    fetched ahead, every chunk scored as it lands) returns exactly what lsqr_upload + lsqr_ransac return: same winner, same
    number of tries, same consensus set, same parameters -- from pageable and from page-locked memory, for sizes below one
    chunk and spanning many."""
    import torch
    for n in (5, 1000, 70_001, 1_200_003):
        data, _ = synth.GENERATORS[name](n, seed=77 + n % 1000)
        a = Engine(name, synth.DELTAS[name])
        a.upload(data)
        want = a.ransac(0.999, precision=precision, seed=21)
        a.close()
        b = Engine(name, synth.DELTAS[name])
        pinned = torch.from_numpy(data).pin_memory()
        for src in (data, pinned.numpy()):
            got = b.compute(src, 0.999, precision=precision, seed=21)
            assert (got["best_index"], got["best_count"], got["tries"], got["fraction"]) == (want["best_index"], want["best_count"], want["tries"], want["fraction"])
            assert np.array_equal(got["mask"], want["mask"]) and np.array_equal(got["params"], want["params"])
        # the data stay resident: the estimator-level calls that follow compute() see them
        assert b.consensus(want["params"]) > 0 or len(want["params"]) == 0
        b.close()
    # invalid input: nothing happens (RANSAC.hxx:16-19)
    e = Engine(name, synth.DELTAS[name])
    r = e.compute(data[:1], 0.999)
    assert r["fraction"] == 0.0 and len(r["params"]) == 0
    assert e.compute(data, 1.0)["fraction"] == 0.0
    e.close()
