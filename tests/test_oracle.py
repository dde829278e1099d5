"""Pins the CPU oracle (oracle/lsqr_oracle.c, the plain-C restatement) before anything trusts it:
against the reference's own golden values, against fixtures minted by the reference itself
(tests/golden/make_golden.py), and against the reference live -- or, without oracle/_ref, what it returned for the same inputs.
No GPU involved."""
import functools
import hashlib

import numpy as np
import pytest

from conftest import SIGN_IDX, golden, ls_types, pinv_tol, same_up_to_sign
from lsqrrecipes_b200 import synth
from oracle.pyoracle import INFO, MODELS

ALL = list(MODELS.items())


# ---- the reference's own literal test vectors -------------------------------------------
def test_circle_agree_literals(port):
    """testing/SphereParametersEstimatorTest.cxx:280-296: circle r=2 at the origin, delta=0.5."""
    prm = [0.0, 0.0, 2.0]
    cases = [((0.0, 0.0), False), ((1.75, 0.0), True), ((2.25, 0.0), True), ((4.0, 0.0), False)]
    for pt, want in cases:
        cnt, out = port.agree(MODELS["circle2"], 0.5, prm, np.array([pt]))
        assert bool(out[0]) == want


def test_pivot_known_answers(port):
    """testing/PivotCalibrationParametersEstimatorTest.cxx:47-48,72,75-78,82-83,102 on
    testing/Data/pivotCalibrationData.txt (frames stored in the fixture)."""
    g = golden("pivot_file")
    frames = g["frames"]
    n = len(frames)
    assert n == 481
    mini = frames[[0, int(n / 2.0), n - 1]]
    exact = port.estimate(MODELS["pivot"], 1.0, mini)
    assert len(exact) == 6 and np.all(np.abs(exact - g["known_exact"]) < 1.0)
    cnt, out = port.agree(MODELS["pivot"], 1.0, exact, mini)
    assert cnt == 3
    ls = port.least_squares(MODELS["pivot"], 1.0, frames)
    assert len(ls) == 6 and np.all(np.abs(ls - g["known_ls"]) < 1.0)
    # and to full precision against what the reference itself computed
    assert np.allclose(exact, g["exact"], rtol=0, atol=1e-9)
    assert np.allclose(ls, g["ls"], rtol=0, atol=1e-9)


def test_dense_file_known_answer(port):
    """testing/DenseLinearEquationSystemParametersEstimatorTest.cxx:153-213 on testing/Data/augmentedMatrix.txt
    (rows stored in the fixture): least squares within 0.5 of the 17-digit solution."""
    g = golden("dense_file")
    assert g["rows"].shape == (1443, 7)
    ls = port.least_squares(MODELS["dense6"], 0.5, g["rows"])
    assert len(ls) == 6 and np.all(np.abs(ls - g["known_ls"]) < 0.5)
    assert np.allclose(ls, g["ls"], rtol=1e-9, atol=1e-9)


# ---- fixtures minted by the reference ---------------------------------------------------
@pytest.mark.parametrize("name,m", ALL)
def test_port_matches_reference_fixture(port, name, m):
    g = golden(name)
    counts, params = port.score_subsets(m, float(g["delta"]), g["data"], g["subsets"])
    assert np.array_equal(counts, g["counts"]), "per-hypothesis inlier counts must be bit-exact"
    assert np.array_equal(np.isnan(params), np.isnan(g["params"])), "same degenerate subsets"
    if pinv_tol(name):  # 9x6 / n x n pseudo-inverse goes through the SVD stand-in: rounding-level agreement
        assert np.allclose(np.nan_to_num(params), np.nan_to_num(g["params"]), rtol=pinv_tol(name), atol=pinv_tol(name))
    else:
        assert np.array_equal(np.nan_to_num(params), np.nan_to_num(g["params"])), "estimate() must be bit-exact"


@pytest.mark.parametrize("name,m", ALL)
def test_port_exhaustive_and_lsq_fixture(port, name, m):
    g = golden(name)
    for ls_type in ls_types(name):
        # Levenberg-Marquardt results: both sides run MINPACK's lmder (oracle/minpack_lm.h) on the reference's scalar residuals;
        # the cross-wire valley is flat (hundreds of evaluations), so its end point is compared at the north star's 1e-6
        tol = 1e-6 if (name == "usxw" and ls_type == 1) else 1e-8
        prm, mask, frac, cnt, rank = port.ransac_exhaustive(m, float(g["delta"]), g["small"], ls_type=ls_type)
        assert np.array_equal(mask, g[f"ex_mask_ls{ls_type}"])
        assert frac == float(g[f"ex_fraction_ls{ls_type}"])
        assert same_up_to_sign(prm, g[f"ex_params_ls{ls_type}"], SIGN_IDX[name], tol)
        b = int(np.argmax(g["counts"]))
        _, bm = port.agree(m, float(g["delta"]), g["params"][b], g["data"])
        ls = port.least_squares(m, float(g["delta"]), g["data"][bm.astype(bool)], ls_type)
        assert same_up_to_sign(ls, g[f"lsq_ls{ls_type}"], SIGN_IDX[name], tol)


def test_config1_plane23(port):
    """BASELINE.json configs[0] restated (SURVEY.md 8d 1a): 23 points, all C(23,3)=1771 subsets."""
    g = golden("config1_plane23")
    prm, mask, frac, cnt, rank = port.ransac_exhaustive(0, 0.5, g["data"])
    assert np.array_equal(mask, g["mask"]) and frac == float(g["fraction"])
    assert rank == int(np.argmax(g["all_counts"])) and cnt == g["all_counts"].max()
    assert same_up_to_sign(prm, g["params"], [0, 1, 2], 1e-9)
    for r in (0, 1, 17, 1014, 1770):
        sub = port.unrank_lex(r, 23, 3)
        c, p = port.score_subsets(0, 0.5, g["data"], sub[None, :])
        assert c[0] == g["all_counts"][r] and np.array_equal(p[0], g["all_params"][r])


# ---- the reference live, or what it returned -------------------------------------------
# With oracle/_ref present these tests compare the restatement with the reference on every row.  Without it they compare with
# tests/golden/reference_cases.npz (tests/golden/make_golden.py): the same inputs, the reference's counts and rejection
# pattern in full, its parameter vectors as a SHA-256 where the comparison is bit-exact and as a fixed sample of rows where it
# has a tolerance.
def _digest(p):
    """SHA-256 of a parameter matrix as array_equal(nan_to_num(.)) sees it (NaN -> 0, -0.0 -> 0.0)."""
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(np.nan_to_num(p) + 0.0).tobytes()).digest(), dtype=np.uint8)


def reduce_answer(counts, params, exact, rows=None, keep=None):
    """What a comparison needs of the reference's answer.  rows: candidate rows for the value comparison (default all);
    keep=None keeps every candidate (live), keep=K a fixed sample of K of them and, where exact, the digest instead (stored)."""
    out = {"counts": counts.astype(np.uint32), "nan": np.isnan(params)}
    if keep is not None and exact:
        out["sha"] = _digest(params)
        return out
    idx = np.flatnonzero(np.ones(len(params), bool) if rows is None else rows)
    if keep is not None and len(idx) > keep:
        idx = np.sort(np.random.default_rng(0).choice(idx, keep, replace=False))
    out["idx"], out["rows"] = idx, params[idx]
    return out


def assert_params(p1, want, tol):
    if "sha" in want:
        assert np.array_equal(_digest(p1), want["sha"])
    elif tol is None:
        assert np.array_equal(np.nan_to_num(p1[want["idx"]]), np.nan_to_num(want["rows"]))
    else:
        assert np.allclose(np.nan_to_num(p1[want["idx"]]), np.nan_to_num(want["rows"]), rtol=tol, atol=tol)


def reference_answer(ref, prefix, live):
    """live(ref) when oracle/_ref is present, else the stored entries <prefix>.*"""
    if ref is not None:
        return live(ref)
    return {k[len(prefix) + 1:]: v for k, v in stored_cases().items() if k.startswith(prefix + ".")}


@functools.lru_cache(maxsize=1)
def stored_cases():
    """tests/golden/reference_cases.npz unpacked: one byte blob, entry i at offsets[i]:offsets[i + 1] with dtypes[i], shapes[i]."""
    g = golden("reference_cases")
    blob, off = g["blob"], g["offsets"]
    return {str(k): np.frombuffer(blob[off[i]:off[i + 1]].tobytes(), dtype=np.dtype(str(g["dtypes"][i]))).reshape([d for d in g["shapes"][i] if d >= 0])
            for i, k in enumerate(g["names"])}


def live_case(name, m):
    n, k = 400, INFO[m][2]
    data, _ = synth.GENERATORS[name](n, seed=4242 + m)
    return data, synth.DELTAS[name], synth.random_subsets(n, k, 1500, seed=99 + m)


def reference_live(orc, name, m, keep=None):
    data, delta, subs = live_case(name, m)
    c, p = orc.score_subsets(m, delta, data, subs)
    return reduce_answer(c, p, pinv_tol(name) is None, keep=keep)


@pytest.mark.parametrize("name,m", ALL)
def test_port_matches_reference_live(port, ref, name, m):
    want = reference_answer(ref, f"live.{name}", lambda r: reference_live(r, name, m))
    data, delta, subs = live_case(name, m)
    c1, p1 = port.score_subsets(m, delta, data, subs)
    assert np.array_equal(c1, want["counts"])
    assert np.array_equal(np.isnan(p1), want["nan"])
    assert_params(p1, want, pinv_tol(name))


def horn_case():
    data, _ = synth.absolute_orientation(500, seed=77, outlier_frac=0.0)
    return data, np.random.default_rng(5).uniform(0.1, 3.0, 500)


def test_weighted_horn_port_matches_reference(port, ref):
    """AbsoluteOrientationParametersEstimator::weightedLeastSquaresEstimate (.cxx:208-297): restatement vs the
    reference itself; unit weights reproduce the unweighted Horn solve; zero weights remove pairs."""
    data, w = horn_case()
    b = reference_answer(ref, "horn", lambda r: {"params": r.weighted_absor(data, w)})["params"]
    a = port.weighted_absor(data, w)
    assert len(a) == 7 and same_up_to_sign(a, b, SIGN_IDX["absor"], 1e-10)
    assert same_up_to_sign(port.weighted_absor(data, np.ones(500)), port.least_squares(MODELS["absor"], 2.0, data), SIGN_IDX["absor"], 1e-9)
    bad = data.copy()
    bad[::5, 3:] += 500.0
    w0 = np.ones(500)
    w0[::5] = 0.0
    assert same_up_to_sign(port.weighted_absor(bad, w0), port.least_squares(MODELS["absor"], 2.0, data[w0 > 0]), SIGN_IDX["absor"], 1e-9)
    assert len(port.weighted_absor(data[:2], np.ones(2))) == 0


def test_ragged_and_empty_inputs(port):
    """Edge cases the reference guards: too few data, degenerate subsets, empty consensus."""
    m = MODELS["plane3"]
    assert len(port.estimate(m, 0.5, np.zeros((2, 3)))) == 0                       # fewer than k points
    assert len(port.estimate(m, 0.5, np.array([[0, 0, 0], [1, 1, 1], [2, 2, 2.]]))) == 0  # collinear
    prm, mask, frac, cnt, _ = port.ransac_exhaustive(m, 0.5, np.zeros((2, 3)))
    assert len(prm) == 0 and frac == 0.0
    # coincident points: every subset degenerate -> no model
    prm, mask, frac, cnt, _ = port.ransac_exhaustive(m, 0.5, np.ones((6, 3)))
    assert len(prm) == 0 and frac == 0.0 and cnt == 0
    # line: points closer than delta are rejected (LineParametersEstimator.hxx:33-35)
    assert len(port.estimate(MODELS["line3"], 0.5, np.array([[0, 0, 0], [0.1, 0, 0.]]))) == 0
    # sphere: coplanar points
    assert len(port.estimate(MODELS["sphere3"], 0.5, np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.]]))) == 0
    # rays: parallel, and intersection behind an origin
    par = np.array([[0, 0, 0, 1, 0, 0], [0, 1, 0, 1, 0, 0.]])
    assert len(port.estimate(MODELS["ray"], 0.5, par)) == 0
    behind = np.array([[0, 0, 0, 1, 0, 0], [-5, 1, 0, 0, 1, 0.]])
    assert len(port.estimate(MODELS["ray"], 0.5, behind)) == 0


def test_choose_unrank_and_stop_rule(port):
    from math import comb
    assert port.choose(23, 3) == 1771 and port.choose(100, 3) == comb(100, 3)
    assert port.choose(10_000_000, 3) == 0xFFFFFFFF                 # saturates, RANSAC.hxx:272-276
    seen = [tuple(port.unrank_lex(r, 7, 3)) for r in range(comb(7, 3))]
    import itertools
    assert seen == list(itertools.combinations(range(7), 3))        # order of RANSAC.hxx:197-213
    # log(1-0.999)/log(1-0.6^3) = 28.4 -> 28
    assert port.num_tries(0.999, 60, 100, 3, 161700) == 28
    assert port.num_tries(0.999, 100, 100, 3, 161700) == 0


def reference_model_table(orc):
    """(D, P, k) of every model id and of the first unknown id (-1s for None)."""
    return {"info": np.array([orc.model_info(m) or (-1, -1, -1) for m in range(35)])}


def test_model_tables_agree_everywhere(port, ref):
    """One id space: the Python tables of the oracle and of the engine binding, the C restatement and the reference harness
    describe every model with the same (doubles per datum, parameters, minimal subset)."""
    from lsqrrecipes_b200 import api
    table = reference_answer(ref, "models", reference_model_table)["info"]
    assert MODELS == api.MODELS and len(MODELS) == 34
    for name, m in MODELS.items():
        assert INFO[m] == api.MODEL_INFO[m] == port.model_info(m) == tuple(int(x) for x in table[m]), name
    assert port.model_info(34) is None and tuple(table[34]) == (-1, -1, -1) and port.model_info(-1) is None


def degenerate_case(name, m):
    data = synth.degenerate_pool(name, seed=31 + m)
    return data, synth.DELTAS[name], synth.random_subsets(len(data), INFO[m][2], 600, seed=7 + m)


def reference_degenerate(orc, name, m, keep=None):
    """Values are compared (pinv_tol models) for the hypotheses that explain more than their own subset; for the dense
    systems only where the n x n system is well conditioned; for the calibration systems not at all (rejection pattern only)."""
    data, delta, subs = degenerate_case(name, m)
    k = INFO[m][2]
    c, p = orc.score_subsets(m, delta, data, subs)
    if pinv_tol(name) is None:
        return reduce_answer(c, p, True, keep=keep)
    ok = ~np.isnan(p[:, 0]) & (c > k)
    if name.startswith("dense"):
        ok &= np.array([np.linalg.cond(data[s][:, :k]) < 1e6 for s in subs])
    if name in ("usxw", "uscp"):
        ok[:] = False
    return reduce_answer(c, p, False, rows=ok, keep=keep)


@pytest.mark.parametrize("name,m", ALL)
def test_port_matches_reference_on_degenerate_subsets(port, ref, name, m):
    """Minimal subsets with repeated, collinear, scaled and all-zero records: the restatement rejects exactly the subsets the
    reference rejects (empty parameter vector, RANSAC.hxx:87-88) and agrees on the rest."""
    want = reference_answer(ref, f"degenerate.{name}", lambda r: reference_degenerate(r, name, m))
    data, delta, subs = degenerate_case(name, m)
    c1, p1 = port.score_subsets(m, delta, data, subs)
    bad1, bad2 = np.isnan(p1[:, 0]), want["nan"][:, 0]
    assert bad2.any() and not bad2.all(), "the pool must mix degenerate and valid subsets"
    assert np.array_equal(bad1, bad2), "same subsets rejected"
    if pinv_tol(name):
        # the reference's absolute rank test (singular values <= 2.2e-16) accepts numerically singular systems, whose "solution" is
        # amplified rounding noise in either SVD: values are compared for the rows reference_degenerate selects
        if name not in ("usxw", "uscp"):
            assert len(want["idx"])
            assert_params(p1, want, 1e-6)
    else:
        assert_params(p1, want, None)
        assert np.array_equal(c1, want["counts"])


def seed_cases(seed):
    """(name, m, data, delta, subsets) of every model on fresh data with a threshold drawn per seed."""
    rng = np.random.default_rng(1000 + seed)
    for name, m in ALL:
        k, n = INFO[m][2], 160
        data, _ = synth.GENERATORS[name](n, seed=5000 + 37 * seed + m)
        delta = synth.DELTAS[name] * float(rng.choice([0.25, 1.0, 3.0]))
        yield name, m, data, delta, synth.random_subsets(n, k, 120, seed=seed + m)


def reference_seed_case(orc, name, m, data, delta, subs, keep=None):
    """The answer to the listed subsets, agree() of the best one (count and mask) and the algebraic least squares over it."""
    c, p = orc.score_subsets(m, delta, data, subs)
    out = reduce_answer(c, p, pinv_tol(name) is None, keep=keep)
    b = int(np.argmax(c))
    cnt, mask = orc.agree(m, delta, p[b], data)
    inl = data[mask.astype(bool)]
    ls = orc.least_squares(m, delta, inl, 0) if (len(inl) >= max(INFO[m][2], 4) and name != "usxw") else np.zeros(0)
    out.update(best_params=p[b], best_agree=np.array([cnt]), mask=mask.astype(bool), ls0=ls)
    return out


@pytest.mark.parametrize("seed", range(4))
def test_port_matches_reference_across_seeds_and_thresholds(port, ref, seed):
    """Every model on fresh data with a threshold drawn per seed (tight thresholds put many data near the decision boundary):
    counts bit-exact, estimate() bit-exact where the reference's arithmetic is plain double, least squares over the best
    consensus set within 1e-8 (1e-6 for the cross-wire valley)."""
    for name, m, data, delta, subs in seed_cases(seed):
        want = reference_answer(ref, f"seed{seed}.{name}", lambda r: reference_seed_case(r, name, m, data, delta, subs))
        c1, p1 = port.score_subsets(m, delta, data, subs)
        c2 = want["counts"]
        assert np.array_equal(np.isnan(p1), want["nan"]), name
        assert_params(p1, want, pinv_tol(name))
        if pinv_tol(name) is None:
            assert np.array_equal(c1, c2), name
        else:
            # counts of the pseudo-inverse models: identical on identical parameter vectors
            b = int(np.argmax(c2))
            assert port.agree(m, delta, want["best_params"], data)[0] == want["best_agree"][0] == c2[b], name
        if len(want["ls0"]):
            inl = data[want["mask"]]
            assert same_up_to_sign(port.least_squares(m, delta, inl, 0), want["ls0"], SIGN_IDX[name], 1e-8), name
