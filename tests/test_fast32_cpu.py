"""The fp32 restatement (oracle/fast32.py) on its own, and the fp32 contract of include/lsqr_b200.h checked through it for all 34
estimators: a datum decided differently from the reference's agree() must lie within the fp32 rounding band of the threshold,
and a record with a non-finite component is an outlier of every hypothesis.  tests/test_fast32_gpu.py pins the kernels to
the restatement count for count."""
from fractions import Fraction

import numpy as np
import pytest

from lsqrrecipes_b200 import synth
from oracle import fast32
from oracle.pyoracle import INFO, MODELS

F32 = np.float32


def _round_f32(a, b, c):
    """a * b + c rounded once to fp32, from exact rationals (round to nearest, ties to even; IEEE zero signs)"""
    fa, fb, fc = (float(v) for v in (a, b, c))
    v = Fraction(fa) * Fraction(fb) + Fraction(fc)
    if v == 0:
        neg_prod = (np.signbit(a) != np.signbit(b))
        return F32(-0.0) if (neg_prod and np.signbit(c)) else F32(0.0)
    sign, v = (-1 if v < 0 else 1), abs(v)
    e = v.numerator.bit_length() - v.denominator.bit_length()
    if Fraction(2) ** e > v:
        e -= 1
    e = max(e, -126)
    q = Fraction(2) ** (e - 23)
    m = v / q
    fl = m.numerator // m.denominator
    rem = m - fl
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and fl % 2 == 1):
        fl += 1
    r = fl * q
    if r >= Fraction(2) ** 128:
        return F32(sign * np.inf)
    return F32(sign * float(r))


def _same_bits(x, y):
    return np.asarray(x, F32).view(np.uint32) == np.asarray(y, F32).view(np.uint32)


def test_fma_is_correctly_rounded():
    rng = np.random.default_rng(1)
    n = 100_000
    a = (rng.uniform(-2, 2, n) * 2.0 ** rng.integers(-30, 30, n)).astype(F32)
    b = (rng.uniform(-2, 2, n) * 2.0 ** rng.integers(-30, 30, n)).astype(F32)
    c = (rng.uniform(-2, 2, n) * 2.0 ** rng.integers(-60, 60, n)).astype(F32)
    # a third with c close to -a*b: massive cancellation
    k = n // 3
    c[:k] = (-(a[:k].astype(np.float64) * b[:k]) * (1 + rng.normal(0, 1e-6, k))).astype(F32)
    got = fast32.fma32(a, b, c)
    want = np.array([_round_f32(x, y, z) for x, y, z in zip(a, b, c)], dtype=F32)
    assert np.all(_same_bits(got, want))


def _tie_cases():
    """a * b exactly on an fp32 midpoint, c a small term that decides the side (the case float32(a*b + c) double-rounds)"""
    out = []
    one_ulp = 2.0 ** -23
    for a_ in (1.0 + one_ulp, 1.5 + one_ulp, 3.0 + 5 * one_ulp):
        for b_ in (1.0 + 2 ** -12, 1.0 + 3 * 2 ** -12):
            p = a_ * b_
            for c_ in (2.0 ** -60, -2.0 ** -60, 2.0 ** -40, -2.0 ** -40, 0.0, -0.0):
                out.append((a_, b_, c_))
    return out


@pytest.mark.parametrize("a,b,c", _tie_cases() + [
    (1.0, 1.0, -1.0),                         # exact cancellation: +0
    (-0.0, 1.0, -0.0),                        # -0
    (2.0 ** -75, 2.0 ** -75, 0.0),            # subnormal result
    (2.0 ** -75, 3.0 * 2.0 ** -76, 2.0 ** -149),
    (1.5 * 2.0 ** -126, 0.5, -2.0 ** -149),
    (2.0 ** -100, 2.0 ** -100, 0.0),          # underflow to 0
    (2.0 ** 100, 2.0 ** 28, 0.0),             # overflow to inf
    (float(np.finfo(F32).max), 1.0, float(np.finfo(F32).max) * 2.0 ** -24),      # exactly the overflow threshold
    (float(np.finfo(F32).max), 1.0, float(np.finfo(F32).max) * 2.0 ** -24 * (1 - 2.0 ** -23)),
    (-float(np.finfo(F32).max), 2.0, float(np.finfo(F32).max)),
])
def test_fma_built_cases(a, b, c):
    a, b, c = F32(a), F32(b), F32(c)
    assert _same_bits(fast32.fma32(a, b, c), _round_f32(a, b, c))


@pytest.mark.parametrize("a,b,c", [(np.inf, 0.0, 1.0), (np.inf, 1.0, -np.inf), (np.nan, 1.0, 1.0), (-np.nan, 1.0, 1.0),
                                   (1.0, 1.0, -np.nan), (np.inf, 2.0, 1.0), (-np.inf, 2.0, 1.0)])
def test_fma_special_operands(a, b, c):
    got = fast32.fma32(F32(a), F32(b), F32(c))
    with np.errstate(invalid="ignore"):
        want = np.float64(a) * np.float64(b) + np.float64(c)
    if np.isnan(want):
        assert got.view(np.uint32) == 0x7FFFFFFF, "NaN results are canonical (a set sign bit would count as an inlier)"
    else:
        assert got == want


def test_nan_results_of_add_and_sub_are_canonical():
    assert fast32.sub32(F32(np.inf), F32(np.inf)).view(np.uint32) == 0x7FFFFFFF
    assert fast32.add32(F32(-np.inf), F32(np.inf)).view(np.uint32) == 0x7FFFFFFF
    assert fast32.mul32(F32(0.0), F32(-np.inf)).view(np.uint32) == 0x7FFFFFFF


def test_center_follows_the_kernel_summation_order():
    """A sum in another order differs in the last bits; at 16 384 records of one magnitude with a few huge ones the fixed
    order is what makes the centre, and with it every fp32 datum, reproducible."""
    rng = np.random.default_rng(3)
    data = rng.uniform(-1000, 1000, (20000, 3))
    data[::997] *= 1e12
    c = fast32.center_single("plane3", data)
    assert np.allclose(c[:3], data[:16384].mean(axis=0), rtol=1e-9, atol=1e-3)
    assert not np.any(c[3:])
    assert not np.any(fast32.center_single("dense5", rng.normal(size=(100, 6))))
    data[5, 1] = np.inf
    assert fast32.center_single("plane3", data)[1] == 0.0, "a non-finite mean leaves the component unshifted"


# ---- the fp32 contract, per datum ------------------------------------------------------------------------
NAMES = fast32.NAMES


def _check(port, name, data, params, delta, centre):
    """every datum whose restated fp32 decision differs from the reference's agree() lies within the fp32 band"""
    m = MODELS[name]
    c = fast32.center_single(name, data) if centre == "single" else fast32.center_batch(name, data)
    x = fast32.copy32(name, data, c)
    dl = fast32.cfg_delta(name, delta)
    checked = 0
    for prm in params:
        if np.isnan(prm[0]):
            continue
        got = fast32.decisions(name, fast32.hoist(name, prm, c, dl), x, dl, delta * delta, centre == "single")
        _, want = port.agree(m, delta, prm, data)
        differ = np.flatnonzero(got != want.astype(bool))
        if len(differ):
            res, thr = fast32.residual64(name, prm, data, delta)
            band = fast32.fp32_band(name, data, prm, delta)
            far = differ[~(np.abs(res[differ] - thr) <= band)]
            assert not len(far), (name, centre, prm, far[:5], res[far[:5]], thr, band, got[far[:5]])
        checked += 1
    return checked


@pytest.mark.parametrize("name", NAMES)
def test_fp32_decisions_stay_in_the_band(port, name):
    m = MODELS[name]
    k = INFO[m][2]
    delta = synth.DELTAS[name]
    data, _ = synth.GENERATORS[name](3001, seed=600 + m)
    if fast32.family(name)[0] != "dense":     # (a shift would change a linear system's solution)
        pos = [d for d in range(data.shape[1]) if fast32.centred(name, d)]
        data[:, pos] += 250.0
    subs = synth.random_subsets(len(data), k, 48, seed=61 + m)
    _, params = port.score_subsets(m, delta, data, subs)
    assert _check(port, name, data, params, delta, "single") >= 24
    assert _check(port, name, data, params, delta, "batch") >= 24


def _non_finite_records(name, data):
    """copies of a datum with one component set to +inf, -inf, NaN or beyond FLT_MAX"""
    recs = []
    for d in range(data.shape[1]):
        for v in (np.inf, -np.inf, np.nan, 1e39, -1e39):
            r = data[d % len(data)].copy()
            r[d] = v
            recs.append(r)
    return np.array(recs)


@pytest.mark.parametrize("name", NAMES)
def test_non_finite_records_are_outliers(port, name):
    """The reference rejects a record with an infinite or NaN component for every hypothesis, and so must fp32; a component
    beyond FLT_MAX is finite in fp64 but not in the fp32 copy, which is outside the fp32 domain: an outlier too."""
    m = MODELS[name]
    k = INFO[m][2]
    delta = synth.DELTAS[name]
    data, _ = synth.GENERATORS[name](400, seed=800 + m)
    _, params = port.score_subsets(m, delta, data, synth.random_subsets(len(data), k, 16, seed=81 + m))
    params = params[~np.isnan(params[:, 0])][:8]
    bad = _non_finite_records(name, data)
    beyond = np.abs(np.nan_to_num(bad, nan=0.0, posinf=0.0, neginf=0.0)).max(axis=1) > 1e38
    for centre in ("single", "batch"):
        c = fast32.center_single(name, data) if centre == "single" else fast32.center_batch(name, data)
        x = fast32.copy32(name, bad, c)
        dl = fast32.cfg_delta(name, delta)
        for prm in params:
            got = fast32.decisions(name, fast32.hoist(name, prm, c, dl), x, dl, delta * delta, centre == "single")
            assert not got.any(), (name, centre, bad[got][:3])
            _, want = port.agree(m, delta, prm, bad[~beyond])
            assert not want.any(), (name, bad[~beyond][want.astype(bool)][:3])


def _sphere_shell(dim, r, delta, n, rng):
    """points at distances spread over [max(0, r - 4 delta), r + 4 delta] from a centre off the origin"""
    ctr = rng.uniform(-2, 2, dim) + 3.0
    u = rng.normal(size=(n, dim))
    u /= np.linalg.norm(u, axis=1)[:, None]
    dist = rng.uniform(max(0.0, r - 4 * delta), r + 4 * delta, n)
    return ctr + u * dist[:, None], np.concatenate([ctr, [r]])


@pytest.mark.parametrize("scale", [1e-4, 1e-2, 1.0, 1e3])
@pytest.mark.parametrize("name", ["circle2", "sphere3", "sphere5"])
@pytest.mark.parametrize("ratio", [0.6, 1.0, 3.0])
def test_hypersphere_decisions_do_not_depend_on_the_scale(port, name, ratio, scale):
    """r < delta, r = delta and r > delta at data scales 1e-4 .. 1e3: every fp32 form but the hypersphere's r < delta one was
    scale-invariant already; that one added an absolute 1 to d^2 and lost its resolution below unit scale."""
    _, dim = fast32.family(name)
    rng = np.random.default_rng(int(ratio * 10) + dim)
    delta = 0.5
    data, prm = _sphere_shell(dim, ratio * delta, delta, 20000, rng)
    data, prm, delta = data * scale, prm * scale, delta * scale
    assert _check(port, name, data, prm[None, :], delta, "single") == 1
    assert _check(port, name, data, prm[None, :], delta, "batch") == 1
    _, want = port.agree(MODELS[name], delta, prm, data)
    assert want.sum() > 1000


@pytest.mark.parametrize("scale", [1e-4, 1e-2, 1.0, 1e3])
@pytest.mark.parametrize("name", ["plane3", "plane2", "plane6"])
def test_hyperplane_decisions_do_not_depend_on_the_scale(port, name, scale):
    m = MODELS[name]
    data, _ = synth.GENERATORS[name](5000, seed=40 + m)
    delta = synth.DELTAS[name] * scale
    data = data * scale
    _, params = port.score_subsets(m, delta, data, synth.random_subsets(len(data), INFO[m][2], 8, seed=4))
    assert _check(port, name, data, params, delta, "single") >= 4


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("delta", [0.0, -0.5, np.nan])
def test_thresholds_that_admit_nothing(port, name, delta):
    """delta = 0 and NaN admit nothing; a negative delta admits nothing where the reference compares an unsquared distance
    (hyperspheres, pivot, dense systems; where it squares delta, -0.5 is 0.5 and the band test covers it)."""
    m = MODELS[name]
    dl = fast32.cfg_delta(name, delta)
    if dl > 0:
        pytest.skip("the reference squares delta")
    data, _ = synth.GENERATORS[name](500, seed=20 + m)
    _, params = port.score_subsets(m, 0.5, data, synth.random_subsets(len(data), INFO[m][2], 8, seed=2))
    params = params[~np.isnan(params[:, 0])]
    for centre in ("single", "batch"):
        c = fast32.center_single(name, data) if centre == "single" else fast32.center_batch(name, data)
        x = fast32.copy32(name, data, c)
        for prm in params:
            assert not port.agree(m, delta, prm, data)[1].any()
            got = fast32.decisions(name, fast32.hoist(name, prm, c, dl), x, dl, delta * delta, centre == "single")
            assert not got.any(), (name, centre, delta, np.flatnonzero(got)[:5])
