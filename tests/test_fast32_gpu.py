"""The fp32 kernels count for count against the restatement of oracle/fast32.py: every step of the fast mode is deterministic
IEEE arithmetic, so each per-hypothesis fp32 count is predicted exactly -- the single-problem kernels (consensus32_kernel
with one and with several hypotheses per thread, the constant-bank kernel) and the batched rounds (batch_kernel,
batch_cluster_kernel), on odd sizes, data off the origin, data on the threshold and records that are not finite."""
import numpy as np
import pytest

from conftest import SIGN_IDX, same_up_to_sign
from lsqrrecipes_b200 import FP32, FP64, SAMPLE_LIST, SAMPLE_PARAMS, SAMPLE_PHILOX, Engine, synth
from oracle import fast32
from oracle.pyoracle import INFO, MODELS
from test_fast32_cpu import _non_finite_records

pytestmark = pytest.mark.gpu

NAMES = fast32.NAMES
BATCH_NAMES = [n for n in NAMES if n not in ("usxw", "uscp")]
CLUSTER_CASES = [("plane3", 1), ("line2d", 1), ("line3", 1), ("sphere3", 0), ("sphere3", 1), ("absor", 1), ("ray", 1), ("pivot", 1),
                 ("plane8", 1), ("dense8", 1)]


def _shifted(name, data, by):
    """data moved off the origin along the centred components (a dense system's rows are not positions)"""
    data = np.array(data, dtype=np.float64)
    pos = [d for d in range(data.shape[1]) if fast32.centred(name, d)]
    if pos:
        data[:, pos] += by
    return data


def _restated(name, data, params, delta, rows):
    return fast32.counts(name, params[rows], data, delta, centre="single")


@pytest.mark.parametrize("name", NAMES)
def test_single_path_counts_equal_the_restatement(port, name):
    m = MODELS[name]
    k = INFO[m][2]
    delta = synth.DELTAS[name]
    n = 7001                                   # odd: the last tile and sub-chunk are ragged
    data = _shifted(name, synth.GENERATORS[name](n, seed=5100 + m)[0], 317.0)
    eng = Engine(name, delta)
    eng.upload(data)
    rng = np.random.default_rng(m)
    # SAMPLE_LIST, 512 hypotheses: consensus32_kernel with one hypothesis per thread
    subs = synth.random_subsets(n, k, 512, seed=52 + m)
    r = eng.score(sampler=SAMPLE_LIST, subsets=subs, precision=FP32, want_counts=True, want_params=True)
    assert np.array_equal(r["counts"], _restated(name, data, r["params"], delta, np.arange(512)))
    # 9000 Philox hypotheses: several per thread; every hypothesis slot of a thread among the 1024 compared
    r = eng.score(count=9000, seed=7, precision=FP32, want_counts=True, want_params=True)
    rows = np.unique(np.concatenate([rng.choice(9000, 1024, replace=False), [r["best_index"]]]))
    assert np.array_equal(r["counts"][rows], _restated(name, data, r["params"], delta, rows))
    # >= 98 304 hypotheses with counts: the constant-bank kernel, full pass
    H = 98304 + 1536 + 7
    c = eng.score(count=H, seed=11, precision=FP32, want_counts=True, want_params=True)
    p = c["params"]
    rows = np.unique(np.concatenate([rng.choice(H, 512, replace=False), [c["best_index"]], np.arange(H - 40, H)]))
    assert np.array_equal(c["counts"][rows], _restated(name, data, p, delta, rows))
    assert c["best_count"] == c["counts"].max() and c["counts"][c["best_index"]] == c["best_count"]
    eng.close()


def _bisect(name, q, c, dl, d2, inside, outside):
    """the last record on either side of the restatement's flip along the segment inside -> outside (adjacent doubles of t)"""
    def dec(t):
        x = inside + t * (outside - inside)
        return bool(fast32.decisions(name, q, fast32.copy32(name, x[None, :], c), dl, d2, False)[0]), x
    lo, hi = 0.0, 1.0
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        if mid in (lo, hi):
            break
        if dec(mid)[0]:
            lo = mid
        else:
            hi = mid
    return dec(lo)[1], dec(hi)[1]


def _sphere_rows(name, prm, delta):
    """hypersphere rows in every branch of hoist_sphere: r > delta, r = delta, r < delta, r = 0, r < -delta"""
    _, dim = fast32.family(name)
    rows = []
    for r in (2.0 * delta, delta, 0.6 * delta, 0.0, -2.0 * abs(delta) - 1.0):
        p = prm.copy()
        p[dim] = r
        rows.append(p)
    return rows


@pytest.mark.parametrize("name", NAMES)
def test_boundary_data_counts_equal_the_restatement(port, name):
    """Records bisected onto the fp32 threshold of a few hypotheses, records that are not finite, hypersphere rows in every
    branch of the hoist, NaN rows, and thresholds whose fp32 rounding matters (0.1, 1/3) or that admit nothing (0, < 0)."""
    m = MODELS[name]
    k = INFO[m][2]
    fam, _ = fast32.family(name)
    base = _shifted(name, synth.GENERATORS[name](fast32.CENTER_SAMPLE, seed=5300 + m)[0], -61.0)   # fixes the centre
    c = fast32.center_single(name, base)
    _, p64 = port.score_subsets(m, synth.DELTAS[name], base, synth.random_subsets(len(base), k, 64, seed=53 + m))
    hyps = p64[~np.isnan(p64[:, 0])][:4]
    deltas = [synth.DELTAS[name], 0.1, 1.0 / 3.0, 0.0] + ([-0.5] if fam in ("sphere", "dense") or name == "pivot" else [])
    for delta in deltas:
        dl = fast32.cfg_delta(name, delta)
        extra = []
        if dl > 0:
            for prm in hyps:
                q = fast32.hoist(name, prm, c, dl)
                dec = fast32.decisions(name, q, fast32.copy32(name, base, c), dl, delta * delta, False)
                ins, outs = np.flatnonzero(dec)[:3], np.flatnonzero(~dec)[:3]
                for i, o in zip(ins, outs):
                    extra.extend(_bisect(name, q, c, dl, delta * delta, base[i], base[o]))
        extra.extend(_non_finite_records(name, base[:8]))
        data = np.concatenate([base, np.array(extra)])
        rows = [h for h in hyps]
        if fam == "sphere":
            rows += _sphere_rows(name, hyps[0], delta)
        nan_row = np.full(len(hyps[0]), np.nan)
        late_nan = hyps[0].copy()
        late_nan[-1] = np.nan
        rows += [nan_row, late_nan]
        params = np.array(rows)
        eng = Engine(name, delta)
        eng.upload(data)
        got = eng.score(sampler=SAMPLE_PARAMS, params=params, precision=FP32, want_counts=True)["counts"]
        eng.close()
        want = fast32.counts(name, params, data, delta, centre="single")
        assert np.array_equal(got, want), (delta, got, want)
        if not dl > 0:
            assert not got.any()


# ---- batched fp32, replayed exactly -----------------------------------------------------------------------
SEED, PROB, TRIES = 20261022, 0.999, 256


def _problems(name, k):
    """sizes k, k + 1 and odd ones, each problem shifted by 40 i; the last one's first record is a far outlier, which sets
    the fp32 centre of that problem"""
    sizes = [k, k + 1, 37, 151, 200, 97]
    out = []
    for i, s in enumerate(sizes):
        d = synth.GENERATORS[name](max(s, k + 1), seed=5500 + 7 * i)[0][:s]
        out.append(_shifted(name, d, 40.0 * i))
    far = synth.GENERATORS[name](121, seed=5599)[0]
    far = _shifted(name, far, 13.0)
    far[0] = _shifted(name, far[:1], 1e5)[0]
    out.append(far)
    return out


def _expect(port, single, name, delta, ls_type, data, gb):
    """(count, mask, params or None, conclusive) of the batched fp32 result for one problem, from the restatement and the replay"""
    m = MODELS[name]
    k = INFO[m][2]
    n = len(data)
    if n < k:
        return 0, np.zeros(n, np.uint8), None, True
    single.upload(data)
    p = single.score(count=TRIES, sampler=SAMPLE_PHILOX, precision=FP64, seed=SEED, first=gb << 32, want_params=True)["params"]
    valid = ~np.isnan(p).any(axis=1)
    c32 = np.zeros(len(p), dtype=np.int64)
    c32[valid] = fast32.counts(name, p[valid], data, delta, centre="batch")
    h, c, conclusive = fast32.replay(c32, valid, n, k, PROB, TRIES)
    if c == 0:
        return 0, np.zeros(n, np.uint8), None, conclusive
    cnt, mask = port.agree(m, delta, p[h], data)
    want = port.least_squares(m, delta, data[mask.astype(bool)], ls_type)
    return cnt, mask, want, conclusive


def _compare(port, single, name, delta, ls_type, out, offsets, problems, first):
    inconclusive = 0
    for i, data in enumerate(problems):
        gb = first + i
        cnt, mask, want, conclusive = _expect(port, single, name, delta, ls_type, data, gb)
        if not conclusive:
            inconclusive += 1
            continue
        lo, hi = int(offsets[gb]), int(offsets[gb + 1])
        assert out["counts"][gb] == cnt, (name, i, out["counts"][gb], cnt)
        assert np.array_equal(out["masks"][lo:hi], mask), (name, i)
        if want is None or not len(want):
            assert np.isnan(out["params"][gb]).all(), (name, i)
        else:
            assert same_up_to_sign(out["params"][gb], want, SIGN_IDX[name], 1e-6), (name, i, out["params"][gb], want)
    return inconclusive


@pytest.mark.parametrize("name", BATCH_NAMES)
def test_batched_fp32_rounds_replay_exactly(port, name):
    m = MODELS[name]
    k = INFO[m][2]
    delta = synth.DELTAS[name]
    first = 3                                  # a non-zero global problem index
    problems = [synth.GENERATORS[name](1, seed=5)[0][:1]] * first + _problems(name, k)
    sizes = [len(p) for p in problems]
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    eng = Engine(name, delta, ls_type=1)
    out = eng.ransac_batch(np.concatenate(problems), offsets, prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True, precision=FP32)
    eng.close()
    single = Engine(name, delta)
    inconclusive = _compare(port, single, name, delta, 1, out, offsets, problems[first:], first)
    single.close()
    assert inconclusive <= 1, inconclusive


@pytest.mark.parametrize("name,ls_type", CLUSTER_CASES)
def test_cluster_fp32_rounds_replay_exactly(port, name, ls_type):
    m = MODELS[name]
    delta = synth.DELTAS[name]
    eng = Engine(name, delta, ls_type=ls_type)
    one, most = eng.batch_capacity(FP32)
    sizes = [one + 3 if (one + 3) % 2 else one + 4, 3 * one + 1 if (3 * one + 1) % 2 else 3 * one]   # clusters of 2 and of 4
    sizes = [min(s, most) for s in sizes]
    first = 2
    problems = [synth.GENERATORS[name](1, seed=5)[0][:1]] * first
    for i, s in enumerate(sizes):
        d = _shifted(name, synth.GENERATORS[name](s, seed=5700 + i)[0][:s], 40.0 * (i + 1))
        if i == 1:
            d[0] = _shifted(name, d[:1], 1e5)[0]
        problems.append(d)
    offsets = np.concatenate([[0], np.cumsum([len(p) for p in problems])]).astype(np.uint64)
    out = eng.ransac_batch(np.concatenate(problems), offsets, prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True, precision=FP32)
    eng.close()
    single = Engine(name, delta)
    inconclusive = _compare(port, single, name, delta, ls_type, out, offsets, problems[first:], first)
    single.close()
    if inconclusive:
        pytest.skip(f"inconclusive: the stop rule of {inconclusive} problem(s) lies within a few ulps of an integer")
