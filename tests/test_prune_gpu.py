"""The early exit of fp32 scoring: a request without per-hypothesis counts stops scoring a hypothesis once its inliers so far
plus the data left cannot reach the full count of one already scored.  Every case scores the same request twice, once with
counts (the full pass) and once without, and the winner -- index, count, subset, parameters -- and n_valid must be the same
bit for bit."""
import numpy as np
import pytest

from lsqrrecipes_b200 import FP32, SAMPLE_PARAMS, Engine, synth

pytestmark = pytest.mark.gpu

CB_MIN_HYPS = 98304          # smallest request the constant-bank kernel (and with it the early exit) takes
HYP_BATCH = 1 << 22          # hypotheses per device batch of one request


def both(eng, **kw):
    full = eng.score(precision=FP32, want_counts=True, **kw)
    fast = eng.score(precision=FP32, want_counts=False, **kw)
    return full, fast


def assert_same_winner(full, fast):
    for k in ("best_index", "best_count", "n_valid"):
        assert full[k] == fast[k], (k, full[k], fast[k])
    assert np.array_equal(full["best_subset"], fast["best_subset"])
    assert np.array_equal(full["best_params"].view(np.uint64), fast["best_params"].view(np.uint64))
    c = full["counts"]
    if full["best_count"]:
        assert full["best_index"] == int(np.argmax(c)) and full["best_count"] == int(c.max())


@pytest.mark.parametrize("name", ["plane3", "dense5", "sphere3", "line2d", "line3", "absor"])
def test_every_counting_form(name):
    """plane3 / dense5 (carry chain), sphere3 (per-hypothesis window), line2d (mixed raw count), line3 / absor (sign bit)."""
    n, H = 300_000, 131_072
    data, _ = synth.GENERATORS[name](n, seed=11)
    eng = Engine(name, synth.DELTAS[name])
    eng.upload(data)
    for seed in (1, 2):
        full, fast = both(eng, count=H, seed=seed)
        assert_same_winner(full, fast)
        assert full["evals"] == H * n
    eng.close()


def test_plane_does_less_work_without_counts():
    n, H = 1_000_000, 131_072
    data, _ = synth.plane(n, seed=5)
    eng = Engine("plane3", synth.DELTAS["plane3"])
    eng.upload(data)
    full, fast = both(eng, count=H, seed=3)
    assert_same_winner(full, fast)
    assert full["evals"] == H * n
    assert fast["evals"] < 0.7 * H * n, fast["evals"] / (H * n)
    eng.close()


def _params_of_random_subsets(eng, H, seed):
    return eng.score(count=H, seed=seed, want_params=True)["params"]


def test_ties_go_to_the_lower_index():
    """The best parameters at two indices of a SAMPLE_PARAMS list: both arms return the lower one."""
    n, H = 200_000, CB_MIN_HYPS
    data, _ = synth.plane(n, seed=6)
    eng = Engine("plane3", synth.DELTAS["plane3"])
    eng.upload(data)
    prm = _params_of_random_subsets(eng, H, seed=4)
    ref = eng.score(params=prm, sampler=SAMPLE_PARAMS, precision=FP32, want_counts=True)
    best = prm[ref["best_index"]].copy()
    prm[ref["best_index"]] = np.nan
    lo, hi = 40_000, 70_000
    prm[lo] = best
    prm[hi] = best
    full, fast = both(eng, params=prm, sampler=SAMPLE_PARAMS)
    assert_same_winner(full, fast)
    assert fast["best_index"] == lo and full["counts"][lo] == full["counts"][hi]
    eng.close()


def test_floor_from_a_misleading_prefix():
    """The first 5 % of the data lie on a plane of their own: the hypothesis with the most inliers among the first 1 % fits
    that plane, so the floor the early exit starts from is far below the winner's count.  The winner is still found."""
    n, H = 1_000_000, CB_MIN_HYPS
    a, ta = synth.plane(n // 20, outlier_frac=0.0, seed=21)
    b, tb = synth.plane(n - n // 20, seed=22)
    data = np.ascontiguousarray(np.concatenate([a, b]))
    eng = Engine("plane3", synth.DELTAS["plane3"])
    eng.upload(data)
    prm = _params_of_random_subsets(eng, H, seed=7)
    prm[100] = ta          # the prefix's plane
    prm[60_000] = tb       # the bulk's plane
    full, fast = both(eng, params=prm, sampler=SAMPLE_PARAMS)
    assert_same_winner(full, fast)
    # the premise: the best on the first 1 % of the data is a prefix-plane hypothesis that ends well below the winner
    head = Engine("plane3", synth.DELTAS["plane3"])
    head.upload(data[: n // 100])
    h = head.score(params=prm, sampler=SAMPLE_PARAMS, precision=FP32, want_counts=True)["best_index"]
    head.close()
    assert full["counts"][h] < full["best_count"] // 2, (full["counts"][h], full["best_count"])
    eng.close()


def test_only_degenerate_hypotheses():
    n, H = 100_000, CB_MIN_HYPS
    data, _ = synth.plane(n, seed=8)
    eng = Engine("plane3", synth.DELTAS["plane3"])
    eng.upload(data)
    prm = np.full((H, eng.n_params), np.nan)
    full, fast = both(eng, params=prm, sampler=SAMPLE_PARAMS)
    assert_same_winner(full, fast)
    assert fast["best_count"] == 0 and fast["best_index"] == 0
    assert not full["counts"].any()
    eng.close()


def test_request_of_several_batches():
    """More hypotheses than one device batch: later batches start from the best count of the earlier ones."""
    n, H = 20_000, HYP_BATCH + 300_000
    data, _ = synth.plane(n, seed=9)
    eng = Engine("plane3", synth.DELTAS["plane3"])
    eng.upload(data)
    full, fast = both(eng, count=H, seed=5)
    assert_same_winner(full, fast)
    assert fast["evals"] < full["evals"] == H * n
    eng.close()
