"""lsqr_ransac_batch above one thread block: problems too large for one block's shared memory are solved by a thread-block
cluster each (batch_cluster_kernel).  The limits come from Engine.batch_capacity; fp64 results are pinned against an
independent path (the same Philox hypotheses scored by lsqr_score, the round loop and stop rule replayed here, the consensus
set from lsqr_consensus, the refit from the CPU oracle); a problem's outputs must not depend on the other problems of the call."""
import math

import numpy as np
import pytest

from conftest import SIGN_IDX, same_up_to_sign
from lsqrrecipes_b200 import FP32, FP64, MODELS, SAMPLE_PHILOX, Engine, LsqrError, synth
from oracle.pyoracle import INFO
from oracle.pyoracle import MODELS as ORACLE_MODELS

pytestmark = pytest.mark.gpu

REFINE_TOL = 1e-6
BATCH_MODELS = [n for n in MODELS if n not in ("usxw", "uscp")]
EXACT_CASES = [("plane3", 1), ("line2d", 1), ("line3", 1), ("sphere3", 0), ("sphere3", 1), ("absor", 1), ("ray", 1), ("pivot", 1),
               ("plane8", 1), ("dense8", 1)]
SEED, PROB, TRIES = 20261021, 0.999, 256


def _data(name, n, seed):
    return np.ascontiguousarray(synth.GENERATORS[name](n, seed=seed)[0][:n])


def _batch(problems):
    sizes = [len(p) for p in problems]
    return np.concatenate(problems), np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)


def _filler(name, count):
    """1-record problems: no hypothesis, count 0, NaN parameters"""
    return [_data(name, 1, 5) for _ in range(count)]


def _sizes(one_block, max_records):
    """just above one block, and near half the capacity; odd and not a multiple of any cluster size"""
    a = one_block + 3 if (one_block + 3) % 2 else one_block + 4
    b = max_records // 2 - 5
    b = b if b % 2 else b - 1
    return [a, b]


def _replay(counts, valid, n, k, prob, max_tries):
    """batch_kernel's round loop (rounds of 32, strict > on the key, the stop rule after a raise).  Returns (winner, count,
    conclusive): conclusive is False when a stop-rule value t + 0.5 lies within a few ulps of an integer, where the device's
    log / pow may round to the other side."""
    tries = min(math.comb(n, k), 0xFFFFFFFF) if n >= k else 0
    tries = min(tries, max_tries)
    best, done, conclusive = 0, 0, True
    log1mp = math.log(1.0 - prob)
    while done < tries:
        keys = [(int(counts[h]) << 32) | (0xFFFFFFFF - h) if valid[h] else 0 for h in range(done, min(done + 32, tries))]
        rb = max(keys, default=0)
        if rb > best:
            best = rb
            c = best >> 32
            if c == n:
                tries = 0
            elif 0.0 < prob < 1.0 and c > 0:
                t = log1mp / math.log(1.0 - (c / n) ** k) + 0.5
                if abs(t - round(t)) <= 8 * math.ulp(t):
                    conclusive = False
                nt = 0xFFFFFFFF if t >= 4294967295.0 else int(t)
                tries = min(nt, tries)
        done += 32
    return 0xFFFFFFFF - (best & 0xFFFFFFFF), best >> 32, conclusive


@pytest.mark.parametrize("precision", [FP64, FP32])
@pytest.mark.parametrize("name", BATCH_MODELS)
def test_capacity_contract(name, precision):
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    one, most = eng.batch_capacity(precision)
    assert most > one > 0
    one64 = eng.batch_capacity(FP64)[0]   # exhaustive mode always scores in fp64, one block per problem
    assert eng.batch_capacity(precision, exhaustive=True) == (one64, one64)
    for n in (one, one + 1, most):
        data = _data(name, n, 11 + n % 7)
        out = eng.ransac_batch(data, [0, n], prob=PROB, max_tries=32, seed=3, want_masks=True, precision=precision)
        assert out["masks"].sum() == out["counts"][0], n
    data = _data(name, most + 1, 12)
    with pytest.raises(LsqrError, match=f"limit of {most} records"):
        eng.ransac_batch(data, [0, most + 1], prob=PROB, max_tries=32, seed=3, precision=precision)
    with pytest.raises(LsqrError, match="does not fit in shared memory"):
        eng.ransac_batch(data[: one64 + 1], [0, one64 + 1], exhaustive=True)
    eng.close()


@pytest.mark.parametrize("name,ls_type", EXACT_CASES)
def test_cluster_results_against_independent_path(port, name, ls_type):
    """fp64: winner, count and mask exactly those of the replayed rounds over lsqr_score's counts, parameters the oracle's
    least squares on that mask.  fp32: deterministic, self-consistent and within the fp32 band of the fp64 winner."""
    m = ORACLE_MODELS[name]
    k = INFO[m][2]
    delta = synth.DELTAS[name]
    eng = Engine(name, delta, ls_type=ls_type)
    inconclusive = []
    for size_i, n in enumerate(_sizes(*eng.batch_capacity(FP64))):
        gb = 3 + size_i
        data = _data(name, n, 900 + n % 97)
        batch, offsets = _batch(_filler(name, gb) + [data])
        o64 = eng.ransac_batch(batch, offsets, prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True, precision=FP64)
        o32 = eng.ransac_batch(batch, offsets, prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True, precision=FP32)
        again = eng.ransac_batch(batch, offsets, prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True, precision=FP32)
        lo = int(offsets[gb])

        single = Engine(name, delta, ls_type=ls_type)
        single.upload(data)
        r = single.score(count=TRIES, sampler=SAMPLE_PHILOX, precision=FP64, seed=SEED, first=gb << 32, want_counts=True, want_params=True)
        valid = ~np.isnan(r["params"]).any(axis=1)
        h, c, conclusive = _replay(r["counts"], valid, n, k, PROB, TRIES)
        if not conclusive:
            inconclusive.append(n)
            single.close()
            continue
        assert o64["counts"][gb] == c, (n, o64["counts"][gb], c)
        assert single.consensus(r["params"][h]) == c
        mask = single.get_mask()
        single.close()
        assert np.array_equal(o64["masks"][lo:], mask), n
        want = port.least_squares(m, delta, data[mask.astype(bool)], ls_type)
        assert len(want) and same_up_to_sign(o64["params"][gb], want, SIGN_IDX[name], REFINE_TOL), (n, o64["params"][gb], want)

        assert np.array_equal(o32["counts"], again["counts"]) and np.array_equal(o32["masks"], again["masks"])
        assert o32["params"].tobytes() == again["params"].tobytes()
        m32 = o32["masks"][lo:]
        assert m32.sum() == o32["counts"][gb]
        want32 = port.least_squares(m, delta, data[m32.astype(bool)], ls_type)
        assert len(want32) and same_up_to_sign(o32["params"][gb], want32, SIGN_IDX[name], REFINE_TOL), (n, o32["params"][gb], want32)
        assert abs(int(o32["counts"][gb]) - int(c)) <= max(2, 0.02 * c), (n, o32["counts"][gb], c)
        assert not o64["masks"][:lo].any() and not o32["masks"][:lo].any()
    eng.close()
    if inconclusive:
        pytest.skip(f"inconclusive: the stop rule of n = {inconclusive} lies within a few ulps of an integer")


def _mixed(name, one_block, max_records):
    """300 small problems and three large ones at indices 0, 150 and 302 (three cluster sizes)"""
    small = [_data(name, 150 + (37 * i) % 113, 3000 + i) + 30.0 * i for i in range(300)]
    large = {0: _data(name, one_block + 1, 41), 150: _data(name, 4 * one_block + 7, 42), 302: _data(name, max_records // 2 - 1, 43)}
    problems = list(small)
    for i in sorted(large):
        problems.insert(i, large[i])
    return problems, sorted(large)


def _pinned(a):
    torch = pytest.importorskip("torch")
    t = torch.empty(a.shape, dtype=torch.float64, pin_memory=True)
    view = t.numpy()
    view[...] = a
    return view, t


def _run(eng, problems, precision, pinned):
    data, offsets = _batch(problems)
    keep = None
    if pinned:
        data, keep = _pinned(data)
    out = eng.ransac_batch(data, offsets, prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True, precision=precision)
    del keep
    return out, offsets


def _same(a, oa, b, ob, i):
    assert a["params"][i].tobytes() == b["params"][i].tobytes(), i
    assert a["counts"][i] == b["counts"][i], i
    assert np.array_equal(a["masks"][int(oa[i]):int(oa[i + 1])], b["masks"][int(ob[i]):int(ob[i + 1])]), i


@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("precision", [FP64, FP32])
def test_results_depend_only_on_the_problem(precision, pinned):
    name = "plane3"
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    problems, large = _mixed(name, *eng.batch_capacity(precision))
    out, off = _run(eng, problems, precision, pinned)
    no_large = [_data(name, 1, 5) if i in large else p for i, p in enumerate(problems)]
    out_s, off_s = _run(eng, no_large, precision, pinned)
    only_large = [p if i in large else _data(name, 1, 5) for i, p in enumerate(problems)]
    out_l, off_l = _run(eng, only_large, precision, pinned)
    eng.close()
    for i in range(len(problems)):
        if i in large:
            _same(out, off, out_l, off_l, i)
            assert out["counts"][i] > 0
        else:
            _same(out, off, out_s, off_s, i)
        assert out["masks"][int(off[i]):int(off[i + 1])].sum() == out["counts"][i], i


@pytest.mark.parametrize("precision", [FP64, FP32])
def test_degenerate_and_exact_large_problems(precision):
    name = "plane3"
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    one, _ = eng.batch_capacity(precision)
    n = 3 * one + 5
    same = np.tile(np.array([[1.0, 2.0, 3.0]]), (n, 1))
    out = eng.ransac_batch(same, [0, n], prob=PROB, max_tries=64, seed=1, want_masks=True, precision=precision)
    assert np.isnan(out["params"][0]).all() and out["counts"][0] == 0 and not out["masks"].any()
    rng = np.random.default_rng(5)
    flat = np.column_stack([rng.uniform(-500, 500, n), rng.uniform(-500, 500, n), np.full(n, 7.0)])   # every record on z = 7
    out = eng.ransac_batch(flat, [0, n], prob=PROB, max_tries=TRIES, seed=1, want_masks=True, precision=precision)
    assert out["counts"][0] == n and out["masks"].all()
    assert abs(abs(out["params"][0][2]) - 1.0) < 1e-9 and abs(out["params"][0][5] - 7.0) < 1e-9
    eng.close()


def test_group_context_matches_one_gpu():
    from lsqrrecipes_b200 import api
    if api.load_library().lsqr_device_count() < 2:
        pytest.skip("needs two GPUs")
    name = "plane3"
    one = Engine(name, synth.DELTAS[name], ls_type=1)
    many = Engine(name, synth.DELTAS[name], ls_type=1, gpus=0)
    for precision in (FP64, FP32):
        problems, _ = _mixed(name, *one.batch_capacity(precision))
        a, _ = _run(one, problems, precision, False)
        b, _ = _run(many, problems, precision, False)
        assert a["params"].tobytes() == b["params"].tobytes()
        assert np.array_equal(a["counts"], b["counts"]) and np.array_equal(a["masks"], b["masks"])
    one.close()
    many.close()
