"""lsqr_least_squares_batch_device / Engine.least_squares_batch_device: leastSquaresEstimate of every problem of a ragged batch in
device memory, optionally over masked records or with weights (absolute orientation).  Every row is pinned to the CPU oracle on
the problem's selected records; a row must not depend on the rest of the call; the call is stream-ordered like
ransac_batch_device and refuses memory that is not the context's device memory before it launches anything."""
import ctypes

import numpy as np
import pytest

from conftest import SIGN_IDX, model_family, same_up_to_sign
from lsqrrecipes_b200 import MODELS, Engine, LsqrError, synth
from oracle.pyoracle import MODELS as ORACLE_MODELS

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

REFINE_TOL = 1e-6
BATCH_MODELS = [n for n in MODELS if n not in ("usxw", "uscp")]
CASES = [(n, t) for n in BATCH_MODELS for t in ((0, 1) if model_family(n)[0] == "sphere" else (1,))]
SLEEP_CYCLES = 200_000_000   # torch.cuda._sleep: ~100 ms at the B200's ~2 GHz
LARGE = 200_003              # above 8 x kLsSliceRecords: a cluster of 16 (8 where the device schedules no 16)


def _data(name, n, seed):
    return np.ascontiguousarray(synth.GENERATORS[name](n, seed=seed)[0][:n])


def _degenerate(name, n=60, seed=3):
    """collinear points for a hyperplane, coincident points for a line, points on a hyperplane for a hypersphere; else None"""
    fam, d = model_family(name)
    rng = np.random.default_rng(seed)
    if name == "line2d":
        fam, d = "line", 2
    if fam == "plane":
        return np.outer(rng.uniform(-50, 50, n), rng.normal(size=d)) + rng.normal(size=d) * 100
    if fam == "line":
        return np.tile(np.round(rng.normal(size=d) * 100), (n, 1))   # integers: the oracle's uncentred sums are exact too
    if fam == "sphere":
        x = rng.normal(size=(n, d)) * 100
        x[:, -1] = 0.0
        return x
    return None


def _batch(problems):
    sizes = [len(p) for p in problems]
    dim = problems[0].shape[1]
    data = np.concatenate([p.reshape(-1, dim) for p in problems]) if sum(sizes) else np.zeros((0, dim))
    return np.ascontiguousarray(data), np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)


def _check_rows(port, name, ls_type, got, problems, sels=None, degenerate=()):
    m = ORACLE_MODELS[name]
    delta = synth.DELTAS[name]
    for i, p in enumerate(problems):
        x = p if sels is None else p[sels[i].astype(bool)]
        want = port.least_squares(m, delta, x, ls_type)
        row = got[i]
        if len(want) == 0:
            assert np.isnan(row).all(), (name, ls_type, i, len(x), row)
            continue
        assert not np.isnan(row).any(), (name, ls_type, i, len(x), want)
        if i in degenerate:   # an eigenvector of a repeated eigenvalue: only the rest is determined
            d = model_family(name)[1] or 2
            assert np.allclose(row[d:], want[d:], rtol=REFINE_TOL, atol=REFINE_TOL), (name, i, row, want)
            continue
        assert same_up_to_sign(row, want, SIGN_IDX[name], REFINE_TOL), (name, ls_type, i, len(x), row, want)


@pytest.mark.parametrize("name,ls_type", CASES)
def test_every_model_against_the_oracle(port, name, ls_type):
    eng = Engine(name, synth.DELTAS[name], ls_type=ls_type)
    k, dim = eng.k, eng.dim
    sizes = [0, 1, k - 1, k, 50, 3001, LARGE]
    problems = [_data(name, n, 100 + i) if n else np.zeros((0, dim)) for i, n in enumerate(sizes)]
    deg = _degenerate(name)
    degenerate = ()
    if deg is not None:
        problems.append(deg)
        degenerate = (len(problems) - 1,) if model_family(name)[0] != "sphere" else ()
    data, offsets = _batch(problems)
    got = eng.least_squares_batch_device(torch.from_numpy(data).cuda(), offsets).cpu().numpy()
    assert got.shape == (len(problems), eng.n_params)
    _check_rows(port, name, ls_type, got, problems, degenerate=degenerate)
    assert not np.isnan(got[sizes.index(LARGE)]).any()
    eng.close()


@pytest.mark.parametrize("name", ["plane3", "line3", "sphere3", "absor", "ray", "dense6"])
def test_random_masks_against_the_oracle(port, name):
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    rng = np.random.default_rng(5)
    sizes = [40, 700, 5000, 0, 90_001, 300]
    problems = [_data(name, n, 200 + i) if n else np.zeros((0, eng.dim)) for i, n in enumerate(sizes)]
    sels = [(rng.random(n) < 0.6).astype(np.uint8) for n in sizes]
    sels[0][:] = 0   # nothing selected: empty
    data, offsets = _batch(problems)
    masks = np.concatenate(sels)
    for as_bool in (False, True):
        mt = torch.from_numpy(masks).cuda()
        got = eng.least_squares_batch_device(torch.from_numpy(data).cuda(), offsets, masks=mt.bool() if as_bool else mt).cpu().numpy()
        _check_rows(port, name, 1, got, problems, sels)
        assert np.isnan(got[0]).all()
    eng.close()


@pytest.mark.parametrize("name", ["plane3", "sphere3", "absor"])
def test_refit_on_ransac_masks_equals_the_ransac_params(name):
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    sizes = [0, eng.k - 1] + [150 + (37 * i) % 400 for i in range(200)] + [30_001]
    problems = [_data(name, n, 300 + i) if n else np.zeros((0, eng.dim)) for i, n in enumerate(sizes)]
    data, offsets = _batch(problems)
    x = torch.from_numpy(data).cuda()
    r = eng.ransac_batch_device(x, offsets, prob=0.999, max_tries=256, seed=9, want_masks=True)
    refit = eng.least_squares_batch_device(x, offsets, masks=r["masks"]).cpu().numpy()
    want = r["params"].cpu().numpy()
    for i in range(len(sizes)):
        assert np.array_equal(np.isnan(refit[i]), np.isnan(want[i])), i
        if not np.isnan(want[i]).any():
            assert same_up_to_sign(refit[i], want[i], SIGN_IDX[name], REFINE_TOL), (i, refit[i], want[i])
    eng.close()


def test_weighted_horn_against_the_oracle(port):
    eng = Engine("absor", synth.DELTAS["absor"], ls_type=1)
    rng = np.random.default_rng(8)
    sizes = [500, 3000, 40, 2, 5, 70_001, 0, 800]
    problems = [_data("absor", n, 400 + i) if n else np.zeros((0, 6)) for i, n in enumerate(sizes)]
    w = [rng.uniform(0.1, 3.0, n) for n in sizes]
    w[1][rng.random(sizes[1]) < 0.3] = 0.0   # some zero weights
    sels = [np.ones(n, dtype=np.uint8) for n in sizes]
    sels[2] = (rng.random(40) < 0.5).astype(np.uint8)   # with a mask
    sels[4][:3] = 0                                      # two selected pairs: empty
    sels[5] = (rng.random(sizes[5]) < 0.7).astype(np.uint8)
    data, offsets = _batch(problems)
    x = torch.from_numpy(data).cuda()
    wt = torch.from_numpy(np.concatenate(w)).cuda()
    mt = torch.from_numpy(np.concatenate(sels)).cuda()
    for masks in (None, mt):
        got = eng.least_squares_batch_device(x, offsets, masks=masks, weights=wt).cpu().numpy()
        for i, n in enumerate(sizes):
            s = np.ones(n, dtype=bool) if masks is None else sels[i].astype(bool)
            want = port.weighted_absor(problems[i][s], w[i][s])
            if len(want) == 0:
                assert np.isnan(got[i]).all(), (i, got[i])
            else:
                assert same_up_to_sign(got[i], want, SIGN_IDX["absor"], REFINE_TOL), (i, got[i], want)
        assert np.isnan(got[3]).all() and np.isnan(got[6]).all()
    assert np.isnan(eng.least_squares_batch_device(x, offsets, masks=mt, weights=wt).cpu().numpy()[4]).all()
    eng.close()


def test_rows_are_bitwise_independent_of_the_call():
    name = "plane3"
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    alone = [_data(name, 7, 1), _data(name, 1001, 2), _data(name, 120_001, 3)]
    mixed = [_data(name, 50 + (13 * i) % 300, 500 + i) for i in range(3000)]
    mixed.insert(17, alone[0])
    mixed.insert(1500, alone[1])
    mixed.insert(2999, alone[2])
    where = [17, 1500, 2999]
    data, offsets = _batch(mixed)
    x = torch.from_numpy(data).cuda()
    big = eng.least_squares_batch_device(x, offsets).cpu().numpy()
    assert big.tobytes() == eng.least_squares_batch_device(x, offsets).cpu().numpy().tobytes(), "two calls"
    for a, i in zip(alone, where):
        one = eng.least_squares_batch_device(torch.from_numpy(a).cuda(), [0, len(a)]).cpu().numpy()
        assert one.tobytes() == big[i].tobytes(), i
        # another position: one record of padding shifts the problem off its 16-byte alignment
        pad = np.concatenate([_data(name, 3, 9), a])
        two = eng.least_squares_batch_device(torch.from_numpy(pad).cuda(), [0, 3, 3 + len(a)]).cpu().numpy()
        assert two[1].tobytes() == big[i].tobytes(), i
    # [B, n, dim] with [B, n] masks is the offsets layout with flat masks
    B, n = 64, 333
    cube = _data(name, B * n, 77)
    mask = (np.random.default_rng(2).random(B * n) < 0.8).astype(np.uint8)
    flat = eng.least_squares_batch_device(torch.from_numpy(cube).cuda(), np.arange(B + 1, dtype=np.uint64) * n,
                                          masks=torch.from_numpy(mask).cuda()).cpu().numpy()
    c3 = eng.least_squares_batch_device(torch.from_numpy(cube).cuda().reshape(B, n, 3), masks=torch.from_numpy(mask).cuda().reshape(B, n))
    assert c3.cpu().numpy().tobytes() == flat.tobytes()
    eng.close()


@pytest.mark.parametrize("name", ["plane3", "line3", "sphere3", "absor"])
def test_offset_data(name):
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    shift = np.array([1e6, -1e6, 1e6])
    problems = [_data(name, n, 600 + i) for i, n in enumerate([100, 5000, 60_001])]
    moved = [p.copy() for p in problems]
    for p in moved:
        if name == "absor":
            p[:, 0:3] += shift
            p[:, 3:6] += shift
        else:
            p[:, :3] += shift
    a = eng.least_squares_batch_device(torch.from_numpy(_batch(problems)[0]).cuda(), _batch(problems)[1]).cpu().numpy()
    b = eng.least_squares_batch_device(torch.from_numpy(_batch(moved)[0]).cuda(), _batch(moved)[1]).cpu().numpy()
    for i in range(len(problems)):
        want = a[i].copy()
        if name == "plane3" or name == "line3":
            want[3:6] += shift
        elif name == "sphere3":
            want[:3] += shift
        else:   # x2 = R x1 + t: both frames shifted by s -> t' = t + s - R s
            from lsqrrecipes_b200.synth import quat_to_matrix
            q = want[:4] / np.linalg.norm(want[:4])
            want[4:7] += shift - quat_to_matrix(*q) @ shift
        assert same_up_to_sign(b[i], want, SIGN_IDX[name], REFINE_TOL), (i, b[i], want)
    eng.close()


def _stream_handle():
    return torch.cuda.current_stream().cuda_stream or 1


def test_stream_semantics():
    name = "sphere3"
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    problems = [_data(name, 200 + i, 700 + i) for i in range(500)]
    first, offsets = _batch(problems)
    second = first + 3.0
    x = torch.from_numpy(first).cuda()
    src = torch.from_numpy(second).cuda()
    want = eng.least_squares_batch_device(src, offsets).cpu().numpy()
    eng.least_squares_batch_device(x, offsets)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        x.copy_(src)
        out = eng.least_squares_batch_device(x, offsets)
        pending = not side.query()
    assert pending, "least_squares_batch_device waited for its stream"
    side.synchronize()
    assert out.cpu().numpy().tobytes() == want.tobytes()

    # ordered against the context's own calls: lsqr_least_squares on its stream before and after a call on a busy side stream
    single = problems[3]
    ref = eng.least_squares(single)
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES // 2)
        out = eng.least_squares_batch_device(x, offsets)
    assert eng.least_squares(single).tobytes() == ref.tobytes()
    side.synchronize()
    assert out.cpu().numpy().tobytes() == want.tobytes()
    eng.close()


def _raw(eng, data_ptr, offsets, masks_ptr, weights_ptr, params_ptr):
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    return eng.lib.lsqr_least_squares_batch_device(eng.h, data_ptr, off.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), len(off) - 1,
                                                   masks_ptr, weights_ptr, params_ptr, _stream_handle())


def test_rejections_before_any_launch():
    eng = Engine("absor", synth.DELTAS["absor"], ls_type=1)
    problems = [_data("absor", 50 + i, 800 + i) for i in range(40)]
    data, offsets = _batch(problems)
    total, B = data.shape[0], len(problems)
    good = {"dev_data": torch.from_numpy(data).cuda(), "dev_masks": torch.ones(total, dtype=torch.uint8, device="cuda"),
            "dev_weights": torch.ones(total, dtype=torch.float64, device="cuda"),
            "dev_params": torch.empty((B, eng.n_params), dtype=torch.float64, device="cuda")}

    def call(a):
        return _raw(eng, a["dev_data"].data_ptr(), offsets, a["dev_masks"].data_ptr(), a["dev_weights"].data_ptr(), a["dev_params"].data_ptr())

    assert call(good) == 0
    torch.cuda.synchronize()
    for bad in good:
        before = eng.kernel_launches
        assert call({k: (torch.empty(v.shape, dtype=v.dtype, pin_memory=True) if k == bad else v) for k, v in good.items()}) == -1, bad
        assert bad in eng.lib.lsqr_last_error(eng.h).decode(), bad
        assert eng.kernel_launches == before, bad
    before = eng.kernel_launches
    assert _raw(eng, good["dev_data"].data_ptr(), [0, 10, 5], None, None, good["dev_params"].data_ptr()) == -1
    assert "non-decreasing" in eng.lib.lsqr_last_error(eng.h).decode() and eng.kernel_launches == before
    eng.close()

    plane = Engine("plane3", 0.5, ls_type=1)
    x = torch.from_numpy(_data("plane3", 100, 1)).cuda()
    w = torch.ones(100, dtype=torch.float64, device="cuda")
    prm = torch.empty((1, 6), dtype=torch.float64, device="cuda")
    assert _raw(plane, x.data_ptr(), [0, 100], None, w.data_ptr(), prm.data_ptr()) == -1
    assert "dev_weights" in plane.lib.lsqr_last_error(plane.h).decode() and plane.kernel_launches == 0
    with pytest.raises(ValueError, match="absor"):
        plane.least_squares_batch_device(x, [0, 100], weights=w)
    plane.close()

    us = Engine("usxw", synth.DELTAS["usxw"], ls_type=1)
    xu = torch.zeros((10, 14), dtype=torch.float64, device="cuda")
    with pytest.raises(LsqrError, match="no batched mode"):
        us.least_squares_batch_device(xu, [0, 10])
    assert us.kernel_launches == 0
    us.close()


def test_group_context_is_refused():
    from lsqrrecipes_b200 import api
    if api.load_library().lsqr_device_count() < 2:
        pytest.skip("needs two GPUs")
    eng = Engine("plane3", 0.5, ls_type=1, gpus=0)
    with pytest.raises(LsqrError, match="status -1"):
        eng.least_squares_batch_device(torch.from_numpy(_data("plane3", 100, 1)).cuda(), [0, 100])
    eng.close()
