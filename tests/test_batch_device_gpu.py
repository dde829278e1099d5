"""lsqr_ransac_batch_device / Engine.ransac_batch_device: lsqr_ransac_batch on data already in device memory, stream-ordered.
Every result is pinned bit for bit to the host path on the same data; the call must return before the device has run it,
run after the work queued before it on the caller's stream, stay ordered against the context's own calls, leave the uploaded
data set alone, and refuse memory that is not the context's device memory before it launches anything."""
import ctypes

import numpy as np
import pytest

from lsqrrecipes_b200 import FP32, FP64, MODELS, Engine, LsqrError, synth
from test_batch_cluster_gpu import _batch, _data, _mixed

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

BATCH_MODELS = [n for n in MODELS if n not in ("usxw", "uscp")]
SEED, PROB, TRIES = 20261022, 0.999, 256
SLEEP_CYCLES = 200_000_000   # torch.cuda._sleep: ~100 ms at the B200's ~2 GHz


def _small_batch(name, k, count=200, seed=7):
    """`count` (> 101) problems of varied sizes from k to k + 196 records; problem 17 is empty, problem 101 has k - 1 records"""
    sizes = [k + (53 * i) % 197 for i in range(count)]
    sizes[17], sizes[101] = 0, k - 1
    data = _data(name, sum(sizes), seed)
    return data, np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)


def _stream_handle():
    return torch.cuda.current_stream().cuda_stream or 1   # 1: cudaStreamLegacy, the stream torch reports as 0


def _assert_same(dev, host, what=""):
    torch.cuda.synchronize()
    assert dev["params"].cpu().numpy().tobytes() == host["params"].tobytes(), what
    assert np.array_equal(dev["counts"].cpu().numpy().astype(np.uint32), host["counts"]), what
    if host["masks"] is not None:
        assert np.array_equal(dev["masks"].cpu().numpy(), host["masks"]), what


def _both(eng, data, offsets, **kw):
    host = eng.ransac_batch(data, offsets, want_masks=True, **kw)
    dev = eng.ransac_batch_device(torch.from_numpy(data).cuda(), offsets, want_masks=True, **kw)
    return dev, host


@pytest.mark.parametrize("precision", [FP64, FP32])
@pytest.mark.parametrize("name", BATCH_MODELS)
def test_equal_to_the_host_path(name, precision):
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    data, offsets = _small_batch(name, eng.k)
    dev, host = _both(eng, data, offsets, prob=PROB, max_tries=TRIES, seed=SEED, precision=precision)
    _assert_same(dev, host, name)
    assert host["counts"][17] == 0 and host["counts"][101] == 0 and np.isnan(host["params"][17]).all()
    eng.close()


@pytest.mark.parametrize("name", ["plane3", "line2d", "sphere3", "absor"])
def test_exhaustive_equal_to_the_host_path(name):
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    sizes = [0, eng.k - 1] + list(range(eng.k, 19)) + [13, 17]
    data = _data(name, sum(sizes), 11)
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    dev, host = _both(eng, data, offsets, exhaustive=True)
    _assert_same(dev, host, name)
    eng.close()


@pytest.mark.parametrize("precision", [FP64, FP32])
def test_cluster_problems_equal_to_the_host_path(precision):
    name = "plane3"
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    problems, large = _mixed(name, *eng.batch_capacity(precision))
    data, offsets = _batch(problems)
    dev, host = _both(eng, data, offsets, prob=PROB, max_tries=TRIES, seed=SEED, precision=precision)
    _assert_same(dev, host)
    assert all(host["counts"][i] > 0 for i in large)
    eng.close()


def _raw(eng, data_ptr, offsets, params_ptr, counts_ptr, masks_ptr, precision=FP64, exhaustive=0, stream=None):
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    return eng.lib.lsqr_ransac_batch_device(eng.h, data_ptr, off.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), len(off) - 1, exhaustive,
                                            PROB, TRIES, SEED, precision, params_ptr, counts_ptr, masks_ptr,
                                            stream if stream is not None else _stream_handle())


def test_layouts_and_every_mask_byte():
    name = "plane3"
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    B, n = 300, 97
    data = _data(name, B * n, 21)
    offsets = np.arange(B + 1, dtype=np.uint64) * n
    host = eng.ransac_batch(data, offsets, prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True)
    cube = torch.from_numpy(data).cuda().reshape(B, n, 3)
    _assert_same(eng.ransac_batch_device(cube, prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True), host, "[B, n, dim]")
    # a view at a non-zero storage offset inside a larger tensor
    big = torch.full((7 + B * n + 5, 3), float("nan"), dtype=torch.float64, device="cuda")
    big[7:7 + B * n] = torch.from_numpy(data).cuda()
    view = big[7:7 + B * n]
    assert view.storage_offset() > 0 and view.is_contiguous()
    _assert_same(eng.ransac_batch_device(view, offsets, prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True), host, "view")
    # the C entry point writes every byte of [offsets[0], offsets[B]) and none outside it
    lead = 5
    padded = torch.cat([torch.zeros((lead, 3), dtype=torch.float64), torch.from_numpy(data)]).cuda()
    prm = torch.empty((B, eng.n_params), dtype=torch.float64, device="cuda")
    cnt = torch.empty(B, dtype=torch.int32, device="cuda")
    mask = torch.full((lead + B * n,), 0xFF, dtype=torch.uint8, device="cuda")
    assert _raw(eng, padded.data_ptr(), offsets + lead, prm.data_ptr(), cnt.data_ptr(), mask.data_ptr()) == 0
    torch.cuda.synchronize()
    m = mask.cpu().numpy()
    assert (m[:lead] == 0xFF).all() and set(np.unique(m[lead:])) <= {0, 1}
    assert np.array_equal(np.add.reduceat(m[lead:].astype(np.int64), offsets[:-1].astype(np.int64)), cnt.cpu().numpy())
    assert prm.cpu().numpy().tobytes() == host["params"].tobytes()
    eng.close()


def test_returns_before_the_device_runs_it_and_runs_after_earlier_work():
    name = "plane3"
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    first, offsets = _small_batch(name, eng.k, count=2000, seed=31)
    second, _ = _small_batch(name, eng.k, count=2000, seed=32)
    x = torch.from_numpy(first).cuda()
    src = torch.from_numpy(second).cuda()
    kw = dict(prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True)
    for _ in range(2):   # both staging slots and every buffer at this size: growing them may synchronise
        eng.ransac_batch_device(x, offsets, **kw)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        x.copy_(src)
        out = eng.ransac_batch_device(x, offsets, **kw)
        pending = not side.query()
    assert pending, "ransac_batch_device waited for its stream"
    side.synchronize()
    _assert_same(out, eng.ransac_batch(second, offsets, **kw))
    eng.close()


def test_ordered_against_the_context():
    name = "plane3"
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    a, off_a = _small_batch(name, eng.k, count=2000, seed=41)
    b, off_b = _small_batch(name, eng.k, count=1500, seed=42)
    kw = dict(prob=PROB, max_tries=TRIES, seed=SEED, want_masks=True)
    ref_a, ref_b = eng.ransac_batch(a, off_a, **kw), eng.ransac_batch(b, off_b, **kw)
    a_dev = torch.from_numpy(a).cuda()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES // 2)
        out_a = eng.ransac_batch_device(a_dev, off_a, **kw)
    out_b = eng.ransac_batch(b, off_b, **kw)   # the host path on the context's stream, while the device call still waits
    side.synchronize()
    _assert_same(out_a, ref_a, "device call")
    assert out_b["params"].tobytes() == ref_b["params"].tobytes() and np.array_equal(out_b["counts"], ref_b["counts"])
    assert np.array_equal(out_b["masks"], ref_b["masks"])

    # the uploaded data set and its stored consensus set are left as they are
    d = _data(name, 20000, 43)
    eng.upload(d)
    r = eng.ransac(PROB, precision=FP64, seed=3, want_mask=False)
    count = eng.consensus(r["params"])
    mask0, refined0 = eng.get_mask(), eng.refine()
    with torch.cuda.stream(side):
        eng.ransac_batch_device(a_dev, off_a, **kw)
    side.synchronize()
    assert eng.get_mask().tobytes() == mask0.tobytes() and int(mask0.sum()) == count
    assert eng.refine().tobytes() == refined0.tobytes()
    eng.close()


def _pinned_like(t):
    return torch.empty(t.shape, dtype=t.dtype, pin_memory=True)


def test_rejections_before_any_launch():
    """Page-locked host memory is reachable from the device, so a missing check could not fault here.  Pageable memory and
    another GPU's memory go through the same check and are not passed on purpose."""
    name = "plane3"
    eng = Engine(name, synth.DELTAS[name], ls_type=1)
    data, offsets = _small_batch(name, eng.k, count=120)
    B, total = len(offsets) - 1, data.shape[0]
    good = {"dev_data": torch.from_numpy(data).cuda(), "dev_params": torch.empty((B, eng.n_params), dtype=torch.float64, device="cuda"),
            "dev_counts": torch.empty(B, dtype=torch.int32, device="cuda"), "dev_masks": torch.empty(total, dtype=torch.uint8, device="cuda")}

    def call(a):
        return _raw(eng, a["dev_data"].data_ptr(), offsets, a["dev_params"].data_ptr(), a["dev_counts"].data_ptr(), a["dev_masks"].data_ptr())

    assert call(good) == 0
    torch.cuda.synchronize()
    for bad in good:
        before = eng.kernel_launches
        assert call({k: (_pinned_like(v) if k == bad else v) for k, v in good.items()}) == -1, bad
        assert bad in eng.lib.lsqr_last_error(eng.h).decode(), bad
        assert eng.kernel_launches == before, bad
    torch.cuda.synchronize()

    def message(fn):
        with pytest.raises(LsqrError) as e:
            fn()
        return str(e.value)

    for precision in (FP64, FP32):
        most = eng.batch_capacity(precision)[1]
        big = _data(name, most + 1, 12)
        host = message(lambda: eng.ransac_batch(big, [0, most + 1], precision=precision))
        assert f"limit of {most} records" in host
        assert message(lambda: eng.ransac_batch_device(torch.from_numpy(big).cuda(), [0, most + 1], precision=precision)) == host
    one = eng.batch_capacity(FP64, exhaustive=True)[0]
    over = _data(name, one + 1, 13)
    host = message(lambda: eng.ransac_batch(over, [0, one + 1], exhaustive=True))
    assert "does not fit in shared memory" in host
    assert message(lambda: eng.ransac_batch_device(torch.from_numpy(over).cuda(), [0, one + 1], exhaustive=True)) == host
    host = message(lambda: eng.ransac_batch(data, offsets, precision=7))
    assert message(lambda: eng.ransac_batch_device(good["dev_data"], offsets, precision=7)) == host == "status -1: bad precision"
    eng.close()


def test_group_context_is_refused():
    from lsqrrecipes_b200 import api
    if api.load_library().lsqr_device_count() < 2:
        pytest.skip("needs two GPUs")
    name = "plane3"
    eng = Engine(name, synth.DELTAS[name], ls_type=1, gpus=0)
    data, offsets = _small_batch(name, eng.k, count=120)
    with pytest.raises(LsqrError, match="status -1"):
        eng.ransac_batch_device(torch.from_numpy(data).cuda(), offsets)
    eng.close()
