"""Argument checks of Engine.least_squares_batch_device (lsqrrecipes_b200.api.check_ls_batch_device_args) on CPU tensors: each
malformed argument raises ValueError before any library call, with no device needed."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from lsqrrecipes_b200.api import MODELS, check_ls_batch_device_args  # noqa: E402

DIM = 6
ABSOR, PLANE = MODELS["absor"], MODELS["plane3"]


def _flat(total=10):
    return torch.zeros((total, DIM), dtype=torch.float64)


def _check(data=None, offsets=(0, 4, 10), model=ABSOR, **kw):
    return check_ls_batch_device_args(_flat() if data is None else data, list(offsets) if offsets is not None else None, DIM, model, **kw)


def test_well_formed_arguments_reach_the_device_check():
    with pytest.raises(ValueError, match="CUDA memory"):
        _check(masks=torch.ones(10, dtype=torch.bool), weights=torch.ones(10, dtype=torch.float64))
    with pytest.raises(ValueError, match="CUDA memory"):
        _check(torch.zeros((2, 5, DIM), dtype=torch.float64), None, masks=torch.ones((2, 5), dtype=torch.uint8))


def test_data_checks_are_those_of_ransac_batch_device():
    with pytest.raises(ValueError, match="torch tensor"):
        _check(np.zeros((10, DIM)))
    with pytest.raises(ValueError, match="float64"):
        _check(torch.zeros((10, DIM), dtype=torch.float32))
    with pytest.raises(ValueError, match="contiguous"):
        _check(torch.zeros((DIM, 10), dtype=torch.float64).t())
    with pytest.raises(ValueError, match=r"\[total, 6\]"):
        _check(torch.zeros((10, DIM + 1), dtype=torch.float64))
    with pytest.raises(ValueError, match="non-decreasing"):
        _check(offsets=(0, 6, 4, 10))


def test_weights_on_another_model():
    with pytest.raises(ValueError, match="absor"):
        _check(model=PLANE, weights=torch.ones(10, dtype=torch.float64))


@pytest.mark.parametrize("what", ["masks", "weights"])
def test_masks_and_weights(what):
    good = torch.uint8 if what == "masks" else torch.float64
    bad = torch.int32 if what == "masks" else torch.float32
    with pytest.raises(ValueError, match=f"{what} must be a torch tensor"):
        _check(**{what: np.ones(10)})
    with pytest.raises(ValueError, match=f"{what} must be torch"):
        _check(**{what: torch.ones(10, dtype=bad)})
    with pytest.raises(ValueError, match=f"{what} must be contiguous"):
        _check(**{what: torch.ones((20,), dtype=good)[::2]})
    for shape in [(9,), (10, 1), (2, 5)]:
        with pytest.raises(ValueError, match=f"{what} must have shape \\[10\\]"):
            _check(**{what: torch.ones(shape, dtype=good)})
    with pytest.raises(ValueError, match=f"{what} must have shape \\[2, 5\\]"):
        _check(torch.zeros((2, 5, DIM), dtype=torch.float64), None, **{what: torch.ones(10, dtype=good)})


def test_masks_on_another_device():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    data = _flat().cuda()
    with pytest.raises(ValueError, match="masks must be in CUDA memory"):
        check_ls_batch_device_args(data, [0, 10], DIM, ABSOR, masks=torch.ones(10, dtype=torch.uint8))
    with pytest.raises(ValueError, match="weights must be in CUDA memory"):
        check_ls_batch_device_args(data, [0, 10], DIM, ABSOR, weights=torch.ones(10, dtype=torch.float64))
