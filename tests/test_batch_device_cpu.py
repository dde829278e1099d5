"""Argument checks of Engine.ransac_batch_device (lsqrrecipes_b200.api.check_batch_device_args), on CPU tensors and numpy arrays:
each malformed argument raises ValueError before any library call, with no device needed."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from lsqrrecipes_b200.api import check_batch_device_args  # noqa: E402

DIM = 3


def _flat(total=10):
    return torch.zeros((total, DIM), dtype=torch.float64)


def test_numpy_data_is_rejected():
    with pytest.raises(ValueError, match="torch tensor"):
        check_batch_device_args(np.zeros((10, DIM)), [0, 10], DIM)


def test_cpu_tensor_is_rejected_after_every_other_check():
    with pytest.raises(ValueError, match="CUDA memory"):
        check_batch_device_args(_flat(), [0, 4, 10], DIM)
    with pytest.raises(ValueError, match="CUDA memory"):
        check_batch_device_args(torch.zeros((2, 5, DIM), dtype=torch.float64), None, DIM)


def test_float32_is_rejected():
    with pytest.raises(ValueError, match="float64"):
        check_batch_device_args(torch.zeros((10, DIM), dtype=torch.float32), [0, 10], DIM)


def test_non_contiguous_is_rejected():
    with pytest.raises(ValueError, match="contiguous"):
        check_batch_device_args(torch.zeros((DIM, 10), dtype=torch.float64).t(), [0, 10], DIM)


@pytest.mark.parametrize("shape,offsets", [((10, DIM + 1), [0, 10]), ((2, 5, DIM + 1), None), ((10 * DIM,), [0, 10]), ((10, DIM), None)])
def test_shape_against_dim(shape, offsets):
    with pytest.raises(ValueError, match=r"\[total, 3\]|dim = 3|needs offsets"):
        check_batch_device_args(torch.zeros(shape, dtype=torch.float64), offsets, DIM)


def test_cuda_offsets_are_rejected():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    with pytest.raises(ValueError, match="host memory"):
        check_batch_device_args(_flat(), torch.tensor([0, 10], device="cuda"), DIM)


@pytest.mark.parametrize("offsets", [[], np.zeros((2, 2), dtype=np.int64), [0.0, 10.0], [-1, 10]])
def test_offsets_length_and_type(offsets):
    with pytest.raises(ValueError, match="offsets"):
        check_batch_device_args(_flat(), offsets, DIM)


@pytest.mark.parametrize("offsets", [[0, 6, 4, 10], np.array([5, 3], dtype=np.uint64), torch.tensor([0, 9, 8])])
def test_decreasing_offsets(offsets):
    with pytest.raises(ValueError, match="non-decreasing"):
        check_batch_device_args(_flat(), offsets, DIM)


@pytest.mark.parametrize("offsets", [[0, 11], [0, 4, 10, 12]])
def test_offsets_past_the_end_of_data(offsets):
    with pytest.raises(ValueError, match="past the 10 records"):
        check_batch_device_args(_flat(), offsets, DIM)
