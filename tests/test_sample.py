"""Argument rules of the affine sampling grid (``_ops.grid_args``), host only: no device work happens here."""
import numpy as np
import pytest

from imgcompressionmps import _ops


def test_grid_args_normalises_its_inputs():
    origin, steps, shape = _ops.grid_args(3, [1, 2, 3], [[0.5, 0, 0], [0, 0.25, 1]], (np.int64(4), 5))
    assert origin.dtype == np.float64 and origin.shape == (3,) and origin.flags.c_contiguous
    assert steps.dtype == np.float64 and steps.shape == (2, 3) and steps.flags.c_contiguous
    assert shape == (4, 5) and all(type(v) is int for v in shape)
    assert _ops.grid_args(2, np.float32([0, 0]), np.eye(2, dtype=np.float32)[:1], [0])[2] == (0,)
    assert _ops.grid_args(1, [0.0], np.ones((8, 1)), [1] * 8)[1].shape == (8, 1)


@pytest.mark.parametrize("origin,steps,shape", [
    ([0.0, 0.0], [[1.0, 0.0, 0.0]], (4,)),                  # origin length
    ([0.0, 0.0, 0.0], [[1.0, 0.0]], (4,)),                  # steps width
    ([0.0, 0.0, 0.0], [1.0, 0.0, 0.0], (4,)),               # steps not 2-D
    ([0.0, 0.0, 0.0], np.zeros((0, 3)), ()),                # m = 0
    ([0.0, 0.0, 0.0], np.zeros((9, 3)), (1,) * 9),          # m = 9
    ([0.0, 0.0, 0.0], [[1.0, 0.0, 0.0]], (4, 4)),           # shape length
    ([0.0, 0.0, 0.0], [[1.0, 0.0, 0.0]], (-1,)),            # negative extent
    ([np.nan, 0.0, 0.0], [[1.0, 0.0, 0.0]], (4,)),
    ([0.0, 0.0, 0.0], [[-np.inf, 0.0, 0.0]], (4,)),
    ([1e308, 0.0, 0.0], [[1e308, 0.0, 0.0]], (4,)),         # the grid overflows to inf
    ([True, False, True], [[1.0, 0.0, 0.0]], (4,)),         # bool
    ([0.0, 0.0, 0.0], [[1j, 0.0, 0.0]], (4,)),              # complex
    (["a", "b", "c"], [[1.0, 0.0, 0.0]], (4,)),
], ids=["origin-len", "steps-width", "steps-1d", "m0", "m9", "shape-len", "negative", "nan", "inf", "overflow", "bool",
        "complex", "str"])
def test_grid_args_errors(origin, steps, shape):
    with pytest.raises(ValueError):
        _ops.grid_args(3, origin, steps, shape)


@pytest.mark.parametrize("shape", [(2.5,), (True,), ("4",)])
def test_grid_args_extents_must_be_integers(shape):
    with pytest.raises(TypeError):
        _ops.grid_args(3, [0.0, 0.0, 0.0], [[1.0, 0.0, 0.0]], shape)
