"""CPU checks of solve_many's shape limits: they are decided from (m, n) before any device is touched, so a shape the
kernels cannot run fails the same way with or without a GPU."""
import os

import numpy as np
import pytest

import lp_b200
from lp_b200 import _ffi


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_ffi.LIB_PATH):
        from lp_b200 import build
        build.build(verbose=False)
    return _ffi.load()


def _zeros(batch, m, n):
    return np.zeros((batch, m, n)), np.zeros((batch, m)), np.zeros((batch, n))


def test_more_than_128_rows_is_refused(lib):
    with pytest.raises(lp_b200.InvalidParameter, match=r"m <= 128"):
        lp_b200.solve_many(*_zeros(1, 129, 200))


def test_shared_memory_footprint_over_227_kb_is_refused(lib):
    # M of 128 x 129 doubles and ten n-vectors: n = 1000 needs ~233 KB
    with pytest.raises(lp_b200.InvalidParameter, match=r"227 KB"):
        lp_b200.solve_many(*_zeros(1, 128, 1000))
    with pytest.raises(lp_b200.InvalidParameter, match=r"227 KB"):
        lp_b200.solve_many(*_zeros(1, 2, 3000))


def test_mismatched_shapes(lib):
    A, b, c = _zeros(2, 8, 16)
    with pytest.raises(lp_b200.IncompatibleInputDimensions):
        lp_b200.solve_many(A, b[:, :7], c)
    with pytest.raises(lp_b200.IncompatibleInputDimensions):
        lp_b200.solve_many(A, b, c[:1])
    with pytest.raises(lp_b200.IncompatibleInputDimensions):
        lp_b200.solve_many(A[0], b[0], c[0])


def test_largest_shapes_pass_the_limits(lib):
    """(128, 768) and (64, 1024) are inside the limits: without a GPU they get as far as the device check."""
    if lib.lpb_device_count() > 0:
        pytest.skip("a GPU is visible")
    for m, n in [(128, 768), (64, 1024), (1, 2)]:
        with pytest.raises(lp_b200.api.DeviceError) as e:
            lp_b200.solve_many(*_zeros(1, m, n))
        assert e.value.code == _ffi.LPB_ERR_NO_DEVICE
