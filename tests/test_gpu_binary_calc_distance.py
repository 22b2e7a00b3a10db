"""b200vs_calc_distance_binary (VectorCalcDistance, METRIC_TYPE_HAMMING) against the CPU binary oracle."""
import numpy as np
import pytest

import b200vs
import oracle_binary_lib
from gpu_util import require_gpu

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dim", [8, 24, 64, 256, 1024, 4096, 32768])
def test_calc_distance_binary_parity(dim):
    require_gpu()
    bo = oracle_binary_lib.load()
    rng = np.random.default_rng(dim)
    left = rng.integers(0, 256, (13, dim // 8), dtype=np.uint8)
    right = rng.integers(0, 256, (29, dim // 8), dtype=np.uint8)
    right[:5] = left[:5]
    out = b200vs.calc_distance_binary(left, right)
    assert np.array_equal(out.view(np.uint32), bo.calc_distance(left, right).view(np.uint32))
    assert (np.diag(out[:5, :5]) == 0).all()


def test_calc_distance_binary_edges():
    require_gpu()
    x = np.zeros((3, 4), np.uint8)
    assert b200vs.calc_distance_binary(x[:0], x).shape == (0, 3)
    assert np.array_equal(b200vs.calc_distance_binary(x, np.full((1, 4), 0xFF, np.uint8)), np.full((3, 1), 32.0, np.float32))
    L = b200vs.lib()
    out = np.zeros(9, np.float32)
    for dim in (0, 12, 32776):
        assert L.b200vs_calc_distance_binary(0, dim, 3, x.ctypes.data, 3, x.ctypes.data, out.ctypes.data) == b200vs.EILLEGAL_PARAMETERS
