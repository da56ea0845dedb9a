"""CPU-side checks of sw_locate_db: a null handle and null arrays are rejected before any device work."""
import numpy as np


def test_locate_rejects_a_null_handle_and_arrays(pkg):
    lib = pkg.load_library()
    row = np.zeros(2, np.uint32)
    index = np.zeros(2, np.uint64)
    score = np.zeros(2, np.int32)
    coord = np.zeros(8, np.uint32)
    args = (row.ctypes.data, index.ctypes.data, 2, score.ctypes.data, coord.ctypes.data)
    assert lib.sw_locate_db(None, *args) == pkg.SW_EINVAL
    assert lib.sw_locate_db(None, None, None, 0, None, None) == pkg.SW_EINVAL
    for k in (0, 1, 3, 4):
        a = list(args)
        a[k] = None
        assert lib.sw_locate_db(None, *a) == pkg.SW_EINVAL
    assert (score == 0).all() and (coord == 0).all()
