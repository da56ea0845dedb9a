"""CPU-side checks of sw_align_db: a null handle, null arrays and a null count are rejected before any device work."""
import ctypes as C

import numpy as np


def test_align_rejects_a_null_handle_arrays_and_count(pkg):
    lib = pkg.load_library()
    row = np.zeros(2, np.uint32)
    index = np.zeros(2, np.uint64)
    score = np.zeros(2, np.int32)
    coord = np.zeros(8, np.uint32)
    off = np.zeros(3, np.uint64)
    cigar = np.zeros(16, np.uint32)
    count = C.c_size_t(7)
    args = (row.ctypes.data, index.ctypes.data, 2, score.ctypes.data, coord.ctypes.data, off.ctypes.data,
            cigar.ctypes.data, 16, C.byref(count))
    assert lib.sw_align_db(None, *args) == pkg.SW_EINVAL
    assert lib.sw_align_db(None, None, None, 0, None, None, None, None, 0, None) == pkg.SW_EINVAL
    for k in (0, 1, 3, 4, 5, 6, 8):
        a = list(args)
        a[k] = None
        assert lib.sw_align_db(None, *a) == pkg.SW_EINVAL
    assert (score == 0).all() and (coord == 0).all() and (off == 0).all() and (cigar == 0).all() and count.value == 7


def test_cigar_str_text():
    import importlib
    pkg = importlib.import_module("smith-waterman-fpga-module_b200")
    assert pkg.cigar_str([]) == "*"
    assert pkg.cigar_str([23 << 4 | 7, 1 << 4 | 1, 24 << 4 | 7]) == "23=1I24="
    assert pkg.cigar_str(np.array([5 << 4 | 7, 2 << 4 | 2, 1 << 4 | 8, 3 << 4 | 7], np.uint32)) == "5=2D1X3="
