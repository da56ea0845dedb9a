"""CPU-side checks of the per-subject best entry points (sw_set_subject_best / sw_fetch_subject_best /
sw_fetch_db_subject_best)."""
import numpy as np


def test_subject_best_calls_reject_a_null_handle_and_arrays(pkg):
    lib = pkg.load_library()
    bs = np.zeros(4, np.int32)
    br = np.zeros(4, np.uint32)
    sec = np.zeros(4, np.int32)
    assert lib.sw_set_subject_best(None, 1) == pkg.SW_EINVAL
    assert lib.sw_set_subject_best(None, 0) == pkg.SW_EINVAL
    assert lib.sw_fetch_subject_best(None, bs.ctypes.data, br.ctypes.data, sec.ctypes.data, 4, -1) == pkg.SW_EINVAL
    assert lib.sw_fetch_db_subject_best(None, bs.ctypes.data, br.ctypes.data, sec.ctypes.data, 4) == pkg.SW_EINVAL
    assert lib.sw_fetch_subject_best(None, None, None, None, 0, -1) == pkg.SW_EINVAL
    assert lib.sw_fetch_db_subject_best(None, None, None, None, 0) == pkg.SW_EINVAL
