"""CPU-side checks of the hit-list entry points (sw_set_hits / sw_fetch_hits / sw_fetch_db_hits)."""
import ctypes as C


def test_hit_list_calls_reject_a_null_handle_and_count(pkg):
    lib = pkg.load_library()
    cnt = C.c_size_t(5)
    assert lib.sw_set_hits(None, 10, 100) == pkg.SW_EINVAL
    assert lib.sw_fetch_hits(None, None, None, None, 0, C.byref(cnt), -1) == pkg.SW_EINVAL
    assert lib.sw_fetch_db_hits(None, None, None, None, 0, C.byref(cnt)) == pkg.SW_EINVAL
    assert lib.sw_fetch_hits(None, None, None, None, 0, None, -1) == pkg.SW_EINVAL
    assert lib.sw_fetch_db_hits(None, None, None, None, 0, None) == pkg.SW_EINVAL
