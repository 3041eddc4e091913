"""CPU: host-side contract of the streaming tensor-core InfoNCE head (dib_infonce_head_tc): its scratch is O(n d) and
out-of-range arguments are refused before anything reaches a device."""
import ctypes


def test_scratch_is_linear_in_n_and_small_at_the_metric_batch():
    from dib_b200 import _lib
    lib = _lib.load()
    assert lib.dib_infonce_head_tc_scratch_bytes(65536, 64) < 64 * 2**20
    assert lib.dib_infonce_head_tc_scratch_bytes(2 * 65536, 64) == 2 * lib.dib_infonce_head_tc_scratch_bytes(65536, 64)
    assert lib.dib_infonce_head_tc_scratch_bytes(1, 1) > 0
    for n, d in ((0, 64), (65536, 0), (65536, 257), (2**26 + 1, 64)):
        assert lib.dib_infonce_head_tc_scratch_bytes(n, d) == -1, (n, d)


def test_bad_arguments_are_refused():
    from dib_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(256)
    for kind, n, d, T in ((2, 8, 4, 1.0), (3, 8, 4, 1.0), (0, 0, 4, 1.0), (1, 8, 257, 1.0), (4, 8, 4, 0.0)):
        assert lib.dib_infonce_head_tc(kind, p, p, n, d, T, p, p, None, None, None) != 0
        assert b"dib_infonce_head_tc" in lib.dib_last_error()
    assert lib.dib_infonce_head_tc(0, p, p, 8, 4, 1.0, ctypes.c_void_p(256 + 64), p, None, None, None) != 0
    assert b"aligned" in lib.dib_last_error()
