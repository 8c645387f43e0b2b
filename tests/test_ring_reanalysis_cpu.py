"""The re-analysis entry points of the replay ring (gmz_set_roots_from_records, gmz_records_writeback,
gmz_records_retarget) validate their arguments before they touch the device: no GPU is needed for these paths."""
import ctypes as C

NAMES = ("gmz_set_roots_from_records", "gmz_records_writeback", "gmz_records_retarget")


def _lib():
    from datou_gomoku_muzero_b200 import _lib
    return _lib.load()


def _check_rejected(lib, name, args, what):
    lib.gmz_set_roots(None, None, None, None, None, None)            # leaves a different message behind
    assert getattr(lib, name)(*args) != 0, (name, what)
    msg = lib.gmz_last_error()
    assert name.encode() in msg, (name, what, msg)
    return msg


def test_writeback_and_retarget_reject_bad_arguments():
    lib = _lib()
    ring = (C.c_uint8 * 8192)()
    pol = (C.c_double * 256)()
    val = (C.c_double * 4)()
    dpow = (C.c_double * 11)()
    # (capacity, board_size, first, n) cases shared by both entry points
    bad = [
        ((4, 0, 0, 1), b"board_size"), ((4, 20, 0, 1), b"board_size"), ((0, 6, 0, 1), b"capacity"),
        ((4, 6, 0, -1), b"n must"), ((4, 6, 4, 1), b"first"), ((4, 6, -1, 1), b"first"), ((4, 6, 0, 5), b"capacity"),
    ]
    for (cap, N, first, n), what in bad:
        assert what in _check_rejected(lib, "gmz_records_writeback", (ring, cap, N, first, n, pol, val, None), what)
        assert what in _check_rejected(lib, "gmz_records_retarget", (ring, cap, N, first, n, dpow, 10, None), what)
    for args in [(None, 4, 6, 0, 1, pol, val, None), (ring, 4, 6, 0, 1, None, val, None), (ring, 4, 6, 0, 1, pol, None, None)]:
        assert b"null" in _check_rejected(lib, "gmz_records_writeback", args, "null")
    for args in [(None, 4, 6, 0, 1, dpow, 10, None), (ring, 4, 6, 0, 1, None, 10, None)]:
        assert b"null" in _check_rejected(lib, "gmz_records_retarget", args, "null")
    assert b"n_steps" in _check_rejected(lib, "gmz_records_retarget", (ring, 4, 6, 0, 1, dpow, -1, None), "n_steps")


def test_set_roots_from_records_rejects_bad_arguments():
    """Without a live engine every call fails; the ring arguments are checked first, each with its own message.
    (n > num_games needs a live engine: tests/test_ring_reanalysis_gpu.py.)"""
    lib = _lib()
    ring = (C.c_uint8 * 8192)()
    name = "gmz_set_roots_from_records"
    assert b"null" in _check_rejected(lib, name, (None, None, 4, 0, 1, None), "null ring")
    assert b"capacity" in _check_rejected(lib, name, (None, ring, 0, 0, 1, None), "capacity")
    assert b"n must" in _check_rejected(lib, name, (None, ring, 4, 0, -1, None), "n < 0")
    assert b"first" in _check_rejected(lib, name, (None, ring, 4, 4, 1, None), "first")
    assert b"first" in _check_rejected(lib, name, (None, ring, 4, -1, 1, None), "first")
    assert b"engine" in _check_rejected(lib, name, (None, ring, 4, 0, 1, None), "null engine")
    assert b"engine" in _check_rejected(lib, name, (None, ring, 4, 0, 0, None), "null engine, n = 0")


def test_zero_records_is_a_noop():
    lib = _lib()
    ring = (C.c_uint8 * 4096)(*([7] * 4096))
    pol, val, dpow = (C.c_double * 36)(), (C.c_double * 1)(), (C.c_double * 11)()
    assert lib.gmz_records_writeback(ring, 4, 6, 3, 0, pol, val, None) == 0
    assert lib.gmz_records_retarget(ring, 4, 6, 3, 0, dpow, 10, None) == 0
    assert list(ring) == [7] * 4096


def test_symbols_are_declared_and_bound():
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    for n in NAMES:
        assert n in _lib.SIGNATURES and hasattr(lib, n)
    assert lib.gmz_version() == 200
