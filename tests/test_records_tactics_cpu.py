"""gmz_records_tactics (missed-win flags of packed move records) validates its arguments before it touches the device:
no GPU is needed for these paths."""
import ctypes as C


def test_records_tactics_rejects_bad_arguments():
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    rec = (C.c_uint8 * 4096)()
    flags = (C.c_uint8 * 4)()
    bad = [
        (None, 1, 9, 5, flags),          # null records
        (rec, 1, 9, 5, None),            # null output
        (rec, 1, 0, 5, flags),           # board 0
        (rec, 1, 20, 5, flags),          # board above GMZ_MAX_BOARD
        (rec, 1, 9, 0, flags),           # n_in_row 0
        (rec, -1, 9, 5, flags),          # negative record count
    ]
    for args in bad:
        lib.gmz_set_roots(None, None, None, None, None, None)            # leaves a different message behind
        assert lib.gmz_records_tactics(*args, None) != 0, args
        assert b"gmz_records_tactics" in lib.gmz_last_error(), args


def test_records_tactics_zero_records_is_a_noop():
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    rec = (C.c_uint8 * 16)()
    flags = (C.c_uint8 * 4)(7, 7, 7, 7)
    assert lib.gmz_records_tactics(rec, 0, 15, 5, flags, None) == 0
    assert list(flags) == [7, 7, 7, 7]


def test_records_tactics_is_declared_and_bound():
    from datou_gomoku_muzero_b200 import _lib
    assert "gmz_records_tactics" in _lib.SIGNATURES
    assert _lib.load().gmz_version() == 200
