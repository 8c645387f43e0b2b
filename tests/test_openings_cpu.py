"""Self-play opening books without a GPU: gmz_set_openings refuses bad arguments with a message, and the packed record
header's `opening` label sits at bytes 56..59 (include/gmz.h gmz_move_record)."""
import ctypes as C

import numpy as np


def _book(n, arrays=True):
    from datou_gomoku_muzero_b200._lib import GmzOpenings
    keep = [(C.c_int8 * 4)(), (C.c_int8 * 1)(1), (C.c_int32 * 1)(-1), (C.c_int32 * 1)(0)]
    ptrs = [C.addressof(x) if arrays else None for x in keep]
    return GmzOpenings(n, 0, *ptrs), keep


def _refuses(lib, handle, book, needle):
    rc = lib.gmz_set_openings(handle, C.byref(book) if book is not None else None, None)
    msg = lib.gmz_last_error().decode()
    assert rc != 0 and needle in msg, (rc, msg)


def test_set_openings_refuses_bad_arguments():
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    dead = C.c_void_p(0x1000)                       # never created: not a live handle
    good, k1 = _book(1)
    _refuses(lib, dead, good, "invalid or destroyed engine handle")
    _refuses(lib, dead, None, "invalid or destroyed engine handle")      # unbinding checks the handle too
    _refuses(lib, None, good, "invalid or destroyed engine handle")
    for n in (0, -3):
        bad, k2 = _book(n)
        _refuses(lib, dead, bad, "n_openings must be >= 1")
    nulls, k3 = _book(1, arrays=False)
    _refuses(lib, dead, nulls, "null array")
    for i, field in enumerate(("boards", "players", "last_moves", "move_counts")):
        one, k4 = _book(2)
        setattr(one, field, None)
        _refuses(lib, dead, one, "null array")


def test_record_dtype_opening_label_offset():
    from datou_gomoku_muzero_b200.trajectory import PackedGames, record_dtype
    for N in (6, 15):
        dt = record_dtype(N)
        assert dt.fields["opening"][1] == 56 and dt.fields["opening"][0] == np.dtype("<i4")
        assert dt.fields["slot"][1] == 52 and dt.fields["policy"][1] == 64
        stride = dt.itemsize
        raw = np.zeros((5, stride), np.uint8)
        for r, lab in enumerate((3, 3, 0, 7, 7)):
            raw[r, 56:60] = np.frombuffer(np.int32(lab).tobytes(), np.uint8)
        pg = PackedGames(raw, np.zeros((3, 4), np.int32), [0, 2, 3, 5], N)
        assert pg.host()["opening"].tolist() == [3, 3, 0, 7, 7]
        assert pg.openings().tolist() == [2, -1, 6] and pg.openings().dtype == np.int32


def test_set_openings_in_the_ctypes_table():
    from datou_gomoku_muzero_b200 import _lib
    assert _lib.SIGNATURES["gmz_set_openings"][1][1]._type_ is _lib.GmzOpenings
    names = [f[0] for f in _lib.GmzTraj._fields_]
    assert names[-1] == "start_opening" and _lib.GmzTraj.start_opening.offset == 88
    assert [f[0] for f in _lib.GmzOpenings._fields_] == ["n_openings", "reserved", "boards", "players", "last_moves",
                                                        "move_counts"]
