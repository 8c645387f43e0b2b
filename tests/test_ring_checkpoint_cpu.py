"""Checkpoint of the device replay ring without a GPU: gmz_records_compact / gmz_records_expand validate their arguments
before they touch the device, and validate_ring_state rejects every malformed state dict on the host."""
import ctypes as C

import numpy as np
import pytest
import torch


def _lib():
    from datou_gomoku_muzero_b200 import _lib
    return _lib.load()


def _check_rejected(lib, name, args, what):
    lib.gmz_set_roots(None, None, None, None, None, None)            # leaves a different message behind
    assert getattr(lib, name)(*args) != 0, (name, what)
    msg = lib.gmz_last_error()
    assert name.encode() in msg, (name, what, msg)
    return msg


def test_compact_rejects_bad_arguments():
    lib = _lib()
    name = "gmz_records_compact"
    ring, hd, pol, fl = (C.c_uint8 * 8192)(), (C.c_uint8 * 256)(), (C.c_double * 256)(), (C.c_uint8 * 4)()
    bad = [((4, 0, 0, 1), b"board_size"), ((4, 20, 0, 1), b"board_size"), ((0, 6, 0, 1), b"capacity"),
           ((4, 6, 0, -1), b"n must"), ((4, 6, 4, 1), b"first"), ((4, 6, -1, 1), b"first"), ((4, 6, 0, 5), b"capacity")]
    for (cap, N, first, n), what in bad:
        assert what in _check_rejected(lib, name, (ring, cap, N, first, n, hd, pol, fl, None), what)
    for i in range(4):
        args = [ring, 4, 6, 0, 1, hd, pol, fl, None]
        args[(0, 5, 6, 7)[i]] = None
        assert b"null" in _check_rejected(lib, name, tuple(args), "null")


def test_expand_rejects_bad_arguments():
    lib = _lib()
    name = "gmz_records_expand"
    ring, hd, pol = (C.c_uint8 * 8192)(), (C.c_uint8 * 256)(), (C.c_double * 256)()
    seg, base = (C.c_int64 * 4)(), (C.c_int8 * 256)()

    def args(n=2, n_seg=1, skip=0, N=6, cap=4, first=0, **null):
        a = dict(headers=hd, policy=pol, seg_start=seg, base_boards=base, ring=ring)
        a.update(null)
        return (a["headers"], a["policy"], n, a["seg_start"], a["base_boards"], n_seg, skip, N, a["ring"], cap, first, None)
    cases = [(dict(N=0), b"board_size"), (dict(N=20), b"board_size"), (dict(cap=0), b"capacity"), (dict(n=-1), b"n must"),
             (dict(skip=-1), b"skip"), (dict(skip=3), b"skip"), (dict(n=6, skip=1), b"capacity"), (dict(first=4), b"first"),
             (dict(first=-1), b"first"), (dict(n_seg=0), b"n_seg"), (dict(n_seg=3), b"n_seg")]
    for kw, what in cases:
        assert what in _check_rejected(lib, name, args(**kw), what)
    for key in ("headers", "policy", "seg_start", "base_boards", "ring"):
        assert b"null" in _check_rejected(lib, name, args(**{key: None}), key)


def test_zero_records_is_a_noop():
    lib = _lib()
    ring = (C.c_uint8 * 4096)(*([7] * 4096))
    hd, pol, fl = (C.c_uint8 * 64)(*([5] * 64)), (C.c_double * 36)(), (C.c_uint8 * 1)(9)
    seg, base = (C.c_int64 * 1)(), (C.c_int8 * 36)()
    assert lib.gmz_records_compact(ring, 4, 6, 3, 0, hd, pol, fl, None) == 0
    assert lib.gmz_records_expand(hd, pol, 0, seg, base, 0, 0, 6, ring, 4, 3, None) == 0
    assert list(ring) == [7] * 4096 and list(hd) == [5] * 64 and fl[0] == 9


def test_symbols_are_declared_and_bound():
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    for n in ("gmz_records_compact", "gmz_records_expand"):
        assert n in _lib.SIGNATURES and hasattr(lib, n)
    assert lib.gmz_version() == 200


# ---- host validation of a state dict
N, CAP = 6, 10
GAMES = [(3, 5), (0, 4), (0, 4)]          # (first t, length): a cut oldest game, then two whole games


def _state(**over):
    """A valid state dict of a full ring of CAP records (write_ptr 3), built by hand."""
    from datou_gomoku_muzero_b200.replay_buffer import RING_STATE_FORMAT, RING_STATE_VERSION
    A = N * N
    t = np.concatenate([np.arange(t0, T) for t0, T in GAMES]).astype(np.int32)
    T = np.concatenate([np.full(T - t0, T) for t0, T in GAMES]).astype(np.int32)
    h = np.zeros((CAP, 16), np.int32)
    h[:, 1], h[:, 2], h[:, 5] = t, T, np.where(t % 2 == 0, 1, -1)
    sd = {"format": RING_STATE_FORMAT, "version": RING_STATE_VERSION, "board_size": N, "capacity": CAP, "count": CAP,
          "write_ptr": 3, "headers": torch.from_numpy(h.view(np.uint8).reshape(CAP, 64).copy()),
          "policies": torch.zeros((CAP, A), dtype=torch.float64), "seg_start": torch.tensor([0, 2, 6]),
          "base_boards": torch.zeros((3, A), dtype=torch.int8), "tree": torch.zeros(2 * CAP - 1, dtype=torch.float64),
          "max_priority": torch.tensor(1.0, dtype=torch.float64)}
    if "seg_start" in over and "base_boards" not in over:       # a wrong segment table, not a wrong shape
        sd["base_boards"] = torch.zeros((len(over["seg_start"]), A), dtype=torch.int8)
    sd.update(over)
    return sd


def _with_t(t=None, T=None):
    h = _state()["headers"].clone()
    v = h.numpy().view(np.int32)
    if t is not None:
        v[:, 1] = t
    if T is not None:
        v[:, 2] = T
    return h


def test_validator_accepts_a_valid_state():
    from datou_gomoku_muzero_b200.replay_buffer import validate_ring_state
    assert validate_ring_state(_state(), N) == 3
    empty = _state(count=0, write_ptr=0, headers=torch.zeros((0, 64), dtype=torch.uint8),
                   policies=torch.zeros((0, N * N), dtype=torch.float64), seg_start=torch.zeros(0, dtype=torch.int64),
                   base_boards=torch.zeros((0, N * N), dtype=torch.int8))
    assert validate_ring_state(empty, N) == 0
    part = _state(count=6, write_ptr=6, headers=_state()["headers"][4:], policies=torch.zeros((6, N * N), dtype=torch.float64),
                  seg_start=torch.tensor([0, 2]), base_boards=torch.zeros((2, N * N), dtype=torch.int8))
    assert validate_ring_state(part, N) == 2


T0 = np.array([3, 4, 0, 1, 2, 3, 0, 1, 2, 3])


@pytest.mark.parametrize("what,over", [
    ("tag", dict(format="something_else")),
    ("version", dict(version=2)),
    ("board size", dict(board_size=9)),
    ("board_size type", dict(board_size=6.0)),
    ("count > capacity", dict(count=CAP + 1)),
    ("write_ptr >= capacity", dict(write_ptr=CAP)),
    ("write_ptr < 0", dict(write_ptr=-1)),
    ("write_ptr != count in a ring that is not full", dict(count=9, write_ptr=3)),
    ("headers dtype", dict(headers=torch.zeros((CAP, 16), dtype=torch.int32))),
    ("headers shape", dict(headers=torch.zeros((CAP, 48), dtype=torch.uint8))),
    ("headers not a tensor", dict(headers=np.zeros((CAP, 64), np.uint8))),
    ("policies dtype", dict(policies=torch.zeros((CAP, N * N), dtype=torch.float32))),
    ("policies shape", dict(policies=torch.zeros((CAP, 81), dtype=torch.float64))),
    ("seg_start dtype", dict(seg_start=torch.tensor([0, 2, 6], dtype=torch.int32))),
    ("base_boards shape", dict(base_boards=torch.zeros((2, N * N), dtype=torch.int8))),
    ("base_boards dtype", dict(base_boards=torch.zeros((3, N * N), dtype=torch.uint8))),
    ("base_boards stone value", dict(base_boards=torch.full((3, N * N), 2, dtype=torch.int8))),
    ("tree length", dict(tree=torch.zeros(2 * CAP, dtype=torch.float64))),
    ("tree dtype", dict(tree=torch.zeros(2 * CAP - 1, dtype=torch.float32))),
    ("max_priority", dict(max_priority=1.0)),
    ("seg_start misses a game start", dict(seg_start=torch.tensor([0, 2]))),
    ("seg_start has an extra start", dict(seg_start=torch.tensor([0, 2, 4, 6]))),
    ("seg_start without k = 0", dict(seg_start=torch.tensor([2, 6]))),
    ("t skips inside a segment", dict(headers=_with_t(t=np.where(np.arange(CAP) == 4, 3, T0)))),
    ("t >= length", dict(headers=_with_t(t=T0 + np.where(np.arange(CAP) < 2, 2, 0)))),
    ("t < 0", dict(headers=_with_t(t=np.where(np.arange(CAP) == 0, -1, T0)))),
    ("length changes inside a segment", dict(headers=_with_t(T=np.array([5, 5, 4, 4, 4, 4, 4, 4, 5, 5])))),
    ("game cut before its last move", dict(headers=_with_t(T=np.array([5, 5, 4, 4, 4, 4, 5, 5, 5, 5])))),
])
def test_validator_rejects(what, over):
    from datou_gomoku_muzero_b200.replay_buffer import validate_ring_state
    with pytest.raises(ValueError):
        validate_ring_state(_state(**over), N)


def test_validator_rejects_a_non_dict():
    from datou_gomoku_muzero_b200.replay_buffer import validate_ring_state
    with pytest.raises(ValueError):
        validate_ring_state([("format", "x")], N)
