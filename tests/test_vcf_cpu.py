"""The VCF solver's definition (include/gmz.h gmz_vcf_solve) pinned on hand-built positions through its CPU restatement
(tests/csrc/vcf_ref.c), and the argument checks of both C entry points, which need no GPU."""
import ctypes as C

import numpy as np
import pytest

import _vcf_ref


def _board(N, X=(), Y=()):
    b = np.zeros((N, N), np.int8)
    for r, c in X:
        b[r, c] = 1
    for r, c in Y:
        b[r, c] = -1
    return b


def _solve(N, X=(), Y=(), n_in_row=5, max_attacks=8, node_budget=1 << 20, player=1):
    b = _board(N, X, Y) * np.int8(player)          # X is the side to move
    length, first, nodes = _vcf_ref.solve(b[None], [player], N, n_in_row, max_attacks, node_budget)
    return int(length[0]), {divmod(int(a), N) for a in np.flatnonzero(first[0])}, int(nodes[0])


# Attacker: a blocked three on row 7 and two on column 8 / row 6 -- (6,8) is a four on row 6 whose forced reply is
# (6,7), after which (7,8) makes two fours at once (row 7 towards (7,7), column 8 towards (8,8)): three stones.
X3 = [(7, 4), (7, 5), (7, 6), (4, 8), (5, 8), (6, 9), (6, 10), (6, 11)]
Y3 = [(7, 3), (3, 8), (6, 12)]


def test_immediate_five_and_overline():
    assert _solve(15, [(7, 3), (7, 4), (7, 5), (7, 6)]) == (1, {(7, 2), (7, 7)}, 1)
    # freestyle: the stone at (7,4) makes six in a row, which wins
    assert _solve(15, [(7, 2), (7, 3), (7, 5), (7, 6), (7, 7)]) == (1, {(7, 4)}, 1)
    # the side to move is what counts, not the colour
    assert _solve(15, [(7, 3), (7, 4), (7, 5), (7, 6)], player=-1)[:2] == (1, {(7, 2), (7, 7)})


def test_open_four_is_two_stones():
    length, first, _ = _solve(15, [(7, 4), (7, 5), (7, 6)])
    assert (length, first) == (2, {(7, 3), (7, 7)})
    assert _solve(15, [(7, 4), (7, 5), (7, 6)], max_attacks=1)[:2] == (0, set())


def test_three_stone_vcf():
    length, first, nodes = _solve(15, X3, Y3)
    assert length == 3 and {(6, 8), (7, 8)} <= first and nodes > 1
    assert _solve(15, X3, Y3, max_attacks=2)[:2] == (0, set())
    # without the column stones there is no double four to reach
    assert _solve(15, X3[:3] + X3[5:], Y3)[0] == 0


def test_longer_vcf_needs_the_attack_budget():
    """Four blocked threes around column 9, closed at both ends: the fewest attacker stones the reference finds is 4;
    a smaller max_attacks finds none, a larger one the same length."""
    X, Y = [], [(1, 9), (7, 9)]
    for i, r in enumerate((2, 3, 4, 5)):
        s = 1 if i % 2 == 0 else -1
        X += [(r, 9 + s * (2 + k)) for k in range(3)]
        Y += [(r, 9 + s * 5)]
    assert _solve(19, X, Y, max_attacks=3)[0] == 0
    l4, f4, _ = _solve(19, X, Y, max_attacks=4)
    l8, f8, _ = _solve(19, X, Y, max_attacks=8)
    assert l4 == l8 == 4 and f4 <= f8 and (5, 9) in f4


def test_defender_five_refutes_the_attack():
    """The defender already has a four: the attacker's only candidate is to block it, which is no four here, so the
    three-stone VCF above is refuted and the search stops at the root."""
    assert _solve(15, X3, Y3 + [(0, 0), (0, 1), (0, 2), (0, 3)]) == (0, set(), 1)


def test_defender_two_completion_cells():
    assert _solve(15, [(7, 4), (7, 5), (7, 6)], [(2, 2), (2, 3), (2, 4), (2, 5)]) == (0, set(), 1)


def test_counter_four_must_be_answered_with_a_four():
    """The defender's column (3..5, 7) turns its forced reply at (6,7) or (7,7) into a four: the attacker's next stone
    must block, and only a block that is itself a four keeps the attack going."""
    Xc, Yc = X3 + [(2, 7)], Y3 + [(3, 7), (4, 7), (5, 7)]
    length, first, nodes = _solve(15, Xc, Yc)
    base_len, base_first, base_nodes = _solve(15, X3, Y3)
    assert length == 3 and (6, 8) not in first and first < base_first
    # the counter-four costs the branch through (6,8): every VCF left starts on row 6 / 7 next to the column
    assert first == {(6, 7), (7, 7), (7, 8)}


def test_lines_at_the_board_edge():
    assert _solve(15, [(0, 0), (0, 1), (0, 2), (0, 3)]) == (1, {(0, 4)}, 1)
    length, first, _ = _solve(15, [(0, 1), (0, 2), (0, 3)])
    assert (length, first) == (2, {(0, 4)})            # (0,0) leaves one completion cell, (0,4) two
    assert _solve(15, [(14, 11), (14, 12), (14, 13), (14, 14)])[:2] == (1, {(14, 10)})
    assert _solve(15, [(10, 14), (11, 13), (12, 12), (13, 11)])[:2] == (1, {(14, 10)})     # (9, 15) is off the board


@pytest.mark.parametrize("N,n,X,want", [
    # the 8 neighbours make two completion cells at once; the 8 cells two steps away force the cell between and win next
    (5, 3, [(2, 2)], (2, {(r, c) for r in range(5) for c in range(5)
                          if (r, c) != (2, 2) and (max(abs(r - 2), abs(c - 2)) == 1 or (r % 2 == 0 and c % 2 == 0))})),
    (6, 4, [(0, 0), (0, 1), (0, 2)], (1, {(0, 3)})),
    (9, 7, [(4, 0), (4, 1), (4, 2), (4, 3), (4, 4), (4, 5)], (1, {(4, 6)})),
    (9, 7, [(4, 0), (4, 1), (4, 2), (4, 4), (4, 5), (4, 6), (4, 7)], (1, {(4, 3)})),
    (1, 1, [], (1, {(0, 0)})),
    (3, 4, [(1, 0), (1, 1)], (0, set())),
])
def test_other_row_lengths(N, n, X, want):
    assert _solve(N, X, n_in_row=n)[:2] == want


def test_budget_cut():
    length, first, nodes = _solve(15, X3, Y3, node_budget=3)
    assert (length, first, nodes) == (-1, set(), 3)
    full = _solve(15, X3, Y3)
    assert _solve(15, X3, Y3, node_budget=full[2]) == full        # exactly enough is no cut


def test_full_board_is_no_vcf():
    N = 3
    b = np.array([[1, -1, 1], [1, -1, -1], [-1, 1, 0]], np.int8)
    length, first, nodes = _vcf_ref.solve(b[None], [1], N, 3, 8, 100)
    assert (int(length[0]), int(first.sum()), int(nodes[0])) == (0, 0, 1)


def test_entry_points_reject_bad_arguments():
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    b, p = (C.c_int8 * 64)(), (C.c_int8 * 1)(1)
    ln, nd, fs = (C.c_int32 * 1)(), (C.c_int32 * 1)(), (C.c_uint64 * 6)()
    rec, flags = (C.c_uint8 * 4096)(), (C.c_uint8 * 4)()
    solve_bad = [
        (None, p, 1, 8, 5, 8, 100, ln, fs, nd), (b, None, 1, 8, 5, 8, 100, ln, fs, nd),
        (b, p, 1, 8, 5, 8, 100, None, fs, nd), (b, p, 1, 8, 5, 8, 100, ln, None, nd), (b, p, 1, 8, 5, 8, 100, ln, fs, None),
        (b, p, 1, 0, 5, 8, 100, ln, fs, nd), (b, p, 1, 20, 5, 8, 100, ln, fs, nd), (b, p, 1, 8, 0, 8, 100, ln, fs, nd),
        (b, p, 1, 8, 5, 0, 100, ln, fs, nd), (b, p, 1, 8, 5, 33, 100, ln, fs, nd), (b, p, 1, 8, 5, 8, 0, ln, fs, nd),
        (b, p, -1, 8, 5, 8, 100, ln, fs, nd),
    ]
    for args in solve_bad:
        lib.gmz_set_roots(None, None, None, None, None, None)            # leaves a different message behind
        assert lib.gmz_vcf_solve(*args, None) != 0, args
        assert b"gmz_vcf_solve" in lib.gmz_last_error(), args
    records_bad = [
        (None, 1, 9, 5, 8, 100, flags), (rec, 1, 9, 5, 8, 100, None), (rec, 1, 0, 5, 8, 100, flags),
        (rec, 1, 20, 5, 8, 100, flags), (rec, 1, 9, 0, 8, 100, flags), (rec, 1, 9, 5, 0, 100, flags),
        (rec, 1, 9, 5, 33, 100, flags), (rec, 1, 9, 5, 8, 0, flags), (rec, -1, 9, 5, 8, 100, flags),
    ]
    for args in records_bad:
        lib.gmz_set_roots(None, None, None, None, None, None)
        assert lib.gmz_records_vcf(*args, None) != 0, args
        assert b"gmz_records_vcf" in lib.gmz_last_error(), args


def test_empty_batches_are_noops():
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    ln = (C.c_int32 * 1)(7)
    flags = (C.c_uint8 * 2)(7, 7)
    assert lib.gmz_vcf_solve((C.c_int8 * 1)(), (C.c_int8 * 1)(), 0, 15, 5, 8, 100, ln, (C.c_uint64 * 6)(),
                             (C.c_int32 * 1)(), None) == 0
    assert lib.gmz_records_vcf((C.c_uint8 * 16)(), 0, 15, 5, 8, 100, flags, None) == 0
    assert list(ln) == [7] and list(flags) == [7, 7]
    assert {"gmz_vcf_solve", "gmz_records_vcf"} <= set(_lib.SIGNATURES)


def test_reference_refuses_what_the_library_refuses():
    b = np.zeros((1, 25), np.int8)
    for kw in ({"max_attacks": 0}, {"max_attacks": 33}, {"node_budget": 0}, {"n_in_row": 0}):
        with pytest.raises(ValueError):
            _vcf_ref.solve(b, [1], 5, **{"n_in_row": 5, **kw})
