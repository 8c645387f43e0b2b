"""The VCT solver's definition (include/gmz.h gmz_vct_solve) pinned through its CPU restatement (tests/csrc/vct_ref.c):
the filtered mode the kernel's shortcuts follow equals brute force, hand-built positions give their expected results in
both colours, VCT never needs more stones than VCF, and both C entry points refuse bad arguments -- no GPU needed."""
import ctypes as C

import numpy as np
import pytest

import _vcf_ref
import _vct_ref
import test_vcf_cpu as vcf_kat


def _board(N, X=(), Y=()):
    b = np.zeros((N, N), np.int8)
    for r, c in X:
        b[r, c] = 1
    for r, c in Y:
        b[r, c] = -1
    return b


def _solve(N, X=(), Y=(), n_in_row=5, max_attacks=8, node_budget=1 << 20):
    """(length, first as a set of cells, nodes), the same for X as black and X as white (the colour-flipped copy)."""
    out = []
    for player in (1, -1):
        b = _board(N, X, Y) * np.int8(player)          # X is the side to move
        length, first, nodes = _vct_ref.solve(b[None], [player], N, n_in_row, max_attacks, node_budget)
        out.append((int(length[0]), {divmod(int(a), N) for a in np.flatnonzero(first[0])}, int(nodes[0])))
    assert out[0] == out[1]
    return out[0]


def _random_positions(N, B, seed, max_fill=0.6):
    rs = np.random.RandomState(seed)
    A = N * N
    boards = np.zeros((B, A), np.int8)
    players = np.ones(B, np.int8)
    k = rs.randint(0, max(1, int(A * max_fill)) + 1, size=B)
    order = np.argsort(rs.rand(B, A), axis=1)
    for i in range(B):
        cells = order[i, :k[i]]
        boards[i, cells[0::2]], boards[i, cells[1::2]] = 1, -1
        players[i] = 1 if k[i] % 2 == 0 else -1
    return boards, players


# Double three: (7,8) makes an open three on row 7 and one on column 8; no single Y stone stops both.
DT = [(7, 6), (7, 7), (5, 8), (6, 8)]


@pytest.mark.parametrize("N,n", [(5, 3), (5, 4), (6, 4), (6, 5), (7, 3), (7, 4), (7, 5), (8, 3), (8, 4), (8, 5)])
def test_filtered_equals_brute_force(N, n):
    boards, players = _random_positions(N, 300, seed=N * 13 + n)
    for L, budget in ((3, 200), (6, 300)):
        f = _vct_ref.solve(boards, players, N, n, L, budget, filtered=True)
        b = _vct_ref.solve(boards, players, N, n, L, budget, filtered=False)
        for x, y in zip(f, b):
            assert np.array_equal(x, y), (N, n, L)
    length = f[0]
    assert (length > 1).any() and (length == 0).any()


def test_filtered_sets_equal_brute_force():
    """X's threat moves where X has no completion cell; Y's replies where, besides, Y has none and F2 is not empty
    (the root then answers length 2 without a search)."""
    boards, _ = _random_positions(8, 300, seed=5, max_fill=0.4)
    replies = 0
    for n in (3, 4, 5):
        length = _vct_ref.solve(boards, np.ones(len(boards), np.int8), 8, n, 2, 1)[0]
        for b, ln in zip(boards.reshape(-1, 8, 8), length):
            if ln == 1:
                continue
            f, r = _vct_ref.sets(b, n, True), _vct_ref.sets(b, n, False)
            assert f[0] == r[0]
            if ln == 2:
                assert f[1] == r[1]
                replies += 1
    assert replies > 50


def test_double_three_is_three_stones():
    length, first, nodes = _solve(15, DT)
    assert length == 3 and (7, 8) in first and nodes > 1
    assert _solve(15, DT, max_attacks=2)[:2] == (0, set())
    assert _vcf_ref.solve(_board(15, DT)[None], [1], 15, 5, 8)[0][0] == 0          # no four in sight


def test_broken_three_defences_include_the_gap():
    """X's broken three on row 7 (gap at (7,7)): its only F2 cell is the gap, so Y's defences are the gap and both
    ends of the four the gap would make."""
    _, replies = _vct_ref.sets(_board(15, [(7, 5), (7, 6), (7, 8)]))
    assert replies == {(7, 4), (7, 7), (7, 9)}
    _, replies = _vct_ref.sets(_board(15, [(7, 5), (7, 6), (7, 7)]))          # a solid open three: the two ends
    assert replies == {(7, 4), (7, 8)}


def test_three_against_the_edge_is_no_threat():
    threats, _ = _vct_ref.sets(_board(15, [(7, 0), (7, 1)]))
    assert threats == set()
    threats, _ = _vct_ref.sets(_board(15, [(7, 5), (7, 6)]))
    assert threats == {(7, 3), (7, 4), (7, 7), (7, 8)}


def test_counter_four_that_gains_tempo_refutes_the_double_three():
    """Y's column 9 (rows 4-6, closed by X at (3,9)) turns (7,9), an end of the row-7 three, into a four: X must block
    at (8,9) and Y then stops the column three.  Within 3 stones the double three at (7,8) no longer wins."""
    Yc = [(4, 9), (5, 9), (6, 9)]
    assert _vct_ref.sets(_board(15, DT + [(3, 9), (7, 8)], Yc))[1] == {(7, 9), (8, 9)}
    length, first, _ = _solve(15, DT + [(3, 9)], max_attacks=3)
    assert length == 3 and (7, 8) in first
    length, first, _ = _solve(15, DT + [(3, 9)], Yc, max_attacks=3)
    assert length == 0 and (7, 8) not in first


def test_defender_four_forces_the_block():
    # the block at (0,4) makes no threat: the root has no candidate
    assert _solve(15, DT, [(0, 0), (0, 1), (0, 2), (0, 3)]) == (0, set(), 1)
    # the block at (0,9) is a four on column 9: the only first move
    length, first, _ = _solve(15, DT + [(0, 4), (2, 9), (3, 9), (4, 9)], [(0, 5), (0, 6), (0, 7), (0, 8)])
    assert length == 3 and first == {(0, 9)}


def test_longer_chain_needs_the_attack_budget():
    """test_vcf_cpu's chain of four blocked threes: a VCF of 4 stones, a VCT of 3; 2 stones find nothing."""
    X, Y = [], [(1, 9), (7, 9)]
    for i, r in enumerate((2, 3, 4, 5)):
        s = 1 if i % 2 == 0 else -1
        X += [(r, 9 + s * (2 + k)) for k in range(3)]
        Y += [(r, 9 + s * 5)]
    assert _solve(19, X, Y, max_attacks=2)[:2] == (0, set())
    l3, f3, _ = _solve(19, X, Y, max_attacks=3)
    assert l3 == 3 and f3
    assert _vcf_ref.solve(_board(19, X, Y)[None], [1], 19, 5, 3)[0][0] == 0


def test_budget_cut():
    assert _solve(15, DT, node_budget=3) == (-1, set(), 3)
    full = _solve(15, DT, max_attacks=3)
    assert _solve(15, DT, max_attacks=3, node_budget=full[2]) == full           # exactly enough is no cut
    assert _solve(15, DT, max_attacks=3, node_budget=full[2] - 1)[0] == -1


@pytest.mark.parametrize("N,n,X,want", [
    # n = 3: every neighbour of the lone stone makes an open two, which is already an open four
    (5, 3, [(2, 2)], (2, {(r, c) for r in range(1, 4) for c in range(1, 4) if (r, c) != (2, 2)})),
    (6, 4, [(0, 0), (0, 1), (0, 2)], (1, {(0, 3)})),
    (6, 4, [(2, 2), (2, 3)], (2, {(2, 1), (2, 4)})),
    (9, 7, [(4, 0), (4, 1), (4, 2), (4, 3), (4, 4), (4, 5)], (1, {(4, 6)})),
    (9, 7, [(4, 1), (4, 2), (4, 3), (4, 4), (4, 5)], (2, {(4, 6)})),
])
def test_other_row_lengths(N, n, X, want):
    assert _solve(N, X, n_in_row=n)[:2] == want


def test_vct_never_longer_than_vcf():
    """On test_vcf_cpu's positions: a VCF within max_attacks is a VCT no longer; with no completion cell and no F2 at
    the root, every VCF first move is a VCT first move."""
    rows = [(vcf_kat.X3, vcf_kat.Y3), (vcf_kat.X3 + [(2, 7)], vcf_kat.Y3 + [(3, 7), (4, 7), (5, 7)]),
            ([(7, 4), (7, 5), (7, 6)], []), ([(0, 1), (0, 2), (0, 3)], []), ([(7, 3), (7, 4), (7, 5), (7, 6)], []),
            (vcf_kat.X3, vcf_kat.Y3 + [(0, 0), (0, 1), (0, 2), (0, 3)]),
            ([(7, 4), (7, 5), (7, 6)], [(2, 2), (2, 3), (2, 4), (2, 5)])]
    boards = np.stack([_board(15, X, Y).reshape(-1) for X, Y in rows])
    p = np.ones(len(rows), np.int8)
    for L in (2, 3, 8):
        vl, vf, _ = _vcf_ref.solve(boards, p, 15, 5, L, 1 << 20)
        tl, tf, _ = _vct_ref.solve(boards, p, 15, 5, L, 1 << 20)
        assert ((vl <= 0) | ((tl > 0) & (tl <= vl))).all(), (L, vl, tl)
        for i in range(len(rows)):
            if vl[i] > 1 and tl[i] != 2:
                assert not (vf[i] & ~tf[i]).any(), (L, i)
    boards, players = _random_positions(9, 400, seed=2)
    vl, vf, _ = _vcf_ref.solve(boards, players, 9, 5, 6, 400)
    tl, tf, _ = _vct_ref.solve(boards, players, 9, 5, 6, 400)
    both = (vl >= 0) & (tl >= 0)
    assert (~both | (vl <= 0) | ((tl > 0) & (tl <= vl))).all()
    assert ((vl > 0) & (tl > 0)).sum() > 20


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
        assert lib.gmz_vct_solve(*args, None) != 0, args
        assert b"gmz_vct_solve" in lib.gmz_last_error(), args
    records_bad = [
        (None, 1, 9, 5, 8, 100, flags), (rec, 1, 9, 5, 8, 100, None), (rec, 1, 0, 5, 8, 100, flags),
        (rec, 1, 20, 5, 8, 100, flags), (rec, 1, 9, 0, 8, 100, flags), (rec, 1, 9, 5, 0, 100, flags),
        (rec, 1, 9, 5, 33, 100, flags), (rec, 1, 9, 5, 8, 0, flags), (rec, -1, 9, 5, 8, 100, flags),
        (rec, 1 << 31, 9, 5, 8, 100, flags),
    ]
    for args in records_bad:
        lib.gmz_set_roots(None, None, None, None, None, None)
        assert lib.gmz_records_vct(*args, None) != 0, args
        assert b"gmz_records_vct" in lib.gmz_last_error(), args


def test_empty_batches_are_noops():
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    ln = (C.c_int32 * 1)(7)
    flags = (C.c_uint8 * 2)(7, 7)
    assert lib.gmz_vct_solve((C.c_int8 * 1)(), (C.c_int8 * 1)(), 0, 15, 5, 8, 100, ln, (C.c_uint64 * 6)(),
                             (C.c_int32 * 1)(), None) == 0
    assert lib.gmz_records_vct((C.c_uint8 * 16)(), 0, 15, 5, 8, 100, flags, None) == 0
    assert list(ln) == [7] and list(flags) == [7, 7]
    assert {"gmz_vct_solve", "gmz_records_vct"} <= set(_lib.SIGNATURES)


def test_reference_refuses_what_the_library_refuses():
    b = np.zeros((1, 25), np.int8)
    for kw in ({"max_attacks": 0}, {"max_attacks": 33}, {"node_budget": 0}, {"n_in_row": 0}):
        with pytest.raises(ValueError):
            _vct_ref.solve(b, [1], 5, **{"n_in_row": 5, **kw})
