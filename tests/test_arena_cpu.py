"""Match statistics, opening books and the match entry points' argument checks, without a GPU."""
import ctypes as C
import math

import numpy as np
import pytest


def _synthetic(pair_points, rs):
    """A finished match whose opening o gave A `pair_points[o]` points (0, 0.5, ..., 2) over its two games."""
    from datou_gomoku_muzero_b200.arena import MatchResult, empty_opening
    O = len(pair_points)
    res = np.zeros((2 * O, 4), np.int32)
    colour = rs.choice([-1, 1], O)
    res[0::2, 3], res[1::2, 3] = colour, -colour
    res[0::2, 2], res[1::2, 2] = 0, 1
    res[:, 1] = rs.randint(5, 30, 2 * O)
    for o, pts in enumerate(pair_points):
        splits = [(x, y) for x in (0, 0.5, 1) for y in (0, 0.5, 1) if x + y == pts]
        for t, s in zip((2 * o, 2 * o + 1), splits[rs.randint(len(splits))]):
            c = res[t, 3]
            res[t, 0] = 0 if s == 0.5 else (c if s == 1 else -c)
    return MatchResult(res, np.full((2 * O, 36), -1, np.int32), empty_opening(6), 6)


@pytest.mark.parametrize("probs", [(0.05, 0.2, 0.4, 0.25, 0.1), (0.3, 0.1, 0.2, 0.1, 0.3), (0.0, 0.0, 0.3, 0.5, 0.2)])
def test_elo_interval_and_los_match_scipy(probs):
    from scipy import stats
    rs = np.random.RandomState(int(probs[0] * 100 + probs[4] * 10))
    pts = rs.choice([0, 0.5, 1, 1.5, 2], 400, p=probs)
    r = _synthetic(pts, rs)
    assert np.array_equal(r.pairs(), np.array([(pts == v).sum() for v in (0, 0.5, 1, 1.5, 2)]))
    x = pts / 2.0
    s = x.mean()
    se = np.sqrt(((x - s) ** 2).mean() / x.size)
    z = stats.norm.ppf(0.975)

    def elo(p):
        return -400.0 * np.log10(1.0 / p - 1.0)
    st = r.elo()
    assert st["pairs"] == 400
    assert st["score"] == pytest.approx(s, rel=1e-12) and r.score() == pytest.approx(s, rel=1e-12)
    assert st["elo"] == pytest.approx(elo(s), rel=1e-9, abs=1e-9)
    assert st["elo_lo"] == pytest.approx(elo(s - z * se), rel=1e-9)
    assert st["elo_hi"] == pytest.approx(elo(s + z * se), rel=1e-9)
    assert st["los"] == pytest.approx(stats.norm.cdf((s - 0.5) / se), rel=1e-9, abs=1e-12)
    w, d, l = r.wdl()
    assert w + d + l == 800 and (w + 0.5 * d) / 800 == pytest.approx(s, rel=1e-12)
    wb, db, lb = r.wdl(1)
    ww, dw, lw = r.wdl(-1)
    assert (wb + ww, db + dw, lb + lw) == (w, d, l)


def test_elo_edge_cases():
    from datou_gomoku_muzero_b200.arena import elo_stats
    st = elo_stats(np.full(10, 0.5))
    assert st["elo"] == 0.0 and st["elo_lo"] == 0.0 and st["elo_hi"] == 0.0 and st["los"] == 0.5
    st = elo_stats(np.ones(10))
    assert st["elo"] == math.inf and st["los"] == 1.0
    st = elo_stats(np.zeros(3))
    assert st["elo"] == -math.inf and st["los"] == 0.0
    assert math.isnan(elo_stats([])["score"])


def test_unfinished_games_are_left_out():
    from datou_gomoku_muzero_b200.arena import MatchResult, empty_opening
    res = np.array([[1, 9, 0, 1], [2, 0, 1, -1], [0, 36, 0, 1], [-1, 12, 1, -1]], np.int32)
    r = MatchResult(res, np.full((4, 36), -1, np.int32), empty_opening(6), 6)
    assert len(r) == 3 and r.wdl() == (2, 1, 0)
    assert np.array_equal(r.pair_scores(), [0.75]) and np.array_equal(r.pairs(), [0, 0, 0, 1, 0])
    with pytest.raises(ValueError):
        r.game_record(1)


def test_game_record_replays_the_moves():
    from datou_gomoku_muzero_b200.arena import MatchResult, Openings
    N = 6
    op = Openings(np.zeros((1, N * N), np.int8), np.array([-1], np.int8), np.array([-1], np.int32), np.array([0], np.int32))
    moves = np.full((2, N * N), -1, np.int32)
    moves[0, :7] = [0, 6, 1, 7, 2, 8, 3]                  # white (first mover) plays 0, 1, 2, 3: four in a row
    res = np.array([[-1, 7, 0, -1], [2, 0, 1, 1]], np.int32)
    rec = MatchResult(res, moves, op, N, 4).game_record(0)
    assert rec.actions == [0, 6, 1, 7, 2, 8, 3] and rec.rewards[-1] == 1.0 and rec.rewards[-2] == -1.0
    assert rec.board_states[-1][0, :3].tolist() == [-1, -1, -1] and rec.board_states[0].sum() == 0
    assert rec.observations[1][2, 0, 0] == 1.0 and rec.observations[1][1, 0, 0] == 1.0      # black to move sees white's stone
    assert all(p.argmax() == a and p.sum() == 1.0 for p, a in zip(rec.policies, rec.actions))


def _book(N, **change):
    from datou_gomoku_muzero_b200.arena import Openings
    A = N * N
    b = np.zeros((2, A), np.int8)
    b[1, 0], b[1, 1] = 1, -1
    d = dict(boards=b, players=np.array([1, 1], np.int8), last_moves=np.array([-1, 1], np.int32),
             move_counts=np.array([0, 2], np.int32))
    d.update(change)
    return Openings(**d)


def test_opening_validation():
    from datou_gomoku_muzero_b200.arena import check_openings
    N, A = 6, 36
    ok = check_openings(_book(N), N, 4)
    assert ok.boards.dtype == np.int8 and ok.boards.shape == (2, A)
    assert check_openings(None, N, 4).boards.shape == (1, A)
    check_openings(_book(N, boards=np.zeros((2, N, N), np.int8)), N, 4)          # [O, N, N] boards are accepted
    bad = []
    b = np.zeros((2, A), np.int8); b[0, 3] = 2
    bad.append(_book(N, boards=b))                                                   # value outside {-1, 0, 1}
    bad.append(_book(N, players=np.array([1, 0], np.int8)))                          # side to move 0
    bad.append(_book(N, boards=np.zeros((2, 25), np.int8)))                          # board shape
    bad.append(_book(N, boards=np.zeros((0, A), np.int8), players=np.zeros(0, np.int8), last_moves=np.zeros(0, np.int32),
                     move_counts=np.zeros(0, np.int32)))                             # no opening
    bad.append(_book(N, players=np.ones(3, np.int8)))                                # length mismatch
    bad.append(_book(N, last_moves=np.array([-1, A], np.int32)))                     # last move off the board
    full = np.where(np.arange(A) % 3 == 0, 1, -1).astype(np.int8)
    bad.append(_book(N, boards=np.stack([full, full]), move_counts=np.array([A - 1, A - 1], np.int32),
                     last_moves=np.array([-1, -1], np.int32)))                       # no empty cell
    bad.append(_book(N, move_counts=np.array([0, 1], np.int32)))                     # fewer moves than stones
    b = np.zeros((2, A), np.int8); b[1, :4] = 1; b[1, 6:9] = -1
    bad.append(_book(N, boards=b, last_moves=np.array([-1, 3], np.int32), move_counts=np.array([0, 7], np.int32)))   # won
    b = np.zeros((2, A), np.int8); b[1, :A - 1] = np.where(np.arange(A - 1) % 3 == 0, 1, -1)
    bad.append(_book(N, boards=b, last_moves=np.array([-1, -1], np.int32), move_counts=np.array([0, A], np.int32)))  # drawn
    for book in bad:
        with pytest.raises(ValueError):
            check_openings(book, N, 4)


@pytest.mark.parametrize("stones", [0, 1, 4, 9])
def test_random_openings(stones):
    from datou_gomoku_muzero_b200.arena import check_openings, random_openings
    N = 9
    op = random_openings(50, stones, N, seed=stones, n_in_row=4)
    check_openings(op, N, 4)
    assert ((op.boards == 1).sum(1) == (stones + 1) // 2).all() and ((op.boards == -1).sum(1) == stones // 2).all()
    assert (op.players == (1 if stones % 2 == 0 else -1)).all() and (op.move_counts == stones).all()
    if stones:
        assert (op.boards[np.arange(50), op.last_moves] == -op.players).all()
        rows, cols = np.nonzero(op.boards.reshape(50, N, N))[1:]
        assert (abs(rows - N // 2) <= 4).all() and (abs(cols - N // 2) <= 4).all()
    assert np.array_equal(random_openings(50, stones, N, seed=stones, n_in_row=4).boards, op.boards)
    with pytest.raises(ValueError):
        random_openings(1, N * N, N)


def test_match_entry_points_reject_bad_handles_without_crashing():
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    bogus, other = C.c_void_p(0x1000), C.c_void_p(0x2000)
    m = _lib.GmzMatch()
    for a, b, mm in ((None, None, None), (bogus, other, C.byref(m)), (None, bogus, C.byref(m))):
        assert lib.gmz_match_start(a, b, mm, None) != 0 and b"handle" in lib.gmz_last_error()
        assert lib.gmz_match_noise(a, b, mm, 0, None, None, None) != 0 and lib.gmz_last_error()
        assert lib.gmz_match_step(a, b, mm, None, None, None) != 0 and lib.gmz_last_error()
