"""The CUDA VCT solver (k_vct, k_records_vct) against its CPU restatement (tests/csrc/vct_ref.c): length, first moves
and node counts exactly equal on random-play positions at test_vcf_gpu's board / row classes and on the hand-built
positions, under a budget that cuts, at batch sizes 1, odd and over 10,000; the VCF-within-VCT relations against
find_vcf; the record flags, missed_vct_counts and opening_vct built on it."""
import numpy as np
import pytest

import _vct_ref
from test_vcf_gpu import _random_positions, _selfplay_packs

pytestmark = pytest.mark.gpu


def _check(boards, players, N, n, max_attacks, budget):
    from datou_gomoku_muzero_b200.tactics import find_vct
    length, first, nodes = find_vct(boards, players, max_attacks, budget, n_in_row=n, board_size=N)
    rl, rf, rn = _vct_ref.solve(boards, players, N, n, max_attacks, budget)
    assert np.array_equal(length.cpu().numpy(), rl), (N, n)
    assert np.array_equal(first.cpu().numpy(), rf), (N, n)
    assert np.array_equal(nodes.cpu().numpy(), rn), (N, n)
    return rl, rf, rn


@pytest.mark.parametrize("N,n", [(1, 1), (5, 3), (5, 4), (6, 4), (6, 5), (9, 5), (13, 5), (15, 5), (15, 4), (19, 5),
                                 (19, 7), (9, 2)])
def test_random_positions_equal_the_reference(N, n):
    boards, players = _random_positions(N, 1001 if N > 1 else 5, seed=N * 37 + n)
    length, _, nodes = _check(boards, players, N, n, 8, 300)
    if N >= 6 and n == 5:
        assert (length > 1).any() and (length == 0).any() and nodes.max() > 1


def test_known_answer_positions_equal_the_reference():
    import test_vct_cpu as kat
    chain_X, chain_Y = [], [(1, 9), (7, 9)]
    for i, r in enumerate((2, 3, 4, 5)):
        s = 1 if i % 2 == 0 else -1
        chain_X += [(r, 9 + s * (2 + k)) for k in range(3)]
        chain_Y += [(r, 9 + s * 5)]
    rows15 = [(kat.DT, []), (kat.DT + [(3, 9)], []), (kat.DT + [(3, 9)], [(4, 9), (5, 9), (6, 9)]),
              (kat.DT, [(0, 0), (0, 1), (0, 2), (0, 3)]),
              (kat.DT + [(0, 4), (2, 9), (3, 9), (4, 9)], [(0, 5), (0, 6), (0, 7), (0, 8)]),
              ([(7, 5), (7, 6), (7, 8)], []), ([(7, 0), (7, 1)], [])]
    b15 = np.stack([kat._board(15, X, Y).reshape(-1) for X, Y in rows15])
    b19 = kat._board(19, chain_X, chain_Y).reshape(1, -1)
    for b, N in ((b15, 15), (b19, 19)):
        for players, bb in ((np.ones(len(b), np.int8), b), (-np.ones(len(b), np.int8), -b)):
            for L in (2, 3):
                _check(bb, players, N, 5, L, 200_000)
    for N, n, X in ((5, 3, [(2, 2)]), (6, 4, [(2, 2), (2, 3)]), (9, 7, [(4, 1), (4, 2), (4, 3), (4, 4), (4, 5)])):
        b = kat._board(N, X).reshape(1, -1)
        _check(b, [1], N, n, 8, 100_000)
        _check(-b, [-1], N, n, 8, 100_000)


def test_budget_cuts_a_share_of_positions():
    boards, players = _random_positions(15, 4001, seed=9, max_fill=0.5)
    length, _, nodes = _check(boards, players, 15, 5, 16, 40)
    assert (length == -1).sum() > 20 and (length >= 0).sum() > 20 and (nodes[length == -1] == 40).all()


def test_batch_sizes_one_odd_and_large():
    boards, players = _random_positions(15, 12_003, seed=4, max_fill=0.6)
    _check(boards[:1], players[:1], 15, 5, 8, 100)
    _check(boards[:777], players[:777], 15, 5, 8, 100)
    length, _, _ = _check(boards, players, 15, 5, 8, 100)
    assert (length > 0).sum() > 1000 and (length == -1).any()


def test_every_vcf_is_a_vct():
    """Where neither search is cut: a VCF within max_attacks gives a VCT no longer; with no completion cell and no F2
    at the root (VCT length != 2 there), every VCF first move is a VCT first move."""
    from datou_gomoku_muzero_b200.tactics import find_vcf, find_vct
    boards, players = _random_positions(15, 20_000, seed=12, max_fill=0.6)
    for L in (4, 8):
        vl, vf, _ = (t.cpu().numpy() for t in find_vcf(boards, players, L, 2000, n_in_row=5, board_size=15))
        tl, tf, _ = (t.cpu().numpy() for t in find_vct(boards, players, L, 2000, n_in_row=5, board_size=15))
        both = (vl >= 0) & (tl >= 0)
        assert (~both | (vl <= 0) | ((tl > 0) & (tl <= vl))).all()
        quiet = both & (vl > 1) & (tl != 2)
        assert not (vf & ~tf & quiet[:, None]).any()
        assert ((vl > 0) & both).sum() > 500 and ((vl == 0) & (tl > 0)).sum() > 10


def test_selfplay_records_flags_and_ring():
    """E0 self-play records: find_vct on their boards equals the reference; vct_record_flags equals find_vct plus the
    played action, from a packed block and from a wrapped DeviceReplayBuffer ring; missed_vct_counts equals a host
    recount."""
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.tactics import missed_vct_counts, vct_record_flags
    N, k, budget = 15, 8, 300
    A = N * N
    packs = _selfplay_packs(N, min_records=6000)
    want_flags, missed = [], 0
    for pg in packs:
        h = pg.host()
        boards, to_move, action = h["board"].reshape(-1, A), h["to_move"], h["action"].astype(np.int64)
        length, first, _ = _check(boards, to_move, N, 5, k, budget)
        played = first[np.arange(len(action)), np.clip(action, 0, A - 1)] & (action >= 0) & (action < A)
        f = ((length > 0) * 1 + played * 2 + (length < 0) * 4).astype(np.uint8)
        assert np.array_equal(vct_record_flags(pg.records, N, k, budget, 5).cpu().numpy(), f)
        want_flags.append(f)
        m = (f & 3) == 1
        per_game = np.add.reduceat(m.astype(np.int64), np.asarray(pg.offsets[:-1]) - pg.offsets[0]) if len(pg) else []
        assert np.array_equal(missed_vct_counts(pg, k, budget, 5).cpu().numpy(), per_game)
        missed += int(m.sum())
    flags = np.concatenate(want_flags)
    assert (flags & 1).sum() > 0 and missed > 0
    cap = 3001
    buf = DeviceReplayBuffer(cap, N)
    for pg in packs:
        buf.add_packed(pg)
    assert len(buf) == cap
    ring = vct_record_flags(buf.ring[:cap], N, k, budget, 5).cpu().numpy()
    start = len(flags) % cap                       # ring position of the oldest record kept
    assert np.array_equal(np.roll(ring, -start), flags[-cap:])


def test_opening_vct_equals_find_vct_and_covers_opening_vcf():
    from datou_gomoku_muzero_b200.arena import opening_vcf, opening_vct, random_openings
    from datou_gomoku_muzero_b200.tactics import find_vct
    book = random_openings(3000, 10, 15, seed=4)
    mover, opp = opening_vct(book, max_attacks=8, node_budget=3000)
    want_m = find_vct(book.boards, book.players, 8, 3000, n_in_row=5, board_size=15)[0].cpu().numpy()
    want_o = find_vct(book.boards, -book.players.astype(np.int64), 8, 3000, n_in_row=5, board_size=15)[0].cpu().numpy()
    assert np.array_equal(mover, want_m) and np.array_equal(opp, want_o)
    vm, vo = opening_vcf(book, max_attacks=8, node_budget=3000)
    for t, v in ((mover, vm), (opp, vo)):
        ok = (t >= 0) & (v >= 0)
        assert not (ok & (v > 0) & (t == 0)).any()
    assert ((mover != 0) | (opp != 0)).any() and ((mover == 0) & (opp == 0)).any()
