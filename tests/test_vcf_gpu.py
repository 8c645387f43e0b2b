"""The CUDA VCF solver (k_vcf, k_records_vcf) against its CPU restatement (tests/csrc/vcf_ref.c): length, first moves
and node counts exactly equal on random-play positions at every board size class, on E0 self-play records, under a
budget that cuts, and at batch sizes 1, odd and 100,000; the record flags, SelfPlayStats counters and opening_vcf built
on it."""
import numpy as np
import pytest

import _vcf_ref

pytestmark = pytest.mark.gpu


def _random_positions(N, B, seed, max_fill=0.6):
    """B random-play boards (alternating stones from black, a random number of them) and the side to move."""
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


def _check(boards, players, N, n, max_attacks, budget):
    from datou_gomoku_muzero_b200.tactics import find_vcf
    length, first, nodes = find_vcf(boards, players, max_attacks, budget, n_in_row=n, board_size=N)
    rl, rf, rn = _vcf_ref.solve(boards, players, N, n, max_attacks, budget)
    assert np.array_equal(length.cpu().numpy(), rl), (N, n)
    assert np.array_equal(first.cpu().numpy(), rf), (N, n)
    assert np.array_equal(nodes.cpu().numpy(), rn), (N, n)
    return rl, rf, rn


@pytest.mark.parametrize("N,n", [(1, 1), (5, 3), (5, 4), (6, 4), (6, 5), (9, 5), (13, 5), (15, 5), (15, 4), (19, 5),
                                 (19, 7), (9, 2)])
def test_random_positions_equal_the_reference(N, n):
    boards, players = _random_positions(N, 3001 if N > 1 else 5, seed=N * 31 + n)
    length, _, nodes = _check(boards, players, N, n, 8, 5000)
    if N >= 6 and n == 5:
        assert (length > 1).any() and (length == 0).any() and nodes.max() > 1


def test_known_answer_positions_equal_the_reference():
    import test_vcf_cpu as kat
    N = 15
    rows = [(kat.X3, kat.Y3), (kat.X3 + [(2, 7)], kat.Y3 + [(3, 7), (4, 7), (5, 7)]), ([(7, 4), (7, 5), (7, 6)], []),
            ([(0, 1), (0, 2), (0, 3)], []), (kat.X3, kat.Y3 + [(0, 0), (0, 1), (0, 2), (0, 3)])]
    boards = np.stack([kat._board(N, X, Y).reshape(-1) for X, Y in rows])
    for players, b in ((np.ones(len(rows), np.int8), boards), (-np.ones(len(rows), np.int8), -boards)):
        for L in (2, 3, 8, 32):
            _check(b, players, N, 5, L, 1 << 20)


def test_budget_cuts_a_share_of_positions():
    boards, players = _random_positions(15, 4001, seed=7, max_fill=0.7)
    length, _, nodes = _check(boards, players, 15, 5, 16, 12)
    assert (length == -1).sum() > 20 and (length >= 0).sum() > 20 and (nodes[length == -1] == 12).all()


def test_batch_sizes_one_odd_and_large():
    boards, players = _random_positions(15, 100_003, seed=3, max_fill=0.5)
    _check(boards[:1], players[:1], 15, 5, 8, 2000)
    _check(boards[:777], players[:777], 15, 5, 8, 2000)
    length, _, _ = _check(boards, players, 15, 5, 8, 2000)
    assert (length > 0).sum() > 1000


def test_consistent_with_the_one_move_classifier():
    """Every FIVE cell starts a one-stone VCF; every OPEN_FOUR cell starts one of two stones when the mover has no
    five and the opponent no completion cell."""
    import torch
    from datou_gomoku_muzero_b200.tactics import FIVE, OPEN_FOUR, classify_boards, find_vcf
    N = 15
    boards, players = _random_positions(N, 20_000, seed=11, max_fill=0.5)
    cls = classify_boards(boards, players, N, n_in_row=5)
    length, first, _ = find_vcf(boards, players, 8, 5000, n_in_row=5, board_size=N)
    has_five = (cls == FIVE).any(1)
    assert torch.equal(has_five, length == 1)
    assert not ((cls == FIVE) & ~first).any()
    _, opp_first, _ = find_vcf(boards, -players.astype(np.int64), 1, 1, n_in_row=5, board_size=N)
    # the opponent's one-stone VCFs are its completion cells; a budget cut reports no first moves
    quiet = ~has_five & ~opp_first.any(1) & (length >= 0)
    assert not ((cls == OPEN_FOUR) & ~first & quiet[:, None]).any()
    assert ((cls == OPEN_FOUR) & quiet[:, None]).sum() > 100


def _selfplay_packs(N=15, G=256, min_records=20_000):
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng = SearchEngine(G, board_size=N, num_simulations=32)
    sp = SelfPlayEngine(eng, "e0", seed=5, noise_seed=6)
    traj = TrajectoryStore(eng, extra_slots=G)
    packs = []
    while sum(p.n_moves for p in packs) < min_records:
        sp.play(moves_per_game=N * N, traj=traj, sink=packs.append)
    return packs


def test_selfplay_records_flags_stats_and_ring():
    """E0 self-play records (rich in fours late in games): find_vcf on their boards equals the reference; the record
    flags equal find_vcf plus the played action, from a packed block and from a wrapped DeviceReplayBuffer ring;
    missed_vcf_counts and SelfPlayStats(vcf_attacks=k) equal a host recount."""
    import torch
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.tactics import SelfPlayStats, find_vcf, missed_vcf_counts, vcf_record_flags
    N, k, budget = 15, 8, 4000
    A = N * N
    packs = _selfplay_packs(N)
    stats = SelfPlayStats(n_in_row=5, vcf_attacks=k, vcf_budget=budget)
    plain = SelfPlayStats(n_in_row=5)
    want_flags, avail, missed, unknown = [], 0, 0, 0
    for pg in packs:
        torch.cuda.set_sync_debug_mode("error")
        try:
            stats.add(pg)
        finally:
            torch.cuda.set_sync_debug_mode(0)
        plain.add(pg)
        h = pg.host()
        boards, to_move, action = h["board"].reshape(-1, A), h["to_move"], h["action"].astype(np.int64)
        length, first, _ = _check(boards, to_move, N, 5, k, budget)
        played = first[np.arange(len(action)), np.clip(action, 0, A - 1)] & (action >= 0) & (action < A)
        f = ((length > 0) * 1 + played * 2 + (length < 0) * 4).astype(np.uint8)
        assert np.array_equal(vcf_record_flags(pg.records, N, k, budget, 5).cpu().numpy(), f)
        want_flags.append(f)
        m = (f & 3) == 1
        per_game = np.add.reduceat(m.astype(np.int64), np.asarray(pg.offsets[:-1]) - pg.offsets[0]) if len(pg) else []
        assert np.array_equal(missed_vcf_counts(pg, k, budget, 5).cpu().numpy(), per_game)
        avail += int((f & 1).sum()); missed += int(m.sum()); unknown += int((f >> 2 & 1).sum())
    s = stats.summary()
    assert (s["vcf_available"], s["missed_vcf"], s["vcf_unknown"]) == (avail, missed, unknown)
    assert s["missed_vcf_per_game"] == missed / s["games"] and avail > 0 and missed > 0
    assert set(plain.summary()) == set(s) - {"vcf_available", "missed_vcf", "missed_vcf_per_game", "vcf_unknown"}
    # a ring smaller than the records: the last `cap` records, wrapped around the end of the ring
    flags = np.concatenate(want_flags)
    cap = 7001
    buf = DeviceReplayBuffer(cap, N)
    for pg in packs:
        buf.add_packed(pg)
    assert len(buf) == cap
    ring = vcf_record_flags(buf.ring[:cap], N, k, budget, 5).cpu().numpy()
    start = len(flags) % cap                       # ring position of the oldest record kept
    assert np.array_equal(np.roll(ring, -start), flags[-cap:])


def test_opening_vcf_equals_find_vcf_on_both_sides():
    from datou_gomoku_muzero_b200.arena import opening_vcf, random_openings
    from datou_gomoku_muzero_b200.tactics import find_vcf
    book = random_openings(3000, 13, 15, seed=4)
    mover, opp = opening_vcf(book, max_attacks=8, node_budget=3000)
    want_m = find_vcf(book.boards, book.players, 8, 3000, n_in_row=5, board_size=15)[0].cpu().numpy()
    want_o = find_vcf(book.boards, -book.players.astype(np.int64), 8, 3000, n_in_row=5, board_size=15)[0].cpu().numpy()
    assert np.array_equal(mover, want_m) and np.array_equal(opp, want_o)
    assert ((mover != 0) | (opp != 0)).any() and ((mover == 0) & (opp == 0)).any()
