"""Missed-win statistics of device self-play (workers.py:191-203) from packed move records: gmz_records_tactics pinned to
the reference's classifier KATs, per-game counts equal to missed_win_stats over GameRecords, the side to move taken from
the record header, every board size, the network evaluator, and SelfPlayStats accumulation without a host sync."""
import os

import numpy as np
import pytest

from _golden_util import GOLDEN_DIR

pytestmark = pytest.mark.gpu


def _expected_flags(pg, n_in_row):
    """The flag byte of every record of `pg`, from classify_boards on the record boards for the header's to_move."""
    from datou_gomoku_muzero_b200.tactics import classify_boards
    h = pg.host()
    N, M = pg.N, pg.n_moves
    A = N * N
    cls = classify_boards(h["board"].reshape(M, A), h["to_move"], N, n_in_row=n_in_row).cpu().numpy()
    a = h["action"].astype(np.int64)
    ok = (a >= 0) & (a < A)
    played = np.where(ok, cls[np.arange(M), np.clip(a, 0, A - 1)], 0)
    return ((cls > 0).any(1) * 1 + (cls == 1).any(1) * 2 + (played > 0) * 4).astype(np.uint8)


def _flags(pg, n_in_row):
    from datou_gomoku_muzero_b200.tactics import record_flags
    return record_flags(pg.records, pg.N, n_in_row).cpu().numpy()


def _selfplay(N, G, S, n_in_row=5, min_games=64, moves=24, evaluator="e0", roots=None, max_rounds=40, **eng_kw):
    """Packed chunks of persistent self-play until at least `min_games` games have finished."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng = SearchEngine(G, board_size=N, n_in_row=n_in_row, num_simulations=S, **eng_kw)
    sp = SelfPlayEngine(eng, evaluator, seed=11, noise_seed=12) if isinstance(evaluator, str) else SelfPlayEngine(eng, evaluator, noise_seed=12)
    if roots is not None:
        eng.set_roots(*roots)
    traj = TrajectoryStore(eng, extra_slots=G)
    packs = []
    for _ in range(max_rounds):
        sp.play(moves_per_game=moves, traj=traj, sink=packs.append)
        if sum(len(p) for p in packs) >= min_games:
            break
    assert sum(len(p) for p in packs) >= min_games
    return packs


def _record_block(N, rows):
    """Device records [len(rows), stride] built with trajectory.record_dtype: rows of (board, to_move, action)."""
    import torch
    from datou_gomoku_muzero_b200.trajectory import record_dtype
    r = np.zeros(len(rows), record_dtype(N))
    for i, (b, p, a) in enumerate(rows):
        r[i]["board"] = np.asarray(b, np.int8).reshape(N, N)
        r[i]["to_move"], r[i]["action"] = p, a
    return torch.from_numpy(r.view(np.uint8).reshape(len(rows), -1).copy()).cuda()


def test_record_flags_match_reference_kat():
    """Every KAT board (9x9, 15x15) as a record: played once on a cell of each class present and once on an empty
    class-0 cell (plus actions outside the board).  The bits are what the reference's classes imply."""
    from datou_gomoku_muzero_b200.tactics import record_flags
    z = np.load(os.path.join(GOLDEN_DIR, "tactics_kat.npz"))
    seen = set()
    for N in (9, 15):
        A = N * N
        rows, want = [], []
        for i in np.flatnonzero(z["N"] == N):
            b, p, cls = z["boards"][i][:A], int(z["player"][i]), z["cls"][i][:A]
            base = int((cls > 0).any()) | 2 * int((cls == 1).any())
            for k in (1, 2, 3):
                cells = np.flatnonzero(cls == k)
                if len(cells):
                    rows.append((b, p, int(cells[len(cells) // 2]))); want.append(base | 4)
            quiet = np.flatnonzero((b == 0) & (cls == 0))
            if len(quiet):
                rows.append((b, p, int(quiet[0]))); want.append(base)
            for a in (-1, A):
                rows.append((b, p, a)); want.append(base)
        got = record_flags(_record_block(N, rows), N, n_in_row=5).cpu().numpy()
        assert np.array_equal(got, np.array(want, np.uint8)), N
        seen |= set(got.tolist())
    assert {0, 1, 3, 5, 7} <= seen          # no win; missed combo / four; missed five; played win; played five


@pytest.mark.parametrize("N,G", [(9, 64), (15, 96)])
def test_missed_win_counts_equal_missed_win_stats_from_reset(N, G):
    """Persistent E0 self-play from reset: the per-game counts from the records equal the host restatement over each
    game's GameRecord (move parity = to_move here)."""
    from datou_gomoku_muzero_b200.tactics import missed_win_counts, missed_win_stats
    packs = _selfplay(N, G, 16, moves=N * N // 4)
    allc = []
    for pg in packs:
        got = missed_win_counts(pg).cpu().numpy()
        assert got.shape == (len(pg), 2) and got.dtype == np.int64
        for i in range(len(pg)):
            assert tuple(got[i]) == missed_win_stats(pg.game_record(i)), (N, i)
        assert np.array_equal(_flags(pg, 5), _expected_flags(pg, 5))
        allc.append(got)
    c = np.concatenate(allc)
    assert (c == 0).any() and (c > 0).any() and c[:, 1].sum() > 0 and (c[:, 0] <= c[:, 1]).all()


def test_mid_game_starts_take_the_colour_from_the_header():
    """Games started from set_roots positions with white to move: the flags follow classify_boards for the header's
    to_move, which differs from move parity for these games."""
    N, G = 15, 64
    A = N * N
    rs = np.random.RandomState(5)
    boards = np.zeros((G, A), np.int8)
    last = np.zeros(G, np.int32)
    mc = np.zeros(G, np.int32)
    for g in range(G):
        k = 2 * int(rs.randint(4, 20)) + 1               # odd number of stones: white to move
        cells = rs.permutation(A)[:k]
        boards[g, cells[0::2]], boards[g, cells[1::2]] = 1, -1
        last[g], mc[g] = cells[-1], k
    packs = _selfplay(N, G, 16, min_games=48, moves=12, roots=(boards, -np.ones(G, np.int8), last, mc))
    mid = 0
    for pg in packs:
        h = pg.host()
        first = h[pg.offsets[:-1]]
        mid += int(((first["to_move"] == -1) & (first["move_count"] > 0)).sum())
        assert np.array_equal(_flags(pg, 5), _expected_flags(pg, 5))
    assert mid >= 16


@pytest.mark.parametrize("N,n_in_row", [(19, 5), (6, 4)])
def test_other_board_shapes(N, n_in_row):
    packs = _selfplay(N, 32, 12, n_in_row=n_in_row, min_games=8, moves=min(N * N // 3, 48))
    for pg in packs:
        assert np.array_equal(_flags(pg, n_in_row), _expected_flags(pg, n_in_row))


def test_network_selfplay_counts():
    """SelfPlayEngine(eng, GomokuNetEZ).play(sink=...) at 6x6: per-game counts equal missed_win_stats."""
    import torch
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.network import GomokuNetEZ
    from datou_gomoku_muzero_b200.tactics import missed_win_counts, missed_win_stats
    torch.manual_seed(0)
    net = GomokuNetEZ(Config(BOARD_SIZE=6, ACTION_SPACE_SIZE=36, NUM_RES_BLOCKS=1, NUM_FILTERS=16, HEAD_HIDDEN_DIM=8)).cuda().eval()
    packs = _selfplay(6, 32, 12, min_games=32, moves=36, evaluator=net, max_rounds=2, accum_dtype="float32")
    n = 0
    for pg in packs:
        got = missed_win_counts(pg).cpu().numpy()
        for i in range(len(pg)):
            assert tuple(got[i]) == missed_win_stats(pg.game_record(i)), i
            n += 1
    assert n >= 32


def test_selfplay_stats_accumulate_without_a_host_sync():
    """SelfPlayStats over a multi-chunk play(sink=...) equals the sums over every packed game; add() runs under
    sync-debug mode "error".  The same records in the replay ring give the same flags."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.tactics import SelfPlayStats, missed_win_counts, record_flags
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    N, G = 9, 64
    eng = SearchEngine(G, board_size=N, num_simulations=16)
    sp = SelfPlayEngine(eng, "e0", seed=3, noise_seed=4)
    traj = TrajectoryStore(eng, extra_slots=G // 2)
    stats = SelfPlayStats(n_in_row=5)
    buf = DeviceReplayBuffer(20_000, N)
    packs = []

    def add(pg):
        torch.cuda.set_sync_debug_mode("error")
        try:
            stats.add(pg)
        finally:
            torch.cuda.set_sync_debug_mode(0)

    sp.play(moves_per_game=120, traj=traj, sink=lambda pg: (add(pg), buf.add_packed(pg), packs.append(pg)))
    assert len(packs) >= 3
    s = stats.summary()
    wins = np.concatenate([p.table[:, 3] for p in packs])
    counts = torch.cat([missed_win_counts(p) for p in packs]).sum(0).tolist()
    assert s["games"] == sum(len(p) for p in packs) == len(wins)
    assert s["moves"] == sum(p.n_moves for p in packs) == len(buf)
    assert (s["wins_black"], s["wins_white"], s["draws"]) == (int((wins == 1).sum()), int((wins == -1).sum()), int((wins == 0).sum()))
    assert [s["missed_fives"], s["missed_all_wins"]] == counts and counts[1] > 0
    assert s["avg_game_length"] == s["moves"] / s["games"]
    ring = record_flags(buf.ring[:len(buf)], N, 5).cpu().numpy()
    assert np.array_equal(ring, np.concatenate([_flags(p, 5) for p in packs]))
    stats.reset()
    assert stats.summary()["games"] == 0 and stats.summary()["missed_all_wins"] == 0


def test_empty_packed_games_launch_nothing():
    import torch
    from torch.profiler import ProfilerActivity, profile
    from datou_gomoku_muzero_b200.tactics import SelfPlayStats, missed_win_counts
    from datou_gomoku_muzero_b200.trajectory import PackedGames, record_dtype
    N = 9
    stride = record_dtype(N).itemsize
    empty = PackedGames(torch.empty((0, stride), dtype=torch.uint8, device="cuda"), np.zeros((0, 4), np.int32),
                        np.zeros(1, np.int64), N)
    one = PackedGames(_record_block(N, [(np.zeros(N * N), 1, 40)]), np.array([[0, 0, 1, 0]], np.int32), np.array([0, 1]), N)
    stats = SelfPlayStats()
    torch.cuda.synchronize()

    def kernels(pg):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            stats.add(pg)
            c = missed_win_counts(pg)
            torch.cuda.synchronize()
        return c, [e.name for e in prof.events() if "k_records_tactics" in e.name]

    c, launched = kernels(empty)
    assert c.shape == (0, 2) and not launched
    assert stats.summary() == SelfPlayStats().summary()
    c, launched = kernels(one)                       # the profiler does see the kernel when there are records
    assert c.tolist() == [[0, 0]] and launched
    assert stats.summary()["games"] == 1 and stats.summary()["moves"] == 1
