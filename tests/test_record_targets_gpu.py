"""The record kernels of csrc/gmz_records.cu at the n-step horizons, unroll lengths, discounts, ring shapes and game
lengths the self-play goldens never reach, bit for bit against the plain references of tests/test_record_targets_cpu.py:
gmz_traj_pack (rewards, value targets, headers, planes), gmz_records_batch (windows under the 8 symmetries),
gmz_records_writeback + gmz_records_retarget (re-analysis in place), the checkpoint round trip, and games longer than the
trajectory store's max_moves, which must not reach the records.  Games are injected into the store's slots, not played,
except in the self-play test at the end."""
import numpy as np
import pytest

from test_record_targets_cpu import (GAMMAS, augment_windows, final_rewards, game_windows, horizons, make_game,
                                     make_games, reanalysis_targets, replay, selfplay_targets)

pytestmark = pytest.mark.gpu

BOARDS = (7, 6)


@pytest.fixture
def cfg():
    from datou_gomoku_muzero_b200.config import config
    saved = (config.N_STEPS, config.NUM_UNROLL_STEPS, config.DISCOUNT)
    yield config
    config.N_STEPS, config.NUM_UNROLL_STEPS, config.DISCOUNT = saved


def _store(N, n_games, max_moves=None):
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng = SearchEngine(4, board_size=N, num_simulations=8)
    return TrajectoryStore(eng, extra_slots=n_games + 4, max_moves=max_moves)


def _bitboards(board):
    """int8 [A] -> the store's start_board row: int64 [2][8] bitboards of the +1 / -1 stones, cell c = bit c % 64 of
    word c // 64."""
    bits = np.zeros((2, 512), np.uint8)
    bits[0, :len(board)] = board == 1
    bits[1, :len(board)] = board == -1
    return np.packbits(bits, axis=1, bitorder="little").view(np.int64)


def _inject(traj, games):
    """Write the games into slots taken from the store's free stack (as the play kernel takes them) -- only the first
    max_moves moves of a longer game, as the play kernel records them -- and queue them finished, full lengths in the
    fin rows.  Returns the slots."""
    import torch
    top = traj.free_slots_left()
    slots = traj.free_slots[top - len(games):top].cpu().numpy()[::-1].tolist()
    traj.free_top.fill_(top - len(games))
    for g, slot in zip(games, slots):
        n = min(len(g["actions"]), traj.max_moves)
        traj.policy[slot, :n] = torch.from_numpy(g["policies"][:n]).cuda()
        traj.value[slot, :n] = torch.from_numpy(g["values"][:n]).cuda()
        traj.action[slot, :n] = torch.from_numpy(g["actions"][:n]).cuda()
        traj.start_board[slot] = torch.from_numpy(_bitboards(g["start_board"])).cuda()
        traj.start_info[slot] = torch.tensor([g["start_player"], g["start_mc"], g["start_last"], g["game"]],
                                             dtype=torch.int32).cuda()
        traj.start_opening[slot] = slot % 3                      # book label + 1, 0 = none
    fin = [[s, g["game"], len(g["actions"]), g["winner"]] for g, s in zip(games, slots)]
    traj.fin_queue[:len(games)] = torch.tensor(fin, dtype=torch.int32).cuda()
    traj.fin_count.fill_(len(games))
    return slots


def _expected(games, slots, N, n, gamma):
    """Packed records of the games, in order, as the references say: record_dtype structured array."""
    from datou_gomoku_muzero_b200.trajectory import record_dtype
    total = sum(len(g["actions"]) for g in games)
    out = np.zeros(total, record_dtype(N))
    o = 0
    for gi, (g, slot) in enumerate(zip(games, slots)):
        T = len(g["actions"])
        r, rp = out[o:o + T], replay(g, N)
        rew = final_rewards(T, g["winner"])
        r["game_seq"], r["t"], r["length"], r["winner"], r["action"] = gi, np.arange(T), T, g["winner"], g["actions"]
        r["to_move"], r["last_move"], r["move_count"] = rp["to_move"], rp["last_move"], rp["move_count"]
        r["reward"], r["value_target"] = rew, selfplay_targets(rew, g["values"], gamma, n)
        r["search_value"], r["game"], r["slot"], r["opening"] = g["values"], g["game"], slot, slot % 3
        r["policy"], r["obs"], r["board"] = g["policies"], rp["obs"], rp["board"]
        o += T
    return out


def _assert_records(got, exp, fields=None):
    """Field by field, as bytes (so -0.0 != +0.0 and NaN patterns count); record padding is not compared."""
    for f in fields or exp.dtype.names:
        assert got[f].tobytes() == exp[f].tobytes(), (f, np.flatnonzero((got[f] != exp[f]).reshape(len(exp), -1).any(1))[:8])


def _packed(N, games, n, gamma, cfg):
    traj = _store(N, len(games))
    slots = _inject(traj, games)
    cfg.N_STEPS, cfg.DISCOUNT = n, gamma
    pg = traj.pack_finished(recycle=False)
    return traj, slots, pg


@pytest.mark.parametrize("N", BOARDS)
def test_traj_pack_over_the_n_steps_gamma_grid(N, cfg):
    """gmz_traj_pack through pack_finished for n_steps in {0, 1, 2, 3, 5, 10, 31, 64} and T - 1, T, T + 1 of every game,
    against gamma in {1, 0.997, 0.9, 0.5, 0}: every header field, the planes, boards and policy bytes."""
    games = make_games(N, seed=N)
    lengths = [len(g["actions"]) for g in games]
    traj = _store(N, len(games))
    slots = _inject(traj, games)
    for i, n in enumerate(horizons(lengths)):
        for gamma in GAMMAS:
            cfg.N_STEPS, cfg.DISCOUNT = n, gamma
            traj.fin_count.fill_(len(games))
            pg = traj.pack_finished(recycle=False)
            assert np.array_equal(np.diff(pg.offsets), lengths) and np.array_equal(pg.table[:, 2], lengths)
            exp = _expected(games, slots, N, n, gamma)
            heavy = i == 0 and gamma == GAMMAS[0]                 # planes, boards, policies do not depend on (n, gamma)
            _assert_records(pg.host(), exp, None if heavy else [f for f in exp.dtype.names if f not in ("policy", "obs", "board")])


def _ring_windows(records, U):
    """Windows of every record of a block of whole games (record order), cut per game by the reference."""
    starts = np.flatnonzero(records["t"] == 0).tolist() + [len(records)]
    parts = [game_windows(records["obs"][a:b], records["policy"][a:b], records["action"][a:b], records["reward"][a:b],
                          records["value_target"][a:b], U) for a, b in zip(starts, starts[1:])]
    return [np.concatenate(x) for x in zip(*parts)]


@pytest.mark.parametrize("N", BOARDS)
def test_records_batch_windows_under_every_symmetry(N, cfg):
    """DeviceReplayBuffer.batch for U in {0, 1, 5, 12, 40} (games shorter than U included) under the 8 symmetries, in
    rings larger than the data, wrapped, and smaller than one game: every live position, obs / act / rew / pi / val
    with their zero and -1 padding."""
    import torch
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    games = make_games(N, seed=N + 1)
    _, _, pg = _packed(N, games, 10, 0.997, cfg)
    recs = pg.host()
    total = len(recs)
    rs = np.random.RandomState(N)
    for U in (0, 1, 5, 12, 40):
        W = _ring_windows(recs, U)
        for cap in (total + 7, total - 11, 5):
            buf = DeviceReplayBuffer(cap, N, unroll_steps=U)
            buf.add_packed(pg)
            live = np.arange(max(0, total - cap), total)              # record j sits at ring position j % cap
            order = rs.permutation(len(live))
            pos = live[order] % cap
            j = live[order]
            for k in range(4):
                for flip in (False, True):
                    obs, act, rew, pi, val = (x.cpu().numpy() for x in buf.batch(torch.as_tensor(pos, device="cuda"), k, flip))
                    eo, ea, ep = augment_windows(W[0][j], W[1][j], W[3][j], N, k, flip)
                    assert obs.dtype == np.float32 and act.dtype == np.int32 and pi.dtype == np.float64
                    assert obs.tobytes() == eo.tobytes() and pi.tobytes() == ep.tobytes(), (U, cap, k, flip)
                    assert act.tobytes() == ea.tobytes(), (U, cap, k, flip)
                    assert rew.tobytes() == W[2][j].tobytes() and val.tobytes() == W[4][j].tobytes(), (U, cap)


@pytest.mark.parametrize("N", BOARDS)
def test_writeback_and_retarget_over_the_grid(N, cfg):
    """gmz_records_writeback of arbitrary float64 search values and policies, then gmz_records_retarget over the
    (n_steps, gamma) grid, on stretches with first > 0, wrapping the ring end, and with n = capacity: value targets by
    the re-analysis reference, search values and policies as written, every other byte of the ring unchanged."""
    import torch
    from datou_gomoku_muzero_b200._lib import check
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.trajectory import record_dtype, record_fields
    from test_record_targets_cpu import SPECIAL_VALUES
    games = make_games(N, seed=N + 2)
    lengths = [len(g["actions"]) for g in games]
    _, _, pg = _packed(N, games, 10, 0.997, cfg)
    total, A = pg.n_moves, N * N
    fields = record_fields(N)
    rs = np.random.RandomState(N + 3)
    for cap, first in ((total + 9, 4), (total + 9, total + 3), (total, 17)):
        buf = DeviceReplayBuffer(cap, N)
        buf.ring.copy_(torch.randint(0, 256, buf.ring.shape, dtype=torch.uint8, device="cuda"))
        pos = (first + np.arange(total)) % cap
        buf.ring[torch.as_tensor(pos, device="cuda")] = pg.records
        before = buf.ring.cpu().numpy()
        stream = buf.sum_tree._stream()
        pol = torch.from_numpy(rs.dirichlet(np.ones(A), size=total)).cuda()
        vals = np.where(rs.rand(total) < 0.6, SPECIAL_VALUES[rs.randint(len(SPECIAL_VALUES), size=total)], rs.uniform(-1, 1, total))
        val = torch.from_numpy(vals).cuda()
        check(buf.lib.gmz_records_writeback(buf.ring.data_ptr(), cap, N, first, total, pol.data_ptr(), val.data_ptr(), stream),
              "gmz_records_writeback")
        for n in horizons(lengths):
            for gamma in GAMMAS:
                dpow = torch.tensor([gamma ** i for i in range(n + 1)], dtype=torch.float64, device="cuda")
                check(buf.lib.gmz_records_retarget(buf.ring.data_ptr(), cap, N, first, total, dpow.data_ptr(), n, stream),
                      "gmz_records_retarget")
                after = buf.ring.cpu().numpy()
                r = after[pos].copy().view(record_dtype(N)).reshape(-1)
                exp = np.concatenate([reanalysis_targets(final_rewards(T, g["winner"]), vals[o:o + T], gamma, n)
                                      for g, T, o in zip(games, lengths, np.cumsum([0] + lengths[:-1]))])
                assert r["value_target"].tobytes() == exp.tobytes(), (cap, first, n, gamma)
        assert r["search_value"].tobytes() == vals.tobytes() and r["policy"].tobytes() == pol.cpu().numpy().tobytes()
        b, a = before.copy(), after.copy()
        for x in (a, b):
            for f in ("policy", "search_value", "value_target"):
                x[pos, fields[f]] = 0
        assert np.array_equal(a, b), (cap, first)


def test_checkpoint_keeps_value_targets_verbatim(cfg):
    """state_dict() of a ring holding records packed under two (n_steps, gamma), loaded under a third: the value
    targets (and every other field of the live records) come back as saved, in a ring of the same and of a smaller
    capacity."""
    import torch
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.trajectory import record_dtype
    N = 7
    games = make_games(N, seed=11)
    traj, _, pg1 = _packed(N, games, 5, 0.9, cfg)
    total = pg1.n_moves
    cfg.N_STEPS, cfg.DISCOUNT = 64, 1.0
    traj.fin_count.fill_(len(games))
    pg2 = traj.pack_finished(recycle=False)
    assert pg1.host()["value_target"].tobytes() != pg2.host()["value_target"].tobytes()
    cap = 2 * total - 20                                          # wrapped, oldest live game cut
    buf = DeviceReplayBuffer(cap, N)
    buf.add_packed(pg1)
    buf.add_packed(pg2)
    sd = buf.state_dict()
    cfg.N_STEPS, cfg.DISCOUNT = 31, 0.5
    host = lambda b: b.ring.cpu().numpy().view(record_dtype(N)).reshape(-1)
    names = [f for f in record_dtype(N).names]
    same = DeviceReplayBuffer(cap, N)
    same.load_state_dict(sd)
    _assert_records(host(same), host(buf), names)
    small = DeviceReplayBuffer(total // 2, N)
    small.load_state_dict(sd)
    newest = (buf.sum_tree.write_ptr - total // 2 + np.arange(total // 2)) % cap
    _assert_records(host(small), host(buf)[newest], names)
    assert host(small)["value_target"].tobytes() == pg2.host()["value_target"][-(total // 2):].tobytes()


# ---------------------------------------------------------------------------------------------------------------------
# Games longer than the store's max_moves.
def _truncation_games(N, M, seed):
    """Games longer than M at every residue (L - M) mod 4, and whole games of length M, M - 3 and 1, interleaved."""
    rs = np.random.RandomState(seed)
    Ls = [M + 4, M, M + 1, M - 3, M + 2, 1, M + 3, M + 8]
    return [make_game(rs, N, 2 * (i % 3), 1, L, 1, 20 + i) for i, L in enumerate(Ls)]


def test_pack_finished_packs_only_whole_games(cfg):
    """A store with max_moves below some game lengths: pack_finished returns the whole games only, with a table whose
    lengths are their record counts, records equal to the reference, every slot released, the rest counted."""
    N, M = 7, 9
    cfg.N_STEPS, cfg.DISCOUNT = 3, 0.997
    games = _truncation_games(N, M, 1)
    whole = [i for i, g in enumerate(games) if len(g["actions"]) <= M]
    traj = _store(N, len(games), max_moves=M)
    free0 = traj.free_slots_left()
    slots = _inject(traj, games)
    pg = traj.pack_finished(recycle=True)
    assert traj.free_slots_left() == free0 and int(traj.fin_count.item()) == 0
    assert pg.table[:, 1].tolist() == [games[i]["game"] for i in whole]
    assert np.array_equal(np.diff(pg.offsets), pg.table[:, 2])
    _assert_records(pg.host(), _expected([games[i] for i in whole], [slots[i] for i in whole], N, 3, 0.997))
    assert traj.truncated_games == len(games) - len(whole)
    # only truncated games: nothing to pack, the slots still come back, the counter keeps counting
    slots = _inject(traj, [games[0], games[2]])
    assert traj.pack_finished(recycle=True) is None
    assert traj.free_slots_left() == free0 and traj.truncated_games == len(games) - len(whole) + 2


def test_harvest_flags_truncated_games_and_build_game_record_refuses_them():
    from datou_gomoku_muzero_b200.trajectory import build_game_record
    N, M = 7, 9
    games = _truncation_games(N, M, 2)
    traj = _store(N, len(games), max_moves=M)
    _inject(traj, games)
    got = traj.harvest()
    assert [r["truncated"] for r in got] == [len(g["actions"]) > M for g in games]
    assert [r["length"] for r in got] == [min(len(g["actions"]), M) for g in games]
    for r, g in zip(got, games):
        if r["truncated"]:
            with pytest.raises(ValueError):
                build_game_record(r, N)
        else:
            gr = build_game_record(r, N)
            assert np.array_equal(np.float32(gr.rewards), final_rewards(len(g["actions"]), g["winner"]))


def _ends_game(board, cell, colour, n_in_row):
    """Does playing `cell` for `colour` on `board` (N x N, before the move) make a line of n_in_row?"""
    N = board.shape[0]
    b = board.copy()
    r0, c0 = divmod(int(cell), N)
    b[r0, c0] = colour
    for dr, dc in ((0, 1), (1, 0), (1, 1), (1, -1)):
        run = 1
        for s in (1, -1):
            r, c = r0 + s * dr, c0 + s * dc
            while 0 <= r < N and 0 <= c < N and b[r, c] == colour:
                run += 1
                r, c = r + s * dr, c + s * dc
        if run >= n_in_row:
            return True
    return False


def test_selfplay_sink_with_small_max_moves_keeps_only_whole_games():
    """Persistent E0 self-play through play(sink=DeviceReplayBuffer.add_packed) with max_moves below many game lengths:
    every game in the ring is whole (t = 0 .. length - 1, its last move ends the game: a five for the mover or a full
    board), every record's reward is the pattern of its own header length and winner, and finished = packed +
    truncated."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore, record_dtype
    N, G, M = 6, 32, 16
    eng = SearchEngine(G, board_size=N, num_simulations=8)
    sp = SelfPlayEngine(eng, "e0", seed=3, noise_seed=4)
    traj = TrajectoryStore(eng, extra_slots=32, max_moves=M)
    buf = DeviceReplayBuffer(100_000, N)
    packed = []
    sp.play(moves_per_game=120, traj=traj, sink=lambda pg: (packed.append(len(pg)), buf.add_packed(pg)))
    n = len(buf)
    assert 0 < n < buf.capacity
    h = buf.ring[:n].cpu().numpy().view(record_dtype(N)).reshape(-1)
    starts = np.flatnonzero(h["t"] == 0).tolist()
    assert starts[0] == 0
    for a, b in zip(starts, starts[1:] + [n]):
        r = h[a:b]
        T, w = int(r["length"][0]), int(r["winner"][0])
        assert T == b - a and (r["t"] == np.arange(T)).all() and (r["length"] == T).all() and (r["winner"] == w).all()
        assert r["reward"].tobytes() == final_rewards(T, w).tobytes()
        last = r[-1]
        if w == 0:
            assert (last["board"] != 0).sum() == N * N - 1
        else:
            assert w == last["to_move"] and _ends_game(last["board"], last["action"], w, 5), (a, T)
    _, nfin = eng.play_counters()
    assert sum(packed) == len(starts) and traj.truncated_games > 0 and len(starts) + traj.truncated_games == nfin
