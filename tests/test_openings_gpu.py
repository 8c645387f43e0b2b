"""Self-play from an opening book (SearchEngine.set_openings, gmz_set_openings): every restarted game of index g takes
opening (k*G + g) mod O at its k-th deal.  Checked against a host loop that deals by that schedule and searches every
move with the CPU oracle; across the persistent and stepwise paths and launch splits; an empty-board book against no
book; the records downstream (replay, checkpoint, re-analysis, missed-win flags, per-opening results); unbinding; the
arena's isolation from a bound book; refusals."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _near_full(N):
    """A position with three empty cells and no three in a row of either colour, white to move."""
    r, c = np.divmod(np.arange(N * N), N)
    b = np.where((c + 2 * r) % 4 < 2, 1, -1).astype(np.int8)
    b[-3:] = 0
    return b


def _book(N, nir):
    """Three black-to-move openings of two stones (one with last move None), two white-to-move ones of three stones and
    a near-full white-to-move board: O = 6."""
    from datou_gomoku_muzero_b200.arena import Openings, check_openings, random_openings
    a, b = random_openings(3, 2, N, seed=N, n_in_row=nir), random_openings(2, 3, N, seed=N + 1, n_in_row=nir)
    nf = _near_full(N)
    op = Openings(np.concatenate([a.boards, b.boards, nf[None]]), np.concatenate([a.players, b.players, [-1]]).astype(np.int8),
                  np.concatenate([a.last_moves, b.last_moves, [-1]]).astype(np.int32),
                  np.concatenate([a.move_counts, b.move_counts, [int((nf != 0).sum())]]).astype(np.int32))
    op.last_moves[1] = -1
    return check_openings(op, N, nir)


def _by_index(finished):
    """harvest() dicts -> {game index: [its finished games in the order they were dealt]}."""
    out = {}
    for r in finished:
        out.setdefault(r["game"], []).append(r)
    return out


def _persistent(N, nir, S, G, mode, accum, book, chunks, seed=5, nseed=77, extra=8):
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=S, mode=mode, accum_dtype=accum)
    sp = SelfPlayEngine(eng, "e0", seed=seed, noise_seed=nseed, openings=book)
    traj = TrajectoryStore(eng, extra_slots=extra)
    fin = []
    for n in chunks:
        sp.play(moves_per_game=n, traj=traj)
        fin += traj.harvest()
    return eng, _by_index(fin)


def _host_games(cfg, book, G, g, nir, noise, n_games):
    """Game index g's first n_games games as the reference's loop plays them from the schedule's openings: one oracle
    search per move with the noise of the game's own search counter."""
    from oracle import oracle
    N, O = cfg.board_size, book.boards.shape[0]
    out, c = [], 0
    for k in range(n_games):
        o = (k * G + g) % O
        board, to_move = book.boards[o].copy(), int(book.players[o])
        last, mc = int(book.last_moves[o]), int(book.move_counts[o])
        acts, vals, pols = [], [], []
        while True:
            r = oracle.search(cfg, board, to_move, last, mc, noise[c, g])
            c += 1
            a = int(r["action"])
            acts.append(a); vals.append(r["value"]); pols.append(r["policy"])
            board[a] = to_move
            last, mc, to_move = a, mc + 1, -to_move
            w = oracle.game_ended(board.reshape(N, N), nir, last, mc)
            if w is not None:
                break
        out.append(dict(opening=o, actions=np.array(acts), values=np.array(vals), policies=np.array(pols), winner=w))
    return out


def _noise(eng, nseed, n_counters):
    """[counter, game, A]: gmz_fill_gumbel's draw for search `counter` of game g, offset (counter*G + g)*A."""
    import torch
    buf = torch.empty(n_counters * eng.G * eng.A, dtype=torch.float64, device=eng.device)
    eng.fill_gumbel(buf, nseed, 0)
    return buf.cpu().numpy().reshape(n_counters, eng.G, eng.A)


def _same_game(a, b, what):
    assert a["length"] == b["length"] and a["winner"] == b["winner"] and a["opening"] == b["opening"], what
    assert np.array_equal(a["actions"], b["actions"]) and np.array_equal(a["values"], b["values"]), what
    assert np.array_equal(a["policies"], b["policies"]), what


@pytest.mark.parametrize("N,nir,S,mode,accum", [(6, 4, 36, "AlphaZero", "float64"), (6, 4, 40, "MuZero", "float32"),
                                                (9, 5, 48, "MuZero", "float64"), (12, 4, 24, "AlphaZero", "float32")])
def test_persistent_selfplay_from_a_book_matches_oracle(N, nir, S, mode, accum):
    from oracle import oracle
    G, seed, nseed = 4, 5, 77
    book = _book(N, nir)
    O = book.boards.shape[0]
    assert O % G and (book.players == -1).any() and (book.last_moves == -1).any()
    chunks = [N * N // 3] * 8
    eng, dev = _persistent(N, nir, S, G, mode, accum, book, chunks, seed, nseed)
    assert sorted(dev) == list(range(G)) and all(len(v) >= 1 for v in dev.values())   # every index dealt at least twice
    cfg = oracle.make_config(board_size=N, n_in_row=nir, num_simulations=S, eval_seed=seed,
                             mode=0 if mode == "AlphaZero" else 1, accum_dtype=1 if accum == "float32" else 0)
    noise = _noise(eng, nseed, sum(chunks) * G)             # more searches than any one game index can have run
    dealt = set()
    for g, games in dev.items():
        host = _host_games(cfg, book, G, g, nir, noise, len(games))
        for k, (d, h) in enumerate(zip(games, host)):
            o = h["opening"]
            dealt.add(o)
            assert d["opening"] == o and d["start_player"] == book.players[o], (g, k)
            assert np.array_equal(d["start_board"].reshape(-1), book.boards[o]), (g, k)
            assert d["start_last_move"] == book.last_moves[o] and d["start_move_count"] == book.move_counts[o], (g, k)
            assert d["length"] == len(h["actions"]) and d["winner"] == h["winner"], (g, k)
            assert np.array_equal(d["actions"], h["actions"]) and np.array_equal(d["values"], h["values"]), (g, k)
            # the device softmax and the oracle's differ in the last bits, as in tests/test_selfplay_gpu.py
            np.testing.assert_allclose(d["policies"], h["policies"], rtol=1e-12, atol=1e-15, err_msg=str((g, k)))
    assert len(dealt) >= 5


def test_paths_and_launch_splits_play_the_same_games():
    """Stepwise self-play (an E0 callable in AlphaZero mode, MuZeroDeviceSearch over TorchE0 in MuZero mode) equals the
    persistent kernel game for game, and play(40) equals five play(8)."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.muzero import MuZeroDeviceSearch, TorchE0
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    N, nir, S, G, seed, nseed = 6, 4, 30, 5, 8, 21
    A, book = N * N, _book(N, nir)
    for mode in ("AlphaZero", "MuZero"):
        _, five = _persistent(N, nir, S, G, mode, "float64", book, [8] * 5, seed, nseed, extra=64)
        _, one = _persistent(N, nir, S, G, mode, "float64", book, [40], seed, nseed, extra=64)
        e2 = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=S, mode=mode)
        if mode == "AlphaZero":
            ev = lambda obs: e2.e0_eval(obs, seed)                    # noqa: E731
        else:
            e0 = TorchE0(N, seed=seed)
            ev = (e0.initial, e0.recurrent)
        sp2 = SelfPlayEngine(e2, ev, noise_seed=nseed, openings=book)
        assert isinstance(sp2.searcher, MuZeroDeviceSearch) == (mode == "MuZero")
        t2 = TrajectoryStore(e2, extra_slots=64)
        gum = torch.empty((G, A), dtype=torch.float64, device="cuda")
        fin = []
        for c in range(40):
            for g in range(G):
                e2.fill_gumbel(gum[g], nseed, (c * G + g) * A)
            pol, val, act, _ = sp2.search(gumbel=gum)
            e2.selfplay_step(pol, val, act, t2, True)
            fin += t2.harvest()
        step = _by_index(fin)
        compared = 0
        for g in range(G):
            for other, name in ((one, "play(40)"), (step, "stepwise")):
                for k, (a, b) in enumerate(zip(five.get(g, []), other.get(g, []))):
                    _same_game(a, b, (mode, name, g, k))
                    compared += 1
        assert compared >= 2 * G, (mode, compared)


def _parked_run(N, nir, S, G, book):
    """Every game plays exactly one game (no restarts) and is packed: records sorted by game index."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=S)
    sp = SelfPlayEngine(eng, "e0", seed=3, noise_seed=4, openings=book)
    traj = TrajectoryStore(eng, extra_slots=0)
    sp.play(moves_per_game=N * N, traj=traj, restart=False)
    pg = traj.pack_finished(recycle=False)
    assert len(pg) == G
    order = np.argsort(pg.table[:, 1], kind="stable")
    body = 64 + 21 * N * N                     # the tail padding of a record is not record content
    raw = np.concatenate([pg.records[int(pg.offsets[i]):int(pg.offsets[i + 1]), :body].cpu().numpy() for i in order])
    return pg, raw


def test_empty_board_book_plays_the_games_of_no_book():
    from datou_gomoku_muzero_b200.arena import empty_opening
    N, nir, S, G = 6, 4, 24, 6
    pg0, raw0 = _parked_run(N, nir, S, G, None)
    pg1, raw1 = _parked_run(N, nir, S, G, empty_opening(N))
    assert (pg0.openings() == -1).all() and (pg1.openings() == 0).all()
    lab0, lab1 = raw0[:, 56:60].copy().view(np.int32), raw1[:, 56:60].copy().view(np.int32)
    assert (lab0 == 0).all() and (lab1 == 1).all()
    for r in (raw0, raw1):
        r[:, 56:60] = 0
        r[:, 0:4] = 0                  # game_seq: the order games finished in, which the kernel does not fix
    assert np.array_equal(raw0, raw1)


def test_records_downstream_of_a_book():
    import torch
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.game import GomokuGame
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.tactics import SelfPlayStats, classify_boards, record_flags
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore, final_rewards
    from test_ring_reanalysis_gpu import _check_parity, _engines, _expected, _host
    N, nir, S, G = 6, 4, 16, 8
    A, book = N * N, _book(N, nir)
    O = book.boards.shape[0]
    saved = config.N_IN_ROW
    config.N_IN_ROW = nir
    try:
        eng = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=S)
        sp = SelfPlayEngine(eng, "e0", seed=11, noise_seed=12, openings=book)
        traj = TrajectoryStore(eng, extra_slots=G)
        buf = DeviceReplayBuffer(4000, N)
        stats = SelfPlayStats(n_in_row=nir, n_openings=O - 1)        # the near-full opening's games: totals only
        packs = []

        def sink(pg):
            packs.append(pg); buf.add_packed(pg); stats.add(pg)
        for _ in range(6):
            sp.play(moves_per_game=8, traj=traj, sink=sink)
        assert len(buf) < buf.capacity
        games = sum(len(p) for p in packs)
        assert games >= 2 * G
        counts = np.zeros((O - 1, 3), np.int64)
        for pg in packs:
            h, labels = pg.host(), pg.openings()
            flags = record_flags(pg.records[:pg.n_moves], N, nir).cpu().numpy()
            cls = classify_boards(h["board"].reshape(-1, A), h["to_move"].astype(np.int8), N, nir).cpu().numpy()
            win = (cls > 0).any(1)
            played = cls[np.arange(len(h)), h["action"]] > 0
            assert np.array_equal(flags, win * 1 + (cls == 1).any(1) * 2 + played * 4)
            for i in range(len(pg)):
                r, o = pg.game(i), int(labels[i])
                assert 0 <= o < O and (r["opening"] == o + 1).all()
                g = GomokuGame(board_size=N, n_in_row=nir)
                g.board = book.boards[o].reshape(N, N).copy()
                g.current_player = int(book.players[o])
                g.last_move = None if book.last_moves[o] < 0 else divmod(int(book.last_moves[o]), N)
                g.move_count = int(book.move_counts[o])
                for t in range(len(r)):
                    assert np.array_equal(r["board"][t], g.board) and r["to_move"][t] == g.current_player
                    lm = -1 if g.last_move is None else g.last_move[0] * N + g.last_move[1]
                    assert r["last_move"][t] == lm and r["move_count"][t] == g.move_count
                    assert np.array_equal(r["obs"][t], g.get_board_state(g.current_player, g.last_move))
                    g.do_move(int(r["action"][t]))
                w = g.get_game_ended()
                assert w is not None and w == r["winner"][0]
                assert np.array_equal(r["reward"], final_rewards(len(r), w))
                gr = pg.game_record(i)
                assert gr.actions == r["action"].tolist() and len(gr.observations) == len(r)
                if o < O - 1:
                    counts[o, 1 if w == 0 else (0 if w == r["to_move"][0] else 2)] += 1
        assert np.array_equal(stats.by_opening(), counts) and stats.games == games
        # checkpoint round trip
        sd = buf.state_dict()
        buf2 = DeviceReplayBuffer(4000, N)
        buf2.load_state_dict(sd)
        body = 64 + 21 * A                           # the tail padding is not record content
        assert torch.equal(buf2.ring[:, :body], buf.ring[:, :body]) and torch.equal(buf2.sum_tree.tree, buf.sum_tree.tree)
        # ring re-analysis against the host driver
        snap, tree0 = _host(buf), buf.sum_tree.tree.clone()
        start, n = buf.reanalyse(_engines(N, (G, G), S, n_in_row=nir), eval_seed=5, noise_seed=7)
        pol, val, vt = _expected(snap, start, n, _engines(N, (G, G), S, n_in_row=nir), eval_seed=5, noise_seed=7)
        _check_parity(buf, snap, tree0, start, n, pol, val, vt)
    finally:
        config.N_IN_ROW = saved


def test_unbinding_and_arena_isolation():
    from datou_gomoku_muzero_b200.arena import Arena
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    N, nir, S, G = 6, 4, 16, 6
    book = _book(N, nir)
    O = book.boards.shape[0]
    eng = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=S)
    sp = SelfPlayEngine(eng, "e0", seed=2, noise_seed=3, openings=book)
    traj = TrajectoryStore(eng, extra_slots=32)
    before, after = [], []
    for _ in range(3):
        sp.play(moves_per_game=6, traj=traj); before += traj.harvest()
    eng.set_openings(None)
    for _ in range(8):
        sp.play(moves_per_game=6, traj=traj); after += traj.harvest()
    carried = 0
    for g, games in _by_index(before + after).items():
        labels = [r["opening"] for r in games]
        n_book = sum(lab >= 0 for lab in labels)
        assert labels[:n_book] == [(k * G + g) % O for k in range(n_book)] and all(lab == -1 for lab in labels[n_book:])
        assert len(games) > n_book                        # the index was dealt again after the unbind: an empty board
        for r in games[n_book:]:
            assert not r["start_board"].any() and r["start_player"] == 1 and r["start_move_count"] == 0
        carried += sum(r["opening"] >= 0 for r in after if r["game"] == g)
    assert carried >= 1                                   # games in flight at the unbind kept their labels
    # a bound book does not reach the match kernels
    results = []
    for bound in (True, False):
        ea, eb = (SearchEngine(4, board_size=N, n_in_row=nir, num_simulations=S) for _ in range(2))
        if bound:
            ea.set_openings(book); eb.set_openings(book)
        results.append(Arena(ea, eb, seed=9).play(book))
    a, b = results
    assert np.array_equal(a.winner, b.winner) and np.array_equal(a.length, b.length) and np.array_equal(a.moves, b.moves)


def test_refusals_launch_nothing():
    from datou_gomoku_muzero_b200._lib import GmzError
    from datou_gomoku_muzero_b200.arena import Openings
    from datou_gomoku_muzero_b200.engine import SearchEngine
    N, nir = 6, 4
    book = _book(N, nir)
    eng = SearchEngine(4, board_size=N, n_in_row=nir, num_simulations=8)
    n0 = eng.launches
    b, p, lm, mc = (x.copy() for x in book)
    won = b[0].copy(); won[:4] = 1                     # four in a row at n_in_row 4
    bad = [Openings(b[:, :-1], p, lm, mc),                                     # shape
           Openings(b, p[:-1], lm, mc),                                        # players shape
           Openings(np.where(b == 1, 2, b).astype(np.int8), p, lm, mc),         # value outside {-1, 0, 1}
           Openings(b, np.zeros_like(p), lm, mc),                              # side to move
           Openings(b, p, np.full_like(lm, N * N), mc),                        # last move
           Openings(np.ones_like(b), p, lm, np.full_like(mc, N * N)),          # no empty cell
           Openings(b, p, lm, np.zeros_like(mc)),                              # move count below the stones
           Openings(np.concatenate([b, won[None]]), np.append(p, 1).astype(np.int8), np.append(lm, 3).astype(np.int32),
                    np.append(mc, 8).astype(np.int32)),                        # already ended
           _book(9, nir)]                                                      # another board size
    for op in bad:
        with pytest.raises(ValueError):
            eng.set_openings(op)
    assert eng.launches == n0
    eng.lib.gmz_destroy(eng.handle)
    with pytest.raises(GmzError, match="invalid or destroyed"):
        eng.set_openings(book)
    with pytest.raises(GmzError, match="invalid or destroyed"):
        eng.set_openings(None)
    assert eng.launches == n0
    eng.handle = None
