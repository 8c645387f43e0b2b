"""Matches between two engines (arena.Arena, csrc/gmz_match.cu): every game checked against a host match driven by the
CPU oracle with each player's own configuration and the match's counter-based noise; independence from G and from the
order of the players; a player against itself; a network player; colour balance."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _openings(N, nir):
    """Four black-to-move openings of two stones and one white-to-move opening of three."""
    from datou_gomoku_muzero_b200.arena import Openings, random_openings
    a, b = random_openings(4, 2, N, seed=N, n_in_row=nir), random_openings(1, 3, N, seed=N + 1, n_in_row=nir)
    return Openings(*(np.concatenate([x, y]) for x, y in zip(a, b)))


class _Noise:
    """The match noise of ply k of opening o, regenerated with the engine's own gmz_fill_gumbel."""

    def __init__(self, eng, seed):
        import torch
        self.eng, self.seed, self.cache = eng, seed, {}
        self.buf = torch.empty(eng.A, dtype=torch.float64, device=eng.device)

    def __call__(self, o, k):
        if (o, k) not in self.cache:
            A = self.eng.A
            self.cache[(o, k)] = self.eng.fill_gumbel(self.buf, self.seed, (o * A + k) * A).cpu().numpy().copy()
        return self.cache[(o, k)]


def _host_match(op, N, nir, search, noise):
    """Ticket t = 2o + q (q = 0: A first): the oracle's moves, winner and length.  search(player, board, to_move, last,
    move_count, gumbel) -> action, player 0 = A."""
    from oracle import oracle
    out = []
    for t in range(2 * op.boards.shape[0]):
        o, q = divmod(t, 2)
        board, to_move = op.boards[o].copy(), int(op.players[o])
        last, mc, moves = int(op.last_moves[o]), int(op.move_counts[o]), []
        while True:
            k = len(moves)
            a = search(q if k % 2 == 0 else 1 - q, board, to_move, last, mc, noise(o, k))
            assert board[a] == 0
            board[a] = to_move
            last, mc, to_move = a, mc + 1, -to_move
            moves.append(a)
            w = oracle.game_ended(board.reshape(N, N), nir, last, mc)
            if w is not None:
                break
        out.append((moves, w))
    return out


def _oracle_search(cfgs):
    from oracle import oracle

    def search(player, board, to_move, last, mc, gum):
        return int(oracle.search(cfgs[player], board, to_move, last, mc, gum)["action"])
    return search


def _check_against(res, expected):
    for t, (moves, w) in enumerate(expected):
        T = len(moves)
        assert res.finished[t] and res.length[t] == T and res.winner[t] == w, (t, res.length[t], T, res.winner[t], w)
        assert np.array_equal(res.moves[t, :T], moves), t
        assert (res.moves[t, T:] == -1).all()


@pytest.mark.parametrize("N,nir", [(6, 4), (9, 5)])
def test_e0_match_matches_oracle(N, nir):
    """Different eval_seed / logit_div / S / K per player, G smaller than the number of tickets (slots recycle),
    a white-to-move opening in the book."""
    from datou_gomoku_muzero_b200.arena import Arena
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    G, seed = 4, 21
    ea = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=24, num_top_actions=8)
    eb = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=40, num_top_actions=4)
    op = _openings(N, nir)
    assert (op.players == -1).any()
    res = Arena(ea, eb, eval_seed_a=3, logit_div_a=16, eval_seed_b=11, logit_div_b=0, seed=seed).play(op)
    cfgs = (oracle.make_config(board_size=N, n_in_row=nir, num_simulations=24, num_top_actions=8, eval_seed=3, logit_div=16),
            oracle.make_config(board_size=N, n_in_row=nir, num_simulations=40, num_top_actions=4, eval_seed=11, logit_div=0))
    _check_against(res, _host_match(op, N, nir, _oracle_search(cfgs), _Noise(ea, seed)))
    assert len(res) == 2 * op.boards.shape[0]


def test_alphazero_against_muzero_matches_oracle():
    from datou_gomoku_muzero_b200.arena import Arena
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    N, nir, G, seed = 6, 4, 3, 8
    ea = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=32, num_top_actions=8, mode="AlphaZero")
    eb = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=32, num_top_actions=8, mode="MuZero")
    op = _openings(N, nir)
    res = Arena(ea, eb, eval_seed_a=5, eval_seed_b=6, seed=seed).play(op)
    cfgs = (oracle.make_config(board_size=N, n_in_row=nir, num_simulations=32, num_top_actions=8, eval_seed=5, mode=0),
            oracle.make_config(board_size=N, n_in_row=nir, num_simulations=32, num_top_actions=8, eval_seed=6, mode=1))
    _check_against(res, _host_match(op, N, nir, _oracle_search(cfgs), _Noise(ea, seed)))


def test_games_do_not_depend_on_G_or_player_order():
    from datou_gomoku_muzero_b200.arena import Arena, random_openings
    from datou_gomoku_muzero_b200.engine import SearchEngine
    N, nir = 6, 4
    op = random_openings(6, 2, N, seed=3, n_in_row=nir)
    runs = {}
    for G in (4, 16, 64):
        ea = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=16, num_top_actions=4)
        eb = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=24, num_top_actions=8)
        runs[G] = Arena(ea, eb, eval_seed_a=1, eval_seed_b=2, seed=9).play(op)
        if G == 16:
            swapped = Arena(eb, ea, eval_seed_a=2, eval_seed_b=1, seed=9).play(op)
    for G in (16, 64):
        assert np.array_equal(runs[G].moves, runs[4].moves) and np.array_equal(runs[G].winner, runs[4].winner)
    r = runs[16]
    mirror = np.arange(r.moves.shape[0]) ^ 1           # ticket 2o <-> 2o + 1: the other player moves first
    assert np.array_equal(swapped.moves, r.moves[mirror]) and np.array_equal(swapped.winner, r.winner[mirror])
    np.testing.assert_array_equal(swapped.a_score, 1.0 - r.a_score[mirror])
    assert swapped.wdl() == r.wdl()[::-1] and swapped.score() == pytest.approx(1.0 - r.score(), abs=1e-15)


def test_self_match_scores_exactly_one_half():
    from datou_gomoku_muzero_b200.arena import Arena, random_openings
    from datou_gomoku_muzero_b200.engine import SearchEngine
    N, nir, G = 9, 5, 8
    ea, eb = (SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=32, num_top_actions=8) for _ in range(2))
    res = Arena(ea, eb, eval_seed_a=4, eval_seed_b=4, seed=2).play(random_openings(10, 3, N, seed=1, n_in_row=nir))
    assert np.array_equal(res.moves[0::2], res.moves[1::2]) and np.array_equal(res.winner[0::2], res.winner[1::2])
    assert res.score() == 0.5 and (res.pair_scores() == 0.5).all()
    st = res.elo()
    assert st["elo"] == 0.0 and st["elo_lo"] == 0.0 and st["elo_hi"] == 0.0 and st["los"] == 0.5


def test_network_player_replayed_through_the_oracle():
    """A small GomokuNetEZ behind an eager callable against E0: every (observation -> logits, value) the network
    produced is recorded, and its plies are replayed through the oracle's tree with a table evaluator; the results
    table equals a GomokuGame replay of the move logs."""
    import torch
    from datou_gomoku_muzero_b200.arena import Arena
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.game import GomokuGame
    from datou_gomoku_muzero_b200.network import DeviceEvaluator, GomokuNetEZ
    from oracle import oracle
    N, nir, G, S, seed = 6, 4, 4, 24, 13
    torch.manual_seed(0)
    net = GomokuNetEZ(Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=N * N, NUM_RES_BLOCKS=1, NUM_FILTERS=16, HEAD_HIDDEN_DIM=16))
    ea = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=S, num_top_actions=8, accum_dtype="float32")
    eb = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=S, num_top_actions=8)
    ev = DeviceEvaluator(net, ea.leaf_obs, dtype=torch.float32, graph=False)
    table = {}

    def player(obs):
        lg, v = ev(obs)
        o, l, vv = obs.cpu().numpy(), lg.cpu().numpy(), v.cpu().numpy()
        for g in range(G):
            cur = (l[g].copy(), float(vv[g]))
            key = o[g].tobytes()
            if key in table:
                assert np.array_equal(table[key][0], cur[0]) and table[key][1] == cur[1]
            table[key] = cur
        return lg, v

    op = _openings(N, nir)
    res = Arena(ea, eb, player, "e0", eval_seed_b=7, seed=seed).play(op)

    def table_eval(board, to_move, last_move):
        o = np.zeros((3, N, N), np.float32)
        o[0] = board == to_move; o[1] = board == -to_move
        if last_move >= 0:
            o[2, last_move // N, last_move % N] = 1.0
        return table[o.tobytes()]
    oracle.set_eval_callback(table_eval)
    try:
        cfgs = (oracle.make_config(board_size=N, n_in_row=nir, num_simulations=S, num_top_actions=8, eval_kind=3, accum_dtype=1),
                oracle.make_config(board_size=N, n_in_row=nir, num_simulations=S, num_top_actions=8, eval_seed=7))
        _check_against(res, _host_match(op, N, nir, _oracle_search(cfgs), _Noise(ea, seed)))
    finally:
        oracle.set_eval_callback(None)
    for t in range(res.moves.shape[0]):                   # the results table is what the move log replays to
        o = t // 2
        g = GomokuGame(board_size=N, n_in_row=nir)
        g.board = op.boards[o].reshape(N, N).copy()
        g.current_player, g.move_count = int(op.players[o]), int(op.move_counts[o])
        g.last_move = None if op.last_moves[o] < 0 else divmod(int(op.last_moves[o]), N)
        assert res.a_colour[t] == (g.current_player if t % 2 == 0 else -g.current_player)
        for k in range(res.length[t]):
            assert g.get_game_ended() is None
            a = int(res.moves[t, k])
            assert 0 <= a < N * N and g.board[a // N, a % N] == 0
            g.do_move(a)
        assert g.get_game_ended() == res.winner[t]
        rec = res.game_record(t)
        assert rec.actions == res.moves[t, :res.length[t]].tolist() and len(rec.observations) == res.length[t]


def test_colour_balance_and_counts():
    """Every opening is played exactly twice, once with each player first, and W/D/L and pair counts equal a host
    recount of the results table."""
    from datou_gomoku_muzero_b200.arena import Arena, random_openings
    from datou_gomoku_muzero_b200.engine import SearchEngine
    N, nir, G = 6, 4, 8
    ea = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=16, num_top_actions=4)
    eb = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=48, num_top_actions=8)
    op = random_openings(12, 1, N, seed=5, n_in_row=nir)
    res = Arena(ea, eb, eval_seed_a=1, eval_seed_b=1, seed=4).play(op)
    O = op.boards.shape[0]
    assert len(res) == 2 * O and res.finished.all()
    assert np.array_equal(np.bincount(res.opening, minlength=O), np.full(O, 2))
    assert res.a_first[0::2].all() and not res.a_first[1::2].any()
    assert np.array_equal(res.a_colour[0::2], op.players) and np.array_equal(res.a_colour[1::2], -op.players)
    w = d = l = 0
    by_colour = {1: [0, 0, 0], -1: [0, 0, 0]}
    pairs = np.zeros(5, np.int64)
    for o in range(O):
        pts = 0.0
        for t in (2 * o, 2 * o + 1):
            c, win = int(res.a_colour[t]), int(res.winner[t])
            k = 1 if win == 0 else (0 if win == c else 2)
            by_colour[c][k] += 1
            pts += (1.0, 0.5, 0.0)[k]
        pairs[int(round(pts * 2))] += 1
    w, d, l = (by_colour[1][i] + by_colour[-1][i] for i in range(3))
    assert res.wdl() == (w, d, l) and res.wdl(1) == tuple(by_colour[1]) and res.wdl(-1) == tuple(by_colour[-1])
    assert np.array_equal(res.pairs(), pairs)
    assert res.score() == pytest.approx((w + 0.5 * d) / (2 * O))


def test_arena_rejects_mismatched_engines():
    from datou_gomoku_muzero_b200.arena import Arena
    from datou_gomoku_muzero_b200.engine import SearchEngine
    ea = SearchEngine(4, board_size=6, n_in_row=4, num_simulations=8, num_top_actions=4)
    for other in (SearchEngine(5, board_size=6, n_in_row=4, num_simulations=8, num_top_actions=4),
                  SearchEngine(4, board_size=7, n_in_row=4, num_simulations=8, num_top_actions=4),
                  SearchEngine(4, board_size=6, n_in_row=5, num_simulations=8, num_top_actions=4)):
        with pytest.raises(ValueError):
            Arena(ea, other)
    with pytest.raises(ValueError):
        Arena(ea, ea)
    eb = SearchEngine(4, board_size=6, n_in_row=4, num_simulations=8, num_top_actions=4)
    with pytest.raises(ValueError):
        Arena(ea, eb, logit_div_a=12)
    with pytest.raises(ValueError):
        Arena(ea, eb, evaluator_b=(lambda x: x, lambda x, y: x))      # a learned-dynamics pair needs a MuZero-mode engine
