"""The reference-facing classes (datou_gomoku_muzero_b200.mcts) exercised the way the reference's
own tests/test_mcts_logic.py exercises mcts.py -- same constructor, same queue shim, same
assertions -- plus bit-exact agreement with the goldens when driven exactly like the reference
(E0 behind the queue protocol, np.random.seed for the Gumbel draw)."""
import numpy as np
import pytest

from _golden_util import load_search_cases

pytestmark = pytest.mark.gpu


@pytest.fixture
def cfg():
    from datou_gomoku_muzero_b200.config import config
    saved = dict(vars(config))
    yield config
    for k, v in saved.items():
        setattr(config, k, v)


def _apply(config, c):
    config.BOARD_SIZE, config.N_IN_ROW, config.ACTION_SPACE_SIZE = c["N"], c["n_in_row"], c["N"] ** 2
    config.NUM_SIMULATIONS, config.NUM_TOP_ACTIONS = c["S"], c["K"]
    config.C_VISIT, config.C_SCALE = c["c_visit"], c["c_scale"]
    config.VALUE_MINMAX_DELTA, config.DISCOUNT = c["delta"], c["discount"]


def _game(c):
    from datou_gomoku_muzero_b200.game import GomokuGame
    g = GomokuGame(board_size=c["N"], n_in_row=c["n_in_row"])
    g.board = c["board"].reshape(c["N"], c["N"]).copy()
    g.current_player, g.move_count = c["player"], c["move_count"]
    g.last_move = None if c["last_move"] < 0 else (c["last_move"] // c["N"], c["last_move"] % c["N"])
    return g


@pytest.mark.parametrize("mode", ["az", "mz"])
@pytest.mark.parametrize("N", [6, 9])
def test_search_game_reproduces_reference(cfg, mode, N):
    from e0_py import E0Queue
    from datou_gomoku_muzero_b200.mcts import AlphaZeroMCTS, MuZeroMCTS
    for c in load_search_cases(mode, N)[::2]:
        _apply(cfg, c)
        q = E0Queue(seed=c["seed"], logit_div=c["logit_div"], kind=c["kind"], const_value=c["const_value"],
                    const_reward=c["const_reward"], value_dtype=np.float32 if c["vdtype"] else None)
        q.set_action_space(N * N)
        eng = (AlphaZeroMCTS if mode == "az" else MuZeroMCTS)(0, q, q)
        g = _game(c)
        board0 = g.board.copy()
        np.random.seed(c["seed"])
        policy, value, action = eng.search(g)
        tag = f"{mode} N={N} case {c['idx']} div={c['logit_div']} f32={c['vdtype']}"
        assert np.array_equal(g.board, board0), tag + ": search mutated the game"
        assert isinstance(value, np.float32) == bool(c["vdtype"]), tag       # the value's type follows the evaluator's, as in the reference
        assert float(value) == c["value"], tag
        assert isinstance(policy, np.ndarray) and policy.dtype == np.float64 and policy.shape == (N * N,)
        assert isinstance(action, int) and action == c["action"], tag
        assert isinstance(value, (float, np.floating))
        np.testing.assert_allclose(value, c["value"], rtol=1e-12, atol=1e-15, err_msg=tag)
        np.testing.assert_allclose(policy, c["policy"], rtol=1e-12, atol=1e-15, err_msg=tag)
        assert q.n_initial == c["n_initial"] and q.n_recurrent == c["n_recurrent"], tag   # same request pattern


def test_reference_behaviour_tests(cfg):
    """Restates tests/test_mcts_logic.py:116-165 against this package."""
    from e0_py import E0Queue
    from datou_gomoku_muzero_b200.game import GomokuGame
    from datou_gomoku_muzero_b200.mcts import AlphaZeroMCTS, MuZeroMCTS
    cfg.BOARD_SIZE, cfg.ACTION_SPACE_SIZE, cfg.NUM_SIMULATIONS = 6, 36, 15
    q = E0Queue(kind=1, const_value=0.5); q.set_action_space(36)
    AlphaZeroMCTS(0, q, q).search(GomokuGame())
    assert q.n_initial == 15 and q.n_recurrent == 0
    q = E0Queue(kind=1, const_value=0.5); q.set_action_space(36)
    MuZeroMCTS(0, q, q).search(GomokuGame())
    assert q.n_initial == 1 and q.n_recurrent > 0
    rs = np.random.RandomState(0)
    g = GomokuGame()
    for a in rs.permutation(36)[:10]:
        g.do_move(int(a))
    for cls in (AlphaZeroMCTS, MuZeroMCTS):
        q = E0Queue(kind=1, const_value=0.5); q.set_action_space(36)
        policy, value, action = cls(0, q, q).search(g)
        assert isinstance(policy, np.ndarray) and abs(policy.sum() - 1.0) < 1e-5
        assert isinstance(action, int) and g.board.reshape(-1)[action] == 0
        assert -1.0 <= value <= 1.0


def test_sentinels(cfg):
    from queue import Empty
    from datou_gomoku_muzero_b200.game import GomokuGame
    from datou_gomoku_muzero_b200.mcts import AlphaZeroMCTS
    from e0_py import E0Queue
    cfg.BOARD_SIZE, cfg.ACTION_SPACE_SIZE, cfg.NUM_SIMULATIONS = 6, 36, 8

    class Dead:
        def put(self, x): pass
        def get(self, timeout=None): raise Empty
        def get_nowait(self): raise Empty
    pol, val, act = AlphaZeroMCTS(0, Dead(), Dead()).search(GomokuGame())
    assert act == -1 and val == 0.0 and not pol.any()            # root inference timed out (mcts.py:209-211)
    g = GomokuGame(); g.board[:] = 1
    q = E0Queue(); q.set_action_space(36)
    pol, val, act = AlphaZeroMCTS(0, q, q).search(g)
    assert act == -1 and val == 0.0 and not pol.any()            # no valid moves (mcts.py:214-215)
    with pytest.raises(ValueError):
        from datou_gomoku_muzero_b200.engine import SearchEngine
        SearchEngine(1, mode="Nonsense")                         # workers.py:142


def test_search_batch_host_api():
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.mcts import AlphaZeroMCTS
    from oracle import oracle
    N, S, G, seed = 9, 64, 32, 11
    A = N * N
    rs = np.random.RandomState(3)
    boards = np.zeros((G, A), np.int8); players = np.ones(G, np.int8); last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    for g in range(G):
        p = 1
        for a in rs.permutation(A)[: g]:
            boards[g, a] = p; last[g] = a; p = -p; mc[g] += 1
        players[g] = p
    gum = rs.gumbel(0, 1, (G, A))
    eng = SearchEngine(G, board_size=N, num_simulations=S)
    m = AlphaZeroMCTS.for_engine(eng, "e0", eval_seed=seed)
    pol, val, act = m.search_batch(boards.reshape(G, N, N), players, last, mc, gum)
    cfgo = oracle.make_config(board_size=N, num_simulations=S, eval_seed=seed)
    opol, oval, oact, _ = oracle.search_batch(cfgo, boards, players, last, mc, gum)
    assert np.array_equal(act, oact) and np.array_equal(val, oval)
    np.testing.assert_allclose(pol, opol, rtol=1e-12, atol=1e-15)


def test_pipelined_batch_search_matches_oracle():
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.mcts import PipelinedBatchSearch
    from oracle import oracle
    N, S, G, seed = 9, 48, 24, 21
    A = N * N
    rs = np.random.RandomState(9)
    engines = [SearchEngine(G, board_size=N, num_simulations=S) for _ in range(2)]
    pipe = PipelinedBatchSearch(engines, evaluator="e0", eval_seed=seed)
    cfgo = oracle.make_config(board_size=N, num_simulations=S, eval_seed=seed)
    batches, tickets = [], []
    for b in range(5):
        boards = np.zeros((G, A), np.int8); players = np.ones(G, np.int8)
        last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
        for g in range(G):
            p = 1
            for a in rs.permutation(A)[: (g + b) % 30]:
                boards[g, a] = p; last[g] = a; p = -p; mc[g] += 1
            players[g] = p
        gum = rs.gumbel(0, 1, (G, A))
        batches.append((boards, players, last, mc, gum))
        tickets.append(pipe.submit(*batches[-1]))
        if b >= 1:      # depth-2 pipeline: collect the previous batch while this one runs
            pol, val, act = (x.copy() for x in pipe.result(tickets[b - 1]))
            opol, oval, oact, _ = oracle.search_batch(cfgo, *batches[b - 1])
            assert np.array_equal(act, oact) and np.array_equal(val, oval), b
            np.testing.assert_allclose(pol, opol, rtol=1e-12, atol=1e-15)
    pol, val, act = pipe.result(tickets[-1])
    opol, oval, oact, _ = oracle.search_batch(cfgo, *batches[-1])
    assert np.array_equal(act, oact) and np.array_equal(val, oval)
