"""BASELINE.json full sizes (config 2: 15x15, 400 simulations, 4096 concurrent games): size-independent
properties of the search + agreement with the oracle on a random subset + fused == stepwise."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, S, K, G = 15, 400, 16, 4096
A = N * N


def _roots(G, seed=7):
    rs = np.random.RandomState(seed)
    boards = np.zeros((G, A), np.int8); players = np.ones(G, np.int8)
    last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    for g in range(G):
        k = (g * 53) % 215
        cells = rs.permutation(A)[:k]
        boards[g, cells[0::2]] = 1; boards[g, cells[1::2]] = -1
        players[g] = 1 if k % 2 == 0 else -1
        last[g] = cells[-1] if k else -1; mc[g] = k
    return boards, players, last, mc


def test_full_size_search_properties_and_oracle_subset():
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    seed = 99
    boards, players, last, mc = _roots(G)
    eng = SearchEngine(G, board_size=N, num_simulations=S, num_top_actions=K)
    gum = torch.empty((G, A), dtype=torch.float64, device="cuda")
    eng.fill_gumbel(gum, 5, 0)
    eng.set_roots(boards, players, last, mc)
    eng.search_e0(gum, seed)
    pol, val, act, vis = (t.cpu().numpy().copy() for t in eng.finalize())
    # --- properties that hold for any size
    assert (vis.sum(1) == S - 1).all()                                   # every simulation after the root went through one root child
    assert ((vis > 0).sum(1) <= K).all()                                 # only the Gumbel top-k are ever visited at the root
    assert (vis[boards != 0] == 0).all() and (pol[boards != 0] == 0).all()   # nothing on occupied cells
    np.testing.assert_allclose(pol.sum(1), 1.0, atol=1e-9)
    assert (np.abs(val) <= 1.0).all()
    assert (vis[np.arange(G), act] == vis.max(1)).all()
    assert ((vis == vis.max(1, keepdims=True)).sum(1) == 1).all()        # S=400: the maximum is strict (SURVEY App. A.9)
    # --- determinism / idempotence: same roots + noise -> same bits, search() does not mutate the roots
    eng.search_e0(gum, seed)
    pol2, val2, act2, vis2 = (t.cpu().numpy() for t in eng.finalize())
    assert np.array_equal(vis, vis2) and np.array_equal(act, act2) and np.array_equal(val, val2) and np.array_equal(pol, pol2)
    # --- oracle on a random subset
    sub = np.random.RandomState(1).choice(G, 160, replace=False)
    cfg = oracle.make_config(board_size=N, num_simulations=S, num_top_actions=K, eval_seed=seed)
    g_host = gum.cpu().numpy()
    opol, oval, oact, ovis = oracle.search_batch(cfg, boards[sub], players[sub], last[sub], mc[sub], g_host[sub])
    assert np.array_equal(vis[sub], ovis) and np.array_equal(act[sub], oact) and np.array_equal(val[sub], oval)
    np.testing.assert_allclose(pol[sub], opol, rtol=1e-12, atol=1e-15)
    # --- the stepwise kernels (external-evaluator path) give the same bits as the fused kernel
    eng.search_stepwise_e0(gum, seed)
    pol3, val3, act3, vis3 = (t.cpu().numpy() for t in eng.finalize())
    assert np.array_equal(vis, vis3) and np.array_equal(act, act3) and np.array_equal(val, val3) and np.array_equal(pol, pol3)


def test_full_size_selfplay_bookkeeping():
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng = SearchEngine(G, board_size=N, num_simulations=64, num_top_actions=K)      # fewer simulations: this checks the game loop
    sp = SelfPlayEngine(eng, "e0", seed=3, noise_seed=4)
    traj = TrajectoryStore(eng, extra_slots=512)
    total = 0
    finished = []
    for _ in range(4):
        sp.play(moves_per_game=6, traj=traj)
        total += 6 * G
        finished += traj.harvest(copy_policies=False)
    moves, nfin = eng.play_counters()
    assert moves == total and eng.tickets_idle == 0 and eng.tickets_unserved == 0, (moves, total, eng.tickets_idle, eng.tickets_unserved)
    assert nfin == len(finished)
    b, pl, lm, mcount = (t.cpu().numpy() for t in eng.get_roots())
    stones = (b.reshape(G, A) != 0).sum(1)
    assert np.array_equal(stones, mcount)                                # one stone per move, none overwritten
    assert ((b.reshape(G, A) == 1).sum(1) - (b.reshape(G, A) == -1).sum(1) == (mcount % 2)).all()
    assert (pl == np.where(mcount % 2 == 0, 1, -1)).all()
    for r in finished[:50]:
        T = r["length"]
        assert 9 <= T <= A and len(set(r["actions"].tolist())) == T      # a win needs >= 9 plies; no cell played twice
        assert r["winner"] in (-1, 0, 1) and (r["winner"] != 0 or T == A)
        if r["winner"] != 0:
            assert r["winner"] == (1 if T % 2 == 1 else -1)              # the side that moved last won


@pytest.mark.parametrize("div,accum", [(16, "float64"), (0, "float32")])
def test_full_size_games_move_for_move_against_the_oracle(div, accum):
    """The bench configuration itself -- 15x15, 400 simulations, the persistent multi-move launch with in-kernel
    restart -- compared MOVE FOR MOVE with the CPU oracle's game loop: every move, root value and the winner of the
    first finished games, policies within 1e-12 relative (quantised float64 and dense-logit float32-accumulation evaluators)."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    from oracle import oracle
    Gs, S_, seed, nseed = 96, 400, 21, 22
    eng = SearchEngine(Gs, board_size=N, num_simulations=S_, num_top_actions=K, accum_dtype=accum)
    sp = SelfPlayEngine(eng, "e0", seed=seed, logit_div=div, noise_seed=nseed)
    traj = TrajectoryStore(eng, extra_slots=Gs)
    finished = []
    for _ in range(8):                                       # several multi-move launches: games cross launch boundaries
        sp.play(moves_per_game=16, traj=traj)
        finished += traj.harvest()
        if len({r["game"] for r in finished}) >= 10:
            break
    first = {}
    for r in finished:                                       # the first game of each index starts at noise counter 0
        first.setdefault(r["game"], r)
    assert len(first) >= 8, len(first)
    cfg = oracle.make_config(board_size=N, num_simulations=S_, num_top_actions=K, eval_seed=seed, logit_div=div,
                             accum_dtype=int(accum == "float32"))
    checked = 0
    for g, r in sorted(first.items())[:10]:
        T = r["length"]
        gum = torch.empty((T, A), dtype=torch.float64, device="cuda")
        for k in range(T):
            eng.fill_gumbel(gum[k], nseed, (k * Gs + g) * A)
        o = oracle.selfplay_game(cfg, np.concatenate([gum.cpu().numpy(), np.zeros((1, A))]))
        assert o["T"] == T and o["winner"] == r["winner"], (g, o["T"], T)
        assert np.array_equal(o["actions"], r["actions"]), g
        assert np.array_equal(o["values"], r["values"]), g
        np.testing.assert_allclose(r["policies"], o["policies"], rtol=1e-12, atol=1e-15)
        checked += 1
    assert checked >= 8
