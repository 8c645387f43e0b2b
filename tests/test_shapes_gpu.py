"""The kernels at every board size and row length the C ABI accepts (board_size 1..19, n_in_row 1..14, num_top_actions
1..32), not only at the 6, 9, 15 and 19 of the golden vectors.  With A = N*N the kernels change shape at NW = ceil(A/64)
bitboard words and NC = ceil(A/128) lane chunks; SEARCH_BOARDS holds one board of every (NW, NC) pair and edge:

    N      A        NW  NC  what it exercises
    1..5   1..25    1   1   fewer cells than lanes; fewer cells than K on an empty board; N = 1
    7, 8   49, 64   1   1   odd board (a centre cell); A a multiple of 64 (the last bitboard word full)
    11     121      2   1   one lane chunk almost full
    12, 13 144, 169 3   2   three bitboard words; the second chunk nearly empty at 12
    16     256      4   2   full words and full chunks: no padding lanes
    17     289      5   3   five bitboard words

Every reference is the CPU oracle (pinned to the reference goldens), tests/golden/e0_py.py, or the tactics restatement
of tests/test_shapes_cpu.py (pinned to the reference KATs).  Counts, actions, winners, root values, traces, records and
batches must match bit for bit; policies within rtol 1e-12, atol 1e-15."""
import numpy as np
import pytest

from test_shapes_cpu import classify_ref, crafted_lines, tactic_patterns

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-12, 1e-15
BOARDS = list(range(1, 20))
SEARCH_BOARDS = [1, 2, 3, 4, 5, 7, 8, 11, 12, 13, 16, 17]
ROWS = [1, 2, 3, 4, 5, 6, 7, 10, 14]
# the row length each search board runs with: short rows (terminal leaves everywhere), the reference's 5, the walking
# branch of the win test (>= 6) and rows longer than the board (no win possible)
SEARCH_ROW = {1: 1, 2: 2, 3: 3, 4: 3, 5: 6, 7: 5, 8: 6, 11: 5, 12: 7, 13: 10, 16: 5, 17: 14}


def _fill(N, k, rs):
    """A position with k stones played alternately from black on random cells: (board [A], to move, last move, count)."""
    A = N * N
    b = np.zeros(A, np.int8)
    p, last = 1, -1
    for a in rs.permutation(A)[:k]:
        b[a] = p; last = int(a); p = -p
    return b, p, last, k


def _roots(N, G, K, rs):
    """G roots: the full board (the sentinel), one empty cell, fewer than K empty cells, the empty board, then random."""
    A = N * N
    ks = [A, A - 1, max(0, A - max(1, K // 2)), 0] + [int(rs.randint(0, A)) for _ in range(G - 4)]
    pos = [_fill(N, k, rs) for k in ks[:G]]
    return (np.stack([p[0] for p in pos]), np.array([p[1] for p in pos], np.int8), np.array([p[2] for p in pos], np.int32),
            np.array([p[3] for p in pos], np.int32))


def _same_search(tag, got, want):
    pol, val, act, vis = got
    opol, oval, oact, ovis = want
    assert np.array_equal(vis, ovis), f"{tag}: visit counts"
    assert np.array_equal(act, oact), f"{tag}: actions {act} vs {oact}"
    assert np.array_equal(val, oval), f"{tag}: root value bits"
    np.testing.assert_allclose(pol, opol, rtol=RTOL, atol=ATOL, err_msg=tag)


@pytest.mark.parametrize("N", SEARCH_BOARDS)
def test_search_matches_oracle(N):
    """Fused and stepwise AlphaZero-mode searches and the fused MuZero-mode search against oracle.search_batch, with the
    per-simulation (leaf action, depth) trace of one game against oracle.search(trace=True).  Float64 and float32
    accumulation, quantised and dense logits, K = 16 everywhere and K = 32 / K = 1 on the small boards."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    A, nir, S, G, seed, T = N * N, SEARCH_ROW[N], 64, 16, 23, 4
    rs = np.random.RandomState(100 + N)
    runs = [(16, acc, div) for acc in ("float64", "float32") for div in (16, 0)]
    if N <= 5:
        runs += [(32, "float64", 16), (1, "float32", 0), (1, "float64", 16)]
    for K, accum, div in runs:
        boards, players, last, mc = _roots(N, G, K, rs)
        gumbel = rs.gumbel(0, 1, (G, A))
        for mode in ("AlphaZero", "MuZero"):
            cfg = oracle.make_config(board_size=N, n_in_row=nir, num_simulations=S, num_top_actions=K, eval_seed=seed,
                                     logit_div=div, accum_dtype=int(accum == "float32"), mode=int(mode == "MuZero"))
            want = oracle.search_batch(cfg, boards, players, last, mc, gumbel)
            ref = oracle.search(cfg, boards[T], players[T], last[T], mc[T], gumbel[T], trace=True)
            n = ref["n_evals"]
            eng = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=S, num_top_actions=K, mode=mode,
                               accum_dtype=accum)
            paths = [("fused", eng.search_e0)] + ([("stepwise", eng.search_stepwise_e0)] if mode == "AlphaZero" else [])
            for path, run in paths:
                tag = f"N={N} nir={nir} K={K} {accum} div={div} {mode} {path}"
                eng.set_roots(boards, players, last, mc)
                ta, td = run(torch.from_numpy(gumbel).cuda(), seed, div, trace=True)
                got = [t.cpu().numpy() for t in eng.finalize()]
                _same_search(tag, got, want)
                assert got[2][0] == -1 and not got[0][0].any() and got[1][0] == 0.0, f"{tag}: full-board sentinel"
                assert np.array_equal(ta[T].cpu().numpy()[:n], ref["leaf_actions"]), f"{tag}: leaf action trace"
                assert np.array_equal(td[T].cpu().numpy()[:n], ref["leaf_depths"]), f"{tag}: leaf depth trace"
                b2, p2, l2, m2 = (t.cpu().numpy() for t in eng.get_roots())
                assert np.array_equal(b2.reshape(G, A), boards) and np.array_equal(p2, players), f"{tag}: roots changed"
                assert np.array_equal(l2, last) and np.array_equal(m2, mc), f"{tag}: roots changed"


@pytest.mark.parametrize("N", [4, 8, 12, 17])
def test_muzero_device_search_matches_oracle(N):
    """MuZero mode on the device with the hidden-state pool and TorchE0 as the evaluator."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.muzero import MuZeroDeviceSearch, TorchE0
    from oracle import oracle
    A, S, G, seed = N * N, 32, 10, 41
    rs = np.random.RandomState(200 + N)
    boards, players, last, mc = _roots(N, G, 16, rs)
    gumbel = rs.gumbel(0, 1, (G, A))
    eng = SearchEngine(G, board_size=N, n_in_row=SEARCH_ROW[N], num_simulations=S, mode="MuZero")
    eng.set_roots(boards, players, last, mc)
    e0 = TorchE0(N, seed=seed)
    MuZeroDeviceSearch(eng, e0.initial, e0.recurrent).search(torch.from_numpy(gumbel).cuda())
    got = [t.cpu().numpy() for t in eng.finalize()]
    cfg = oracle.make_config(board_size=N, n_in_row=SEARCH_ROW[N], num_simulations=S, mode=1, eval_seed=seed)
    _same_search(f"N={N} MuZeroDeviceSearch", got, oracle.search_batch(cfg, boards, players, last, mc, gumbel))


def _win_cases(N, nir, rs):
    """(board after the move [N,N], move (r, c)) pairs: random boards at several densities and crafted lines."""
    cases = []
    for dens in (0.3, 0.6, 0.9, 1.0):
        for _ in range(6):
            b = np.where(rs.random_sample((N, N)) < dens, np.where(rs.randint(2, size=(N, N)) == 1, 1, -1), 0).astype(np.int8)
            r, c = int(rs.randint(N)), int(rs.randint(N))
            if b[r, c] == 0:
                b[r, c] = 1 if rs.randint(2) else -1
            cases.append((b, (r, c)))
    return cases + crafted_lines(N, nir, rs)


@pytest.mark.parametrize("N", [1, 2, 3, 5, 8, 12, 16, 19])
def test_game_step_win_rule_matches_oracle(N):
    """do_move + get_game_ended on the device (the play kernel's lane-window win test) against oracle.game_ended, for
    every row length of the table, with lines of n_in_row - 1 .. 2 n_in_row + 3 stones, gaps, and lines on the edges and
    in the corners; then the roots against numpy."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    A = N * N
    rs = np.random.RandomState(300 + N)
    wins = draws = 0
    for nir in ROWS:
        cases = _win_cases(N, nir, rs)
        G = len(cases)
        after = np.stack([b.reshape(A) for b, _ in cases])
        acts = np.array([r * N + c for _, (r, c) in cases], np.int32)
        colour = after[np.arange(G), acts].copy()
        before = after.copy()
        before[np.arange(G), acts] = 0
        mc = (after != 0).sum(1).astype(np.int32)
        eng = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=2)
        eng.set_roots(before, colour, np.full(G, -1, np.int32), mc - 1)
        w = eng.game_step(acts).cpu().numpy()
        want = np.array([2 if x is None else x for x in (oracle.game_ended(after[g].reshape(N, N), nir, int(acts[g]), int(mc[g]))
                                                       for g in range(G))])
        bad = np.flatnonzero(w != want)
        assert not len(bad), f"N={N} nir={nir}: game {bad[0]} winner {w[bad[0]]} vs {want[bad[0]]}"
        b2, p2, l2, m2 = (t.cpu().numpy() for t in eng.get_roots())
        assert np.array_equal(b2.reshape(G, A), after) and np.array_equal(p2, -colour), (N, nir)
        assert np.array_equal(l2, acts) and np.array_equal(m2, mc), (N, nir)
        wins += int((np.abs(want) == 1).sum()); draws += int((want == 0).sum())
    assert wins > 0 and (N < 5 or draws > 0)


# (N, n_in_row, mode, accumulation) of the self-play games compared move for move with the oracle's game loop
SELFPLAY = [(1, 1, "AlphaZero", "float64"), (1, 5, "AlphaZero", "float32"), (2, 2, "AlphaZero", "float64"),
            (3, 3, "AlphaZero", "float32"), (4, 3, "AlphaZero", "float64"), (5, 6, "AlphaZero", "float32"),
            (7, 5, "AlphaZero", "float64"), (8, 5, "AlphaZero", "float32"), (8, 6, "AlphaZero", "float64"),
            (11, 5, "AlphaZero", "float32"), (12, 5, "MuZero", "float64"), (13, 7, "AlphaZero", "float32"),
            (16, 5, "AlphaZero", "float64"), (17, 5, "AlphaZero", "float32"), (19, 14, "AlphaZero", "float64")]


@pytest.mark.parametrize("N,nir,mode,accum", SELFPLAY)
def test_selfplay_games_match_oracle(N, nir, mode, accum):
    """Whole games of the persistent self-play kernel against oracle.selfplay_game with the kernel's own Gumbel noise
    regenerated per move (as tests/test_selfplay_gpu.py does at 6x6 and 9x9)."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    from oracle import oracle
    from test_selfplay_gpu import _noise_for_game
    A, S, G, seed, nseed = N * N, 16, 6, 5, 70 + N
    eng = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=S, mode=mode, accum_dtype=accum)
    sp = SelfPlayEngine(eng, "e0", seed=seed, noise_seed=nseed)
    traj = TrajectoryStore(eng, extra_slots=2 * G)
    first = {}
    for _ in range(12):
        sp.play(moves_per_game=max(4, A // 2), traj=traj, restart=True)
        for r in traj.harvest():
            first.setdefault(r["game"], r)
        if len(first) == G:
            break
    assert len(first) == G, f"only {len(first)} of {G} games finished"
    cfg = oracle.make_config(board_size=N, n_in_row=nir, num_simulations=S, eval_seed=seed, mode=int(mode == "MuZero"),
                             accum_dtype=int(accum == "float32"))
    for g, r in sorted(first.items()):
        assert r["start_move_count"] == 0 and not r["start_board"].any() and r["start_player"] == 1
        o = oracle.selfplay_game(cfg, np.concatenate([_noise_for_game(eng, g, r["length"], nseed), np.zeros((1, A))]))
        assert o["T"] == r["length"], (g, o["T"], r["length"])
        assert np.array_equal(o["actions"], r["actions"]) and o["winner"] == r["winner"], g
        assert np.array_equal(o["values"], r["values"]), g
        np.testing.assert_allclose(r["policies"], o["policies"], rtol=RTOL, atol=ATOL)
        if nir > N:
            assert r["winner"] == 0 and r["length"] == A, g       # no row fits: every game fills the board
        if (N, nir) == (19, 14):
            assert r["winner"] == 0 or r["length"] >= 27, g      # a row of 14 takes at least 27 moves


def _planes(board, player, last):
    N = board.shape[0]
    out = np.zeros((3, N, N), np.float32)
    out[0][board == player] = 1.0
    out[1][board == -player] = 1.0
    if last >= 0:
        out[2, last // N, last % N] = 1.0
    return out


def test_root_obs_and_e0_every_board_size():
    """gmz_root_obs into float32 NCHW and into channels_last bf16 (obs_write_nhwc_bf16) against the numpy planes of
    game.py:26-33, and gmz_e0_eval_obs on them against e0_py, for N = 1..19."""
    import torch
    import e0_py
    from datou_gomoku_muzero_b200.engine import SearchEngine
    rs = np.random.RandomState(400)
    for N in BOARDS:
        A, G = N * N, 8
        boards = np.zeros((G, A), np.int8)
        for g in range(1, G):
            boards[g] = rs.randint(-1, 2, size=A)
        boards[G - 1] = np.where(np.arange(A) % 3 == 0, -1, 1)           # full
        players = np.where(np.arange(G) % 2 == 0, 1, -1).astype(np.int8)
        last = np.array([-1] + [int(rs.randint(A)) for _ in range(G - 1)], np.int32)
        last[2] = A - 1
        eng = SearchEngine(G, board_size=N, num_simulations=2)
        eng.set_roots(boards, players, last, (boards != 0).sum(1).astype(np.int32))
        want = np.stack([_planes(boards[g].reshape(N, N), players[g], last[g]) for g in range(G)])
        f32 = eng.root_obs().cpu().numpy()
        assert np.array_equal(f32, want), N
        bf = eng.obs_buffer_bf16()
        eng.root_obs(bf)
        assert np.array_equal(bf.float().cpu().numpy(), want), N
        for div in (16, 0, 3):
            seed = int(rs.randint(1 << 30))
            lg, v = (x.cpu().numpy() for x in eng.e0_eval(torch.from_numpy(want).cuda(), seed, div))
            for g in range(G):
                l2, v2 = e0_py.heads(e0_py.hash_obs(want[g], seed), A, div)
                assert np.array_equal(lg[g], l2) and v[g] == v2, (N, div, g)


def _tactics_boards(N, rs):
    """(board [N,N], player) pairs: random boards at several densities and crafted runs of 2..5 stones against every
    edge and corner (off the board counts as an opponent stone)."""
    out = []
    for dens in (0.15, 0.35, 0.6):
        for _ in range(2):
            b = np.where(rs.random_sample((N, N)) < dens, np.where(rs.randint(2, size=(N, N)) == 1, 1, -1), 0).astype(np.int8)
            out.append((b, 1 if rs.randint(2) else -1))
    for run in (3, 4):
        for b, (r, c) in crafted_lines(N, run, rs)[::5]:
            out.append((b, int(b[r, c]) if rs.randint(4) else -int(b[r, c])))
    return out


@pytest.mark.parametrize("N", BOARDS)
def test_tactics_match_restatement(N):
    """classify_boards (k_tactics) and record_flags (k_records_tactics) against the restatement of the reference's
    classifier, for every row length including the walking branch (n_in_row >= 6) and rows longer than the board."""
    from datou_gomoku_muzero_b200.tactics import classify_boards, record_flags
    from test_records_tactics_gpu import _record_block
    A = N * N
    rs = np.random.RandomState(500 + N)
    pairs = _tactics_boards(N, rs)
    boards = np.stack([b.reshape(A) for b, _ in pairs])
    players = np.array([p for _, p in pairs], np.int8)
    pats = [tactic_patterns(b, p) for b, p in pairs]
    seen = set()
    for nir in (1, 2, 3, 4, 5, 6, 7, 14):
        want = np.stack([classify_ref(b, p, nir, pt) for (b, p), pt in zip(pairs, pats)])
        got = classify_boards(boards, players, N, n_in_row=nir).cpu().numpy()
        bad = np.flatnonzero((got != want).any(1))
        assert not len(bad), f"N={N} nir={nir} board {bad[0]}: {got[bad[0]]} vs {want[bad[0]]}"
        seen |= set(np.unique(want).tolist())
        rows, flags = [], []
        for (b, p), cls in zip(pairs, want):
            base = int((cls > 0).any()) | 2 * int((cls == 1).any())
            for k in (1, 2, 3):
                cells = np.flatnonzero(cls == k)
                if len(cells):
                    rows.append((b, p, int(cells[int(rs.randint(len(cells)))]))); flags.append(base | 4)
            quiet = np.flatnonzero((b.reshape(A) == 0) & (cls == 0))
            if len(quiet):
                rows.append((b, p, int(quiet[0]))); flags.append(base)
            for a in (-1, A):
                rows.append((b, p, a)); flags.append(base)
        got = record_flags(_record_block(N, rows), N, n_in_row=nir).cpu().numpy()
        assert np.array_equal(got, np.array(flags, np.uint8)), (N, nir)
    assert 1 in seen and (N < 6 or {2, 3} <= seen)      # an open four needs six cells in a line


# ---------------------------------------------------------------------------------------------- records and the ring
RING_BOARDS = [(7, 4), (8, 5), (12, 5), (13, 6), (16, 5), (17, 5)]


def _played_packs(N, nir, G=8, S=8, min_games=8, seed=3):
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=S)
    sp = SelfPlayEngine(eng, "e0", seed=seed, noise_seed=seed + 1)
    traj = TrajectoryStore(eng, extra_slots=G)
    packs = []
    for _ in range(30):
        sp.play(moves_per_game=N * N // 3, traj=traj, sink=packs.append)
        if sum(len(p) for p in packs) >= min_games:
            return packs
    raise AssertionError("too few games finished")


def _check_records_replay(pg, N, nir):
    """Every record of every game against a numpy replay of the game from the empty board."""
    from datou_gomoku_muzero_b200.config import config
    from oracle import oracle
    A = N * N
    for i in range(len(pg)):
        r = pg.game(i)
        T, winner = len(r), int(pg.table[i][3])
        board, player, last = np.zeros((N, N), np.int8), 1, -1
        for t in range(T):
            tag = (N, i, t)
            assert np.array_equal(r["board"][t], board), tag
            assert np.array_equal(r["obs"][t], _planes(board, player, last)), tag
            assert (r["to_move"][t], r["last_move"][t], r["move_count"][t], r["t"][t]) == (player, last, t, t), tag
            assert r["length"][t] == T and r["winner"][t] == winner, tag
            a = int(r["action"][t])
            assert 0 <= a < A and board[a // N, a % N] == 0, tag
            board[a // N, a % N] = player
            player, last = -player, a
        ended = oracle.game_ended(board, nir, last, T)
        assert ended is not None and ended == winner, (N, i)
        rew = oracle.final_rewards(T, winner)
        assert np.array_equal(r["reward"], rew), (N, i)
        vt = oracle.n_step_returns(rew, r["search_value"], config.DISCOUNT, config.N_STEPS)
        assert np.array_equal(r["value_target"], vt), (N, i)


def _check_augmented(tag, batch, k, flip, slices):
    """A trainer batch built with the symmetry (k, flip) against oracle.augment_batch over the host training slices."""
    from oracle import oracle
    obs, act, rew, pi, val = (x.cpu().numpy() for x in batch)
    o0, a0, p0 = (np.stack([getattr(s, f) for s in slices]) for f in ("observation", "action_history", "policy_history"))
    eo, ea, ep = oracle.augment_batch(o0, a0, p0, k, flip)
    assert np.array_equal(obs, eo) and np.array_equal(pi, ep), tag
    assert np.array_equal(act[a0 != -1], ea[a0 != -1]) and (act[a0 == -1] == -1).all(), tag
    assert np.array_equal(rew, np.stack([s.reward_history for s in slices])), tag
    assert np.array_equal(val, np.stack([s.value_history for s in slices])), tag


@pytest.mark.parametrize("N,nir", RING_BOARDS)
def test_packed_records_and_ring_batches(N, nir):
    """gmz_traj_pack records of kernel-played games against a numpy replay (boards, planes, header fields, final rewards
    and n-step targets from the oracle); DeviceReplayBuffer.batch over them for all eight (rot_k, flip) against
    oracle.augment_batch of the host-cut training slices."""
    import torch
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    packs = _played_packs(N, nir)
    slices = []
    buf = DeviceReplayBuffer(sum(p.n_moves for p in packs), N)
    for pg in packs:
        _check_records_replay(pg, N, nir)
        buf.add_packed(pg)
        for i in range(len(pg)):
            slices += pg.training_slices(i)
    n = len(slices)
    assert n == len(buf)
    rs = np.random.RandomState(600 + N)
    pos = np.concatenate([[0, n - 1], rs.choice(n, 40, replace=False)])
    for k in range(4):
        for flip in (False, True):
            _check_augmented((N, k, flip), buf.batch(torch.as_tensor(pos, device="cuda"), k, flip), k, flip,
                             [slices[int(p)] for p in pos])


@pytest.fixture
def _per():
    from datou_gomoku_muzero_b200.config import config
    saved = config.ENABLE_PER
    config.ENABLE_PER = True
    yield
    config.ENABLE_PER = saved


@pytest.mark.parametrize("N,nir", RING_BOARDS)
def test_ring_checkpoint_round_trip(tmp_path, _per, N, nir):
    """state_dict / load_state_dict of a wrapped ring whose oldest game is cut: every ring position's meaningful bytes,
    the tree, write_ptr, count and max_priority come back identical, and so do sampled batches."""
    from test_ring_checkpoint_gpu import _assert_same, _fill, _round_trip, _same_batches, _train_a_little
    A = N * N
    buf, _ = _fill(N, 16, 8, 3 * A + 17, moves=max(8, A // 4), n_in_row=nir)
    _train_a_little(buf)
    out = _round_trip(buf, tmp_path)
    _assert_same(buf, out)
    _same_batches(buf, out, B=32)


def test_ring_reanalysis_at_twelve():
    """DeviceReplayBuffer.reanalyse at 12x12 (three bitboard words, two lane chunks) against the host driver."""
    from test_ring_reanalysis_gpu import _check_parity, _engines, _expected, _fill, _host
    N, S, G = 12, 8, 24
    buf = _fill(N, 16, S, 700, moves=36)
    snap, tree0 = _host(buf), buf.sum_tree.tree.clone()
    start, n = buf.reanalyse(_engines(N, (G, G), S), eval_seed=5, noise_seed=7)
    assert (start, n) == (buf.sum_tree.write_ptr, buf.capacity)
    pol, val, vt = _expected(snap, start, n, _engines(N, (G, G), S), eval_seed=5, noise_seed=7)
    _check_parity(buf, snap, tree0, start, n, pol, val, vt)
