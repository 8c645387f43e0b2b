"""Plain references for the packed move records (rewards, n-step value targets, training windows under the 8
symmetries), restated here from the reference's semantics -- workers.py:144-152 (compute_n_step_returns),
183-187 (final rewards), 208-222 (training slices), 291-292 (re-analysis on float32 rewards), loss.py:37-51 (D4
augmentation) -- and checked on the CPU: against exact rational targets, against the augmentation golden, and
gather_packed_games over gloo with a truncated game.  tests/test_record_targets_gpu.py compares the record kernels
with them."""
import math
import os
import socket
from fractions import Fraction

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from _golden_util import GOLDEN_DIR

# n-step horizons and discounts the record kernels are checked at (plus T - 1, T, T + 1 for each game length T)
N_STEPS_GRID = (0, 1, 2, 3, 5, 10, 31, 64)
GAMMAS = (1.0, 0.997, 0.9, 0.5, 0.0)
TINY = 2.0 ** -149                       # smallest float32 subnormal

# search values at the float32 rounding corners: signed zeros, ties between two float32 values (round to even, both
# directions), float32 subnormals and ties below the subnormal grid, and values a hair off a tie
SPECIAL_VALUES = np.array([1.0, -1.0, 0.0, -0.0, 1 + 2.0 ** -24, -(1 + 2.0 ** -24), 1 + 3 * 2.0 ** -24, 0.5 + 2.0 ** -25,
                           -(0.75 + 3 * 2.0 ** -26), 1 - 2.0 ** -25, 1 - 3 * 2.0 ** -26, 2.0 ** -149, -2.0 ** -149,
                           2.0 ** -150, 3 * 2.0 ** -150, -5 * 2.0 ** -150, 1.5 * 2.0 ** -140, 2.0 ** -126 - 2.0 ** -150,
                           1e-45, -1e-39, 1 + 2.0 ** -24 + 2.0 ** -50, 1 + 2.0 ** -24 - 2.0 ** -50, 0.3, -0.7],
                          np.float64)


def horizons(lengths):
    return sorted(set(N_STEPS_GRID) | {x for T in lengths for x in (T - 1, T, T + 1) if x >= 0})


def final_rewards(T, winner):
    """workers.py:183-187: the last mover gets +1, the one before -1, then r[i] = -r[i + 2] backwards; 0 on a draw."""
    r = [0.0] * T
    if winner != 0 and T > 0:
        r[T - 1] = 1.0
        if T > 1:
            r[T - 2] = -1.0
        for i in range(T - 3, -1, -1):
            r[i] = -r[i + 2]
    return np.array(r, np.float32)


def selfplay_targets(rewards, values, gamma, n):
    """Self-play n-step targets (workers.py:144-152 on Python-float rewards): the reward sum in float64, in order, then
    float32(acc) + float32(v_b) * float32(gamma**n), each step rounded to float32; no bootstrap when b = t + n >= T.
    Vectorised over t only: every target keeps its own order of operations."""
    T = len(rewards)
    r = np.asarray(rewards, np.float64)
    acc = np.zeros(T, np.float64)
    for i in range(n):
        ok = np.arange(T) + i < T
        acc[ok] = acc[ok] + (gamma ** i) * r[np.arange(T)[ok] + i]
    out = acc.astype(np.float32)
    b = np.arange(T) + n
    ok = b < T
    boot = np.asarray(values, np.float64)[b[ok]].astype(np.float32) * np.float32(gamma ** n)
    out[ok] = out[ok] + boot
    return out


def reanalysis_targets(rewards, values, gamma, n):
    """Re-analysis n-step targets (workers.py:291-292: the same function on float32 rewards): every term a float32
    product float32(gamma**i) * r, summed in float32 from 0 in order, plus the float32 bootstrap product."""
    T = len(rewards)
    r = np.asarray(rewards, np.float32)
    acc = np.zeros(T, np.float32)
    for i in range(n):
        ok = np.arange(T) + i < T
        acc[ok] = acc[ok] + np.float32(gamma ** i) * r[np.arange(T)[ok] + i]
    b = np.arange(T) + n
    ok = b < T
    boot = np.zeros(T, np.float32)
    boot[ok] = np.asarray(values, np.float64)[b[ok]].astype(np.float32) * np.float32(gamma ** n)
    return acc + boot


def exact_target(rewards, values, gamma, n, t):
    """The exact rational n-step target of move t, sum_{i<n, t+i<T} gamma**i r_{t+i} + gamma**n v_{t+n} (if t+n < T),
    from the inputs the kernels get (the float64 powers gamma**i the host computes, float64 values), and m = the
    largest magnitude among its terms and partial sums."""
    T = len(rewards)
    acc, m = Fraction(0), Fraction(0)
    for i in range(min(n, T - t)):
        term = Fraction(gamma ** i) * Fraction(float(rewards[t + i]))
        acc += term
        m = max(m, abs(term), abs(acc))
    if t + n < T:
        term = Fraction(gamma ** n) * Fraction(float(values[t + n]))
        acc += term
        m = max(m, abs(term), abs(acc))
    return acc, m


def ulp32(x):
    """Spacing of float32 values at magnitude |x| (the subnormal spacing 2^-149 at and below 2^-126)."""
    x = abs(float(x))
    if x < 2.0 ** -126:
        return TINY
    return 2.0 ** (math.frexp(x)[1] - 24)


# k, the roundings on the path of one target with `terms` = min(n, T - t) reward terms (the first add, 0 + x, is exact).
# Self-play: terms - 1 float64 adds, the cast of the sum, the casts of gamma**n and of v, the product and the final add:
# k = terms + 4 <= n + 4.  Re-analysis: the cast of gamma**i per term (the product with r in {-1, 0, 1} is exact),
# terms - 1 float32 adds, then the same four bootstrap roundings: k = 2 terms + 3 <= 2n + 3.
# Bound: a rounding to float32 moves its quantity q by at most 1/2 ulp32(q) (a subnormal result by at most 2^-150 =
# ulp32(0) / 2), a float64 rounding by far less.  Every rounded q is within a hair of a term, a partial sum, the final
# target (all <= m in magnitude) or of gamma**n, v (<= 1, entering the target multiplied by the other, <= 1); so |q| < 2m
# for those of the first kind, and an error of the second kind reaches the target scaled to at most 2^-24 (1 + 2^-23)
# of the term.  Either way one rounding costs at most ulp32(m) (1 + 2^-23), and errors add up unscaled or scaled down:
# |target - exact| <= k * ulp32(m) * (1 + 2^-22).
def rounding_count(n, T, t, reanalysis):
    terms = min(n, T - t)
    return 2 * terms + 3 if reanalysis else terms + 4


def apply_symmetry(planes, k, flip):
    """torch.rot90(x, k, dims=(-2, -1)) then a left-right flip, as calculate_loss augments planes (loss.py:37-44)."""
    out = np.rot90(planes, k, axes=(-2, -1))
    return np.ascontiguousarray(np.flip(out, -1) if flip else out)


def symmetry_action(a, N, k, flip):
    """loss.py:46-51 as written (for k = 1, 3 the opposite quarter turn of the planes'); padding (-1) stays -1."""
    a = np.asarray(a, np.int64)
    rows, cols = a // N, a % N
    if k == 1:
        rows, cols = cols, N - 1 - rows
    elif k == 2:
        rows, cols = N - 1 - rows, N - 1 - cols
    elif k == 3:
        rows, cols = N - 1 - cols, rows
    if flip:
        cols = N - 1 - cols
    return np.where(a >= 0, rows * N + cols, -1).astype(np.int32)


def game_windows(obs, policy, action, reward, value_target, U):
    """workers.py:208-222: the U + 1 window of every move t of one game, zero padded (actions -1) past its end."""
    T = len(action)
    A = policy.shape[1]
    pad = lambda x, k, fill=0: np.concatenate([x, np.full((k,) + x.shape[1:], fill, x.dtype)])
    o, p = pad(np.asarray(obs, np.float32), U + 1), pad(np.asarray(policy, np.float64), U + 1)
    a, r = pad(np.asarray(action, np.int32), U, -1), pad(np.asarray(reward, np.float32), U)
    v = pad(np.asarray(value_target, np.float32), U + 1)
    idx1 = np.arange(T)[:, None] + np.arange(U + 1)[None, :]
    idx0 = np.arange(T)[:, None] + np.arange(U)[None, :]
    return o[idx1], a[idx0].reshape(T, U), r[idx0].reshape(T, U), p[idx1].reshape(T, U + 1, A), v[idx1]


def augment_windows(obs, act, pi, N, k, flip):
    """Windows -> what the trainer sees under symmetry (k, flip): planes and policies turned, actions by loss.py."""
    pis = apply_symmetry(pi.reshape(pi.shape[:-1] + (N, N)), k, flip).reshape(pi.shape)
    return apply_symmetry(obs, k, flip), symmetry_action(act, N, k, flip), pis


def make_game(rs, N, stones, player, T, winner, game_index):
    """One game to inject into a trajectory store, host arrays: `stones` stones of alternating colours already on the
    board with `player` to move, T distinct empty cells played (all of them for a draw, winner = 0), float64 search
    values mostly at the rounding corners, random policies; a win goes to the last mover."""
    A = N * N
    board = np.zeros(A, np.int8)
    cells = rs.permutation(A)
    p = 1 if stones % 2 == 0 else -1
    for c in cells[:stones]:
        board[c] = p
        p = -p
    last = int(cells[stones - 1]) if stones else -1
    empty = cells[stones:]
    T = min(T, len(empty)) if winner != 0 else len(empty)
    actions = rs.permutation(empty)[:T].astype(np.int32)
    vals = np.where(rs.rand(T) < 0.6, SPECIAL_VALUES[rs.randint(len(SPECIAL_VALUES), size=T)], rs.uniform(-1, 1, T))
    pol = rs.dirichlet(np.ones(A), size=T)
    pol[rs.rand(T) < 0.2] = 0.0
    pol[:, rs.randint(A)] = 2.0 ** -1074                        # a float64 subnormal survives the copy
    last_mover = player if T % 2 == 1 else -player
    return dict(start_board=board, start_player=player, start_mc=stones, start_last=last, actions=actions,
                values=vals.astype(np.float64), policies=pol, winner=last_mover if winner else 0, game=game_index)


def make_games(N, seed):
    """The test games: lengths 1 (the n_in_row = 1 first-move win), 2, every residue mod 4, a draw that fills the
    board and a game from the empty board to its last cell; mid-game starts with either side to move."""
    rs = np.random.RandomState(seed)
    A = N * N
    games = [make_game(rs, N, 0, 1, 1, 1, 0), make_game(rs, N, 5, -1, 2, 1, 1)]
    for j, T in enumerate((8, 13, 22, 15, 4, 3, 7, 12)):       # residues 0, 1, 2, 3 mod 4 twice
        st = int(rs.randint(0, A // 3))
        games.append(make_game(rs, N, st, 1 if st % 2 == 0 else -1, T, 1, 2 + j))
    games.append(make_game(rs, N, 9, -1, 0, 0, 10))             # draw on a full board
    games.append(make_game(rs, N, 0, 1, A, 1, 11))
    return games


def replay(g, N):
    """Per move of an injected game: board before the move, observation planes, to_move, last_move, move_count."""
    A = N * N
    board, player, last, mc = g["start_board"].copy(), g["start_player"], g["start_last"], g["start_mc"]
    boards, obs, to_move, lasts, mcs = [], [], [], [], []
    for a in g["actions"]:
        o = np.zeros((3, A), np.float32)
        o[0][board == player] = 1.0
        o[1][board == -player] = 1.0
        if 0 <= last < A:
            o[2, last] = 1.0
        boards.append(board.reshape(N, N).copy()); obs.append(o.reshape(3, N, N))
        to_move.append(player); lasts.append(last); mcs.append(mc)
        board[a] = player
        player, last, mc = -player, int(a), mc + 1
    return dict(board=np.array(boards, np.int8), obs=np.array(obs, np.float32), to_move=np.array(to_move),
                last_move=np.array(lasts), move_count=np.array(mcs))


# ---------------------------------------------------------------------------------------------------------------------
def target_errors():
    """(max |target - exact| / (k ulp32(m)), max |target - exact| / ulp32(m), max |target - exact| / ulp32(exact)) of
    both restated targets over every move of every test game and the whole (n_steps, gamma) grid."""
    worst = [0.0, 0.0, 0.0]
    for N in (7, 6):
        for g in make_games(N, seed=N):
            T = len(g["actions"])
            rew = final_rewards(T, g["winner"])
            for n in horizons([T]):
                for gamma in GAMMAS:
                    sp = selfplay_targets(rew, g["values"], gamma, n)
                    ra = reanalysis_targets(rew, g["values"], gamma, n)
                    for t in range(T):
                        ex, m = exact_target(rew, g["values"], gamma, n, t)
                        for got, re in ((sp[t], False), (ra[t], True)):
                            err = float(abs(Fraction(float(got)) - ex))
                            u = ulp32(m)
                            worst[0] = max(worst[0], err / (rounding_count(n, T, t, re) * u))
                            worst[1] = max(worst[1], err / u)
                            worst[2] = max(worst[2], err / ulp32(ex))
    return worst


def test_reference_targets_within_their_rounding_bound_of_the_exact_target():
    """Both restated targets lie within k * ulp32(m) of the exact rational target (k and the bound derived above
    rounding_count) for every move of every test game over the whole (n_steps, gamma) grid."""
    bound, in_m, _ = target_errors()
    assert bound <= 1 + 2.0 ** -22, (bound, in_m)


def test_reference_targets_at_the_corners():
    """Hand-checked corners of the restatements: gamma = 0 keeps only r_t (and v_t when n = 0), n = 0 is float32(v_t)
    (a tie 1 + 2^-24 rounds to even 1.0, 1 + 3 * 2^-24 up, 2^-150 to +0.0, -0.0 to +0.0), and the float64 reward sum of
    self-play differs from the float32 sum of re-analysis where float32(0.997**i) rounds."""
    vals = np.array([1 + 2.0 ** -24, 1 + 3 * 2.0 ** -24, 2.0 ** -150, -0.0, 3 * 2.0 ** -150])
    r = final_rewards(5, 1)
    assert r.tolist() == [1.0, 1.0, -1.0, -1.0, 1.0]
    assert final_rewards(4, 0).tolist() == [0.0] * 4 and final_rewards(1, -1).tolist() == [1.0]
    for f in (selfplay_targets, reanalysis_targets):
        out = f(np.zeros(5, np.float32), vals, 0.997, 0)
        assert out.tolist() == [1.0, 1 + 2.0 ** -22, 0.0, 0.0, 2.0 ** -148] and not np.signbit(out[3])
        assert f(r, vals, 0.0, 3).tolist() == r.tolist()
    sp = selfplay_targets(r, vals, 0.997, 4)
    ra = reanalysis_targets(r, vals, 0.997, 4)
    assert sp[0] == np.float32(1 + 0.997 - 0.997 ** 2 - 0.997 ** 3) + np.float32(0.997 ** 4) * np.float32(vals[4])
    acc32 = np.float32(1) + np.float32(0.997) - np.float32(0.997 ** 2) - np.float32(0.997 ** 3)
    assert ra[0] == acc32 + np.float32(0.997 ** 4) * np.float32(vals[4])
    assert not np.array_equal(sp, ra)


def test_window_augmentation_matches_the_reference_loss_path():
    """augment_windows (np.rot90 / fliplr planes and policies, loss.py's action formula) == what the reference's
    calculate_loss fed its networks for all 8 symmetries (tests/golden/augment_kat.npz)."""
    g = np.load(os.path.join(GOLDEN_DIR, "augment_kat.npz"))
    N = g["obs"].shape[-1]
    valid = g["act"] != -1
    for k in range(4):
        for f in (0, 1):
            o, a, p = augment_windows(g["obs"], g["act"], g["pi"], N, k, bool(f))
            tag = f"k{k}f{f}"
            assert np.array_equal(o, g["obs_" + tag]) and np.array_equal(p.astype(np.float32), g["pi_" + tag])
            assert np.array_equal(a[valid], g["act_" + tag][valid]) and (a[~valid] == -1).all()


def test_games_are_legal_and_cover_the_lengths():
    for N in (7, 6):
        gs = make_games(N, seed=N)
        lengths = [len(g["actions"]) for g in gs]
        assert {1, 2} <= set(lengths) and {T % 4 for T in lengths} == {0, 1, 2, 3}
        assert any(g["winner"] == 0 and len(g["actions"]) == int((g["start_board"] == 0).sum()) for g in gs)
        assert any(g["start_player"] == -1 for g in gs)
        for g in gs:
            assert len(set(g["actions"].tolist())) == len(g["actions"]) and (g["start_board"][g["actions"]] == 0).all()


# ---------------------------------------------------------------------------------------------------------------------
# gather_packed_games with a truncated game in one rank's batch: the records are synthetic (header fields only), laid
# out as TrajectoryStore.pack_finished lays them out, from the same host helper (trajectory.whole_games).
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


_FINS = {0: np.array([[0, 100, 5, 1], [1, 101, 9, -1], [2, 102, 3, 0], [3, 103, 6, 1]], np.int32),   # 101 is truncated
         1: np.array([[0, 200, 4, -1], [1, 201, 7, 1], [2, 202, 2, 1]], np.int32)}                     # 201 is truncated
_MAX_MOVES = 6


def _packed(rank, N):
    from datou_gomoku_muzero_b200.trajectory import PackedGames, record_dtype, whole_games
    q, off = whole_games(_FINS[rank], _MAX_MOVES)
    rec = np.zeros(int(off[-1]), record_dtype(N))
    for i, (slot, game, T, winner) in enumerate(q):
        r = rec[off[i]:off[i + 1]]
        r["game_seq"], r["t"], r["length"], r["winner"], r["game"], r["slot"] = i, np.arange(T), T, winner, game, slot
        r["reward"] = final_rewards(T, winner)
    raw = torch.from_numpy(rec.view(np.uint8).reshape(len(rec), -1).copy())
    return PackedGames(raw, q, off, N)


def _gather_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from datou_gomoku_muzero_b200 import parallel
    N = 5
    pg = _packed(rank, N)
    mine = (np.diff(pg.offsets).tolist(), pg.table[:, 2].tolist())
    got = parallel.gather_packed_games(pg, N, dst=0)
    out = None
    if got is not None:
        out = []
        for i in range(len(got)):
            r = got.game(i)
            out.append((int(got.table[i, 4]), int(got.table[i, 1]), r["game"].tolist(), r["t"].tolist(),
                        r["length"].tolist(), r["reward"].tolist()))
    q.put((rank, mine, out))
    dist.destroy_process_group()


def test_gather_packed_games_slices_every_game_after_a_truncated_one():
    """Rank 0's and rank 1's batches each held a truncated game: every rank's table matches its offsets, and on the
    destination every gathered game is exactly its own records, t = 0..length-1, with its own reward pattern."""
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gather_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (_, mine0, out0), (_, mine1, out1) = res
    assert mine0[0] == mine0[1] == [5, 3, 6] and mine1[0] == mine1[1] == [4, 2] and out1 is None
    expect = [(r, int(g), int(T), int(w)) for r in (0, 1) for _, g, T, w in _FINS[r] if T <= _MAX_MOVES]
    assert [(rank, game) for rank, game, *_ in out0] == [(r, g) for r, g, _, _ in expect]
    for (rank, game, games, ts, lens, rews), (_, g, T, w) in zip(out0, expect):
        assert games == [g] * T and ts == list(range(T)) and lens == [T] * T and rews == final_rewards(T, w).tolist()
