"""Every board size and row length the C ABI accepts, on the host: the record layout, the config bounds, the torch E0
against e0_py, the host win rule against the oracle, the Gumbel halving schedule against the oracle's search, and a
plain-Python restatement of the reference's tactics classifier (workers.py:49-123) pinned to the reference KATs.
tests/test_shapes_gpu.py uses that restatement as the reference for the kernels at shapes the KATs do not cover."""
import os

import numpy as np

from _golden_util import GOLDEN_DIR

DIRS = ((0, 1), (1, 0), (1, 1), (1, -1))


def tactic_patterns(board, player):
    """Per cell, for `player` to move: the number of directions whose 9-cell line centred on the cell (the stone placed,
    off-board counted as an opponent stone) holds an open four `0PPPP0`, a blocked four `XPPP0` / `0PPPX` (three stones:
    the reference's pattern) and an open three `0PPP0`.  int [3, A]; zero on occupied cells."""
    board = np.asarray(board, np.int8)
    N = board.shape[0]
    out = np.zeros((3, N * N), np.int64)
    for r in range(N):
        for c in range(N):
            if board[r, c] != 0:
                continue
            for dr, dc in DIRS:
                line = ""
                for i in range(-4, 5):
                    rr, cc = r + i * dr, c + i * dc
                    v = (player if i == 0 else board[rr, cc]) if 0 <= rr < N and 0 <= cc < N else -player
                    line += "P" if v == player else ("0" if v == 0 else "X")
                out[:, r * N + c] += ("0PPPP0" in line, "XPPP0" in line or "0PPPX" in line, "0PPP0" in line)
    return out


def classify_ref(board, player, n_in_row, patterns=None):
    """find_winning_moves_rebuilt (workers.py:49-123) restated: int8 [A] classes of every cell for `player` to move,
    1 = five (oracle.check_win after placing the stone), 2 = open four, 3 = combo (>= 2 blocked fours, a blocked four and
    an open three, or >= 2 open threes), 0 = none or occupied.  `patterns`: tactic_patterns(board, player), which does
    not depend on n_in_row."""
    from oracle import oracle
    board = np.asarray(board, np.int8)
    N = board.shape[0]
    of, bf, ot = tactic_patterns(board, player) if patterns is None else patterns
    out = np.zeros(N * N, np.int8)
    for a in np.flatnonzero(board.reshape(-1) == 0):
        b2 = board.copy()
        b2[a // N, a % N] = player
        if oracle.check_win(b2, n_in_row, a // N, a % N):
            out[a] = 1
        elif of[a]:
            out[a] = 2
        elif bf[a] >= 2 or (bf[a] >= 1 and ot[a] >= 1) or ot[a] >= 2:
            out[a] = 3
    return out


def test_tactics_restatement_matches_reference_kat():
    z = np.load(os.path.join(GOLDEN_DIR, "tactics_kat.npz"))
    n = int(z["n"])
    assert n == 240
    for i in range(n):
        N = int(z["N"][i])
        A = N * N
        got = classify_ref(z["boards"][i][:A].reshape(N, N), int(z["player"][i]), 5)
        assert np.array_equal(got, z["cls"][i][:A]), i


def test_record_layout_every_board_size():
    from datou_gomoku_muzero_b200 import _lib
    from datou_gomoku_muzero_b200.trajectory import record_dtype
    lib = _lib.load()
    for N in range(1, 20):
        A = N * N
        dt = record_dtype(N)
        assert dt.itemsize == lib.gmz_move_record_bytes(N) and dt.itemsize % 16 == 0, N
        assert dt.itemsize >= 64 + 21 * A, N
        assert dt.fields["policy"][1] == 64 and dt.fields["search_value"][1] == 40, N
        assert dt.fields["obs"][1] == 64 + 8 * A and dt.fields["board"][1] == 64 + 20 * A, N
    assert lib.gmz_move_record_bytes(0) == 0 and lib.gmz_move_record_bytes(20) == 0


def test_config_bounds():
    """board_size 1..19, n_in_row 1..14, num_top_actions 1..32 are accepted (K = 32 also on a 1x1 board); one step
    outside each range is refused with a message."""
    import ctypes as C
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()

    def cfg(N=9, nir=5, K=16):
        return _lib.GmzConfig(N, nir, 16, K, 0, 2, 0, 0, 30.0, 1.0, 1e-3, 0.997)
    for N, nir, K in ((1, 5, 16), (19, 5, 16), (9, 1, 16), (9, 14, 16), (9, 5, 1), (9, 5, 32), (1, 1, 32), (1, 14, 1),
                      (19, 14, 32)):
        assert lib.gmz_workspace_bytes(C.byref(cfg(N, nir, K))) > 0, (N, nir, K)
    for kw, what in ((dict(N=0), b"board_size"), (dict(N=20), b"board_size"), (dict(nir=0), b"n_in_row"),
                     (dict(nir=15), b"n_in_row"), (dict(K=0), b"num_top_actions"), (dict(K=33), b"num_top_actions")):
        assert lib.gmz_workspace_bytes(C.byref(cfg(**kw))) == 0, kw
        assert what in lib.gmz_last_error(), kw


def test_torch_e0_matches_python_e0_every_board_size():
    import torch
    import e0_py
    from datou_gomoku_muzero_b200.muzero import TorchE0
    rs = np.random.RandomState(19)
    for N in range(1, 20):
        A = N * N
        B = 6
        obs = np.zeros((B, 3, N, N), np.float32)
        for b in range(B):
            cells = rs.randint(-1, 2, size=(N, N))
            if b == 0:
                cells[:] = 1                   # every bit of every word set, the sign bit included where A > 63
            obs[b, 0] = cells == 1; obs[b, 1] = cells == -1
            if b % 3:
                a = rs.randint(A); obs[b, 2, a // N, a % N] = 1
        for div in (16, 0):
            seed = int(rs.randint(1 << 30))
            e0 = TorchE0(N, seed=seed, logit_div=div, device="cpu")
            lg, v, h = e0.initial(torch.from_numpy(obs))
            acts = torch.from_numpy(rs.randint(0, A, size=B))
            lg2, v2, r2, h2 = e0.recurrent(h, acts)
            for b in range(B):
                hp = e0_py.hash_obs(obs[b], seed)
                assert (int(h[b]) & ((1 << 64) - 1)) == hp, (N, div, b)
                l_ref, v_ref = e0_py.heads(hp, A, div)
                assert np.array_equal(lg[b].numpy(), l_ref) and float(v[b]) == v_ref, (N, div, b)
                hc = e0_py.child_hidden(hp, int(acts[b]))
                assert (int(h2[b]) & ((1 << 64) - 1)) == hc, (N, div, b)
                l2, vr2 = e0_py.heads(hc, A, div)
                assert np.array_equal(lg2[b].numpy(), l2) and float(v2[b]) == vr2, (N, div, b)
                assert float(r2[b]) == e0_py.reward_of(hc, div), (N, div, b)


def crafted_lines(N, n_in_row, rs):
    """(board int8 [N,N], last move (r, c)) pairs: a line of `length` stones of one colour through the last move in each
    direction, for lengths around n_in_row (exact, one short, overlines), with and without a gap next to the last move,
    starting or ending on the edges and in the corners (plus one random placement); the rest of the board is random
    opponent stones."""
    out = []
    for dr, dc in DIRS:
        for length in sorted({n_in_row - 1, n_in_row, n_in_row + 1, n_in_row + 2, 2 * n_in_row + 3, N}):
            if length < 1:
                continue
            # every start cell keeping the whole line on the board; keep the corner / edge ones and a few inside
            starts = [(r0, c0) for r0 in range(N) for c0 in range(N)
                      if 0 <= r0 + (length - 1) * dr < N and 0 <= c0 + (length - 1) * dc < N]
            if not starts:
                continue
            edge = [s for s in starts if s[0] in (0, N - 1) or s[1] in (0, N - 1)
                    or s[0] + (length - 1) * dr in (0, N - 1) or s[1] + (length - 1) * dc in (0, N - 1)]
            pick = edge[:: max(1, len(edge) // 6)] + [edge[-1], starts[int(rs.randint(len(starts)))]]
            for r0, c0 in pick:
                colour = 1 if rs.randint(2) else -1
                b = np.where(rs.random_sample((N, N)) < 0.3, -colour, 0).astype(np.int8)
                cells = [(r0 + i * dr, c0 + i * dc) for i in range(length)]
                for rr, cc in cells:
                    b[rr, cc] = colour
                for rr, cc in ((r0 - dr, c0 - dc), (r0 + length * dr, c0 + length * dc)):
                    if 0 <= rr < N and 0 <= cc < N:     # the cells just outside both ends: an opponent stone or empty
                        b[rr, cc] = -colour if rs.randint(2) else 0
                last = cells[int(rs.randint(length))]
                out.append((b.copy(), last))
                if length >= 3:                 # a gap one cell away from the last move breaks the run there
                    k = cells.index(last)
                    gap = cells[k + 1] if k + 1 < length else cells[k - 1]
                    g2 = b.copy(); g2[gap] = 0
                    out.append((g2, last))
    return out


def test_host_win_rule_matches_oracle():
    """GomokuGame.check_win / get_game_ended (the reference's game.py:20-63) against oracle.game_ended on random positions
    and on crafted lines in every direction, for row lengths shorter and longer than the board."""
    from datou_gomoku_muzero_b200.game import GomokuGame
    from oracle import oracle
    rs = np.random.RandomState(7)
    n, wins = 0, 0
    for N in (3, 5, 8, 12, 19):
        for nir in (1, 2, 3, 6, 7, 14):
            cases = []
            for _ in range(40):
                b = rs.randint(-1, 2, size=(N, N)).astype(np.int8)
                cases.append((b, (int(rs.randint(N)), int(rs.randint(N)))))
            cases += crafted_lines(N, nir, rs)
            for b, (r, c) in cases:
                if b[r, c] == 0:
                    b = b.copy(); b[r, c] = 1
                mc = int((b != 0).sum()) if rs.randint(4) else N * N
                g = GomokuGame(N, nir)
                g.board, g.last_move, g.move_count = b.copy(), (r, c), mc
                got = g.get_game_ended()
                want = oracle.game_ended(b, nir, r * N + c, mc)
                assert (None if got is None else int(got)) == want, (N, nir, r, c)
                n += 1
                wins += want is not None and want != 0
    assert n >= 1200 and wins > n // 4


def test_evals_per_search_matches_oracle_on_small_boards():
    """The number of recurrent evaluations of a MuZero-mode search (the halving schedule driven with the number of
    survivors, mcts.py:158-181) against the oracle's count, where fewer empty cells than K is the normal case."""
    from datou_gomoku_muzero_b200.muzero import evals_per_search
    from oracle import oracle
    rs = np.random.RandomState(3)
    n = short = 0
    for N in (1, 2, 3, 4, 5, 7, 8):
        A = N * N
        for S in (1, 2, 7, 16, 64):
            for K in (1, 2, 4, 16, 32):
                for k in sorted({0, A // 2, max(0, A - 3), A - 1}):
                    b = np.zeros(A, np.int8); p, last = 1, -1
                    for a in rs.permutation(A)[:k]:
                        b[a] = p; last = a; p = -p
                    cfg = oracle.make_config(board_size=N, num_simulations=S, num_top_actions=K, mode=1, eval_seed=4)
                    r = oracle.search(cfg, b, p, last, k, rs.gumbel(0, 1, A))
                    n_valid = A - k
                    assert evals_per_search(S, K, min(K, n_valid)) == r["n_evals"], (N, S, K, k)
                    n += 1
                    short += n_valid < K
    assert n > 500 and short > n // 3
