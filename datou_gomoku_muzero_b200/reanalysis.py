"""Surge re-analysis (reference workers.py:243-305): re-run the search on every stored position of
finished games with the latest model and rebuild the policy / value targets.

The reference walks one game at a time, one position at a time (`mcts_engine.search(temp_game)` per
stored board, workers.py:254-266).  Here all positions of all supplied games go through the engine in
batches of G -- the positions are independent roots (`board_states[i]`, player = +1 if i even else -1,
last move = actions[i-1], move_count = i).
"""
from __future__ import annotations

import numpy as np

from .config import config
from .trajectory import compute_n_step_returns


def positions_of(game_record, board_size):
    """The roots the reference rebuilds from one GameRecord (workers.py:258-263)."""
    T = len(game_record.actions)
    N = board_size
    boards = np.stack([np.asarray(b, dtype=np.int8).reshape(N * N) for b in game_record.board_states[:T]])
    players = np.where(np.arange(T) % 2 == 0, 1, -1).astype(np.int8)
    last = np.array([-1] + [int(a) for a in game_record.actions[:T - 1]], dtype=np.int32)
    return boards, players, last, np.arange(T, dtype=np.int32)


def reanalyse(game_records, batch_search, board_size=None, gumbel_fn=None):
    """game_records: list of GameRecord.  batch_search: an `AlphaZeroMCTS.for_engine(...)`-style object
    (search_batch over exactly G roots; `MuZeroMCTS.for_engine(engine, (initial_fn, recurrent_fn))` re-analyses with the
    learned dynamics, any evaluator of mcts.resolve_searchers works).  Returns, per game, (new_policies [T,A] float64,
    new_value_targets list[float], search_values float64 [T]) -- the first two are what
    `finish_reanalysis_for_game` is handed (workers.py:292-294).
    gumbel_fn(n, A) supplies the noise rows (default: np.random.gumbel like each reference search)."""
    N = board_size or config.BOARD_SIZE
    A = N * N
    eng = batch_search._batch["engine"]
    G = eng.G
    pos = [positions_of(gr, N) for gr in game_records]
    boards = np.concatenate([p[0] for p in pos]); players = np.concatenate([p[1] for p in pos])
    last = np.concatenate([p[2] for p in pos]); mc = np.concatenate([p[3] for p in pos])
    n = len(boards)
    pol = np.zeros((n, A), np.float64); val = np.zeros(n, np.float64)
    for s in range(0, n, G):
        e = min(n, s + G)
        k = e - s
        b = np.zeros((G, A), np.int8); b[:k] = boards[s:e]
        b[k:, :] = 1                                      # padding roots: full boards -> inactive games
        pl = np.ones(G, np.int8); pl[:k] = players[s:e]
        lm = np.full(G, -1, np.int32); lm[:k] = last[s:e]
        m = np.zeros(G, np.int32); m[:k] = mc[s:e]
        g = gumbel_fn(G, A) if gumbel_fn else np.random.gumbel(0, 1, (G, A))
        p, v, _ = batch_search.search_batch(b, pl, lm, m, g)
        pol[s:e], val[s:e] = p[:k], v[:k]
    out, off = [], 0
    for gr in game_records:
        T = len(gr.actions)
        rewards = np.array(gr.rewards, dtype=np.float32)          # workers.py:291: float32 here, unlike self-play
        targets = compute_n_step_returns(rewards, [np.float64(x) for x in val[off:off + T]], config.DISCOUNT, config.N_STEPS)
        out.append((pol[off:off + T].copy(), targets, val[off:off + T].copy()))
        off += T
    return out


def writeback_windows(new_policies, new_value_targets, unroll_steps=None):
    """The write-back format of a re-analysed game (db_manager.py:189-203, `finish_reanalysis_for_game`): for every move
    t the window of U + 1 policies / value targets starting at t, zero-padded past the end of the game -- what replaces
    `policy_history` / `value_history` of the stored TrainingSlice of move t.  Returns (policy windows float64
    [T, U+1, A], value windows float32 [T, U+1])."""
    U = int(config.NUM_UNROLL_STEPS if unroll_steps is None else unroll_steps)
    pol = np.asarray(new_policies, dtype=np.float64)
    T, A = pol.shape
    val = np.asarray(new_value_targets, dtype=np.float64)
    win = np.lib.stride_tricks.sliding_window_view
    pw = win(np.concatenate([pol, np.zeros((U, A), np.float64)]), U + 1, axis=0)           # [T, A, U+1]
    vw = win(np.concatenate([val, np.zeros(U, np.float64)]), U + 1)                         # [T, U+1]
    return np.ascontiguousarray(np.moveaxis(pw, -1, 1)), vw.astype(np.float32)


def apply_writeback(slices, new_policies, new_value_targets, unroll_steps=None):
    """`original_slice._replace(policy_history=..., value_history=...)` for every stored slice of the game
    (db_manager.py:209-214); `slices` in move order."""
    pw, vw = writeback_windows(new_policies, new_value_targets, unroll_steps)
    if len(slices) != len(pw):
        raise ValueError("one stored slice per move expected")
    return [s._replace(policy_history=pw[t], value_history=vw[t]) for t, s in enumerate(slices)]


def reanalyse_positions(engines, boards, players, last_moves, move_counts, evaluator="e0", eval_seed=0, logit_div=16,
                        noise_seed=0, gumbel=None, want_policies=True, cls=None):
    """Re-search `n` stored positions (host arrays: boards int8 [n, A], players [n], last_moves [n], move_counts [n])
    with the latest evaluator -- the inner loop of the reference's re-analysis mode (workers.py:254-266) for any number of
    positions.  They stream through `len(engines)` engines in flight (PipelinedBatchSearch: pinned staging, H2D, search,
    D2H), G positions per batch; the last batch is padded with inactive (full-board) roots.  evaluator: anything
    mcts.resolve_searchers takes -- "e0", a callable, a GomokuNetEZ module, a pair (initial_fn, recurrent_fn) for
    MuZero-mode engines (pass cls=MuZeroMCTS), or one already-built NetworkSearch / MuZeroDeviceSearch per engine; MuZero
    searchers get per-game node budgets from the host boards, as DeviceReplayBuffer.reanalyse does.  Noise: `gumbel` float64
    [n, A] from the host, or drawn on the device from `noise_seed` (position i uses counters i*A .. i*A + A - 1).
    Returns (policies float64 [n, A], values float64 [n]); want_policies=False returns (None, values),
    "checksum" returns (sum of all policy entries, values) without materialising the [n, A] array."""
    from .mcts import PipelinedBatchSearch
    eng0 = engines[0]
    G, A = eng0.G, eng0.A
    boards = np.asarray(boards, dtype=np.int8).reshape(-1, A)
    n = boards.shape[0]
    pipe = PipelinedBatchSearch(list(engines), cls=cls, evaluator=evaluator, eval_seed=eval_seed, logit_div=logit_div)
    keep = want_policies is True
    pol = np.zeros((n, A), np.float64) if keep else None
    checksum = 0.0
    val = np.zeros(n, np.float64)
    pad_b = np.ones((G, A), np.int8); pad_p = np.ones(G, np.int8); pad_l = np.full(G, -1, np.int32); pad_m = np.zeros(G, np.int32)
    inflight = []

    def collect():
        nonlocal checksum
        ticket, s0, k = inflight.pop(0)
        p, v, _ = pipe.result(ticket)
        if keep:
            pol[s0:s0 + k] = p[:k]
        elif want_policies == "checksum":
            checksum += float(p[:k].sum())
        val[s0:s0 + k] = v[:k]
    for s0 in range(0, n, G):
        k = min(G, n - s0)
        if k == G:
            b, pl, lm, m = boards[s0:s0 + G], players[s0:s0 + G], last_moves[s0:s0 + G], move_counts[s0:s0 + G]
        else:
            b, pl, lm, m = pad_b.copy(), pad_p.copy(), pad_l.copy(), pad_m.copy()
            b[:k], pl[:k], lm[:k], m[:k] = boards[s0:s0 + k], players[s0:s0 + k], last_moves[s0:s0 + k], move_counts[s0:s0 + k]
        if gumbel is not None:
            g = np.zeros((G, A), np.float64); g[:k] = np.asarray(gumbel[s0:s0 + k], np.float64)
            t = pipe.submit(b, pl, lm, m, g)
        else:
            t = pipe.submit(b, pl, lm, m, device_noise=(noise_seed, s0 * A))
        inflight.append((t, s0, k))
        if len(inflight) >= len(engines):
            collect()
    while inflight:
        collect()
    return (pol if keep else (checksum if want_policies == "checksum" else None)), val
