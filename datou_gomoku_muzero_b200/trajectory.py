"""Trajectories of the persistent self-play kernel -> the reference's data-queue items.

`TrajectoryStore` owns the device buffers the kernel records into (include/gmz.h `gmz_traj`) and
harvests finished games; `build_game_record` / `cut_training_slices` turn one finished game into
the `(GameRecord, [TrainingSlice])` pair the reference's self-play loop emits (workers.py:183-230),
with the same dtypes and the same arithmetic (final-reward pattern, n-step value targets, padding).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from ._lib import GmzTraj, check
from .config import config
from .data_structures import GameRecord, TrainingSlice


def record_dtype(board_size):
    """numpy view of one packed move record (include/gmz.h gmz_move_record + payload)."""
    N = int(board_size)
    A = N * N
    stride = (64 + 21 * A + 15) // 16 * 16
    names = ["game_seq", "t", "length", "winner", "action", "to_move", "last_move", "move_count", "reward", "value_target",
             "search_value", "game", "slot", "policy", "obs", "board"]
    formats = ["<i4"] * 8 + ["<f4", "<f4", "<f8", "<i4", "<i4", ("<f8", (A,)), ("<f4", (3, N, N)), ("i1", (N, N))]
    offsets = [0, 4, 8, 12, 16, 20, 24, 28, 32, 36, 40, 48, 52, 64, 64 + 8 * A, 64 + 20 * A]
    return np.dtype({"names": names, "formats": formats, "offsets": offsets, "itemsize": stride})


class PackedGames:
    """Finished games as packed move records (csrc/gmz_records.cu): `records` uint8 [M, stride] (device or host
    tensor), `table` int32 [n, 4] = (slot, game, length, winner) per game, `offsets` int64 [n + 1] = first record of
    each game.  What the reference puts on data_queue per game -- (GameRecord, [TrainingSlice], version),
    workers.py:230 -- is a set of numpy views of these bytes."""

    def __init__(self, records, table, offsets, board_size):
        self.records, self.table, self.offsets, self.N = records, np.asarray(table), np.asarray(offsets, np.int64), int(board_size)
        self._host = None

    def __len__(self):
        return len(self.table)

    @property
    def n_moves(self):
        return int(self.offsets[-1])

    def host(self):
        """Structured numpy array [M] over the record bytes (one D2H copy, cached)."""
        if self._host is None:
            raw = self.records.cpu().numpy() if torch.is_tensor(self.records) else np.asarray(self.records)
            self._host = np.ascontiguousarray(raw).view(record_dtype(self.N)).reshape(-1)
        return self._host

    def game(self, i):
        return self.host()[self.offsets[i]:self.offsets[i + 1]]

    def game_record(self, i):
        """GameRecord of game i (data_structures.py:9-16): lists of per-move array views / Python scalars."""
        r = self.game(i)
        return GameRecord(list(r["obs"]), r["action"].tolist(), r["reward"].tolist(), list(r["policy"]),
                          r["value_target"].tolist(), list(r["board"]))

    def training_slices(self, i):
        """[TrainingSlice] of game i (workers.py:208-222): windows of U+1 moves over the zero / -1 padded arrays."""
        r, U = self.game(i), int(config.NUM_UNROLL_STEPS)
        T = len(r)
        if T == 0:
            return []
        win = np.lib.stride_tricks.sliding_window_view
        obs = np.concatenate([r["obs"], np.zeros((U + 1,) + r["obs"].shape[1:], np.float32)])
        pol = np.concatenate([r["policy"], np.zeros((U + 1, r["policy"].shape[1]), np.float64)])
        act = np.concatenate([r["action"].astype(np.int32), np.full(U, -1, np.int32)])
        rew = np.concatenate([r["reward"].astype(np.float32), np.zeros(U, np.float32)])
        val = np.concatenate([r["value_target"].astype(np.float32), np.zeros(U + 1, np.float32)])
        ow, pw = win(obs, U + 1, axis=0), win(pol, U + 1, axis=0)             # window axis comes last
        ow, pw = np.moveaxis(ow, -1, 1), np.moveaxis(pw, -1, 1)
        aw, rw, vw = (win(act, U) if U else np.zeros((T + 1, 0), np.int32)), (win(rew, U) if U else np.zeros((T + 1, 0), np.float32)), win(val, U + 1)
        return [TrainingSlice(ow[t], aw[t], rw[t], pw[t], vw[t]) for t in range(T)]

    def data_queue_items(self, model_version=0):
        """The tuples universal_worker puts on data_queue (workers.py:230), one per game."""
        return [(self.game_record(i), self.training_slices(i), model_version) for i in range(len(self))]


class TrajectoryStore:
    def __init__(self, engine, extra_slots=None, max_moves=None):
        e = self.e = engine
        G, A = e.G, e.A
        self.n_slots = G + (max(64, G // 4) if extra_slots is None else int(extra_slots))
        self.max_moves = A if max_moves is None else int(max_moves)
        if self.max_moves < 1:
            raise ValueError("max_moves must be >= 1")
        dev = e.device
        n, T = self.n_slots, self.max_moves
        self.policy = torch.zeros((n, T, A), dtype=torch.float64, device=dev)
        self.value = torch.zeros((n, T), dtype=torch.float64, device=dev)
        self.action = torch.full((n, T), -1, dtype=torch.int32, device=dev)
        self.start_board = torch.zeros((n, 2, 8), dtype=torch.int64, device=dev)
        self.start_info = torch.zeros((n, 4), dtype=torch.int32, device=dev)
        self.free_slots = torch.zeros(n, dtype=torch.int32, device=dev)
        self.free_top = torch.zeros(1, dtype=torch.int32, device=dev)
        self.fin_queue = torch.zeros((n, 4), dtype=torch.int32, device=dev)
        self.fin_count = torch.zeros(1, dtype=torch.int32, device=dev)
        p = lambda t: t.data_ptr()
        self.c = GmzTraj(n, T, n, 0, p(self.policy), p(self.value), p(self.action), p(self.start_board),
                         p(self.start_info), p(self.free_slots), p(self.free_top), p(self.fin_queue), p(self.fin_count))
        check(e.lib.gmz_traj_init(e.handle, C.byref(self.c), e._stream()), "gmz_traj_init")
        e.launches += 1

    def harvest(self, copy_policies=True, unpark=True):
        """Finished games since the last harvest -> list of dicts (host arrays).  Their slots go back on the free
        stack and (with `unpark`) parked games restart -- pass unpark=False after play(restart=False) to leave
        finished games finished.  A game that recorded more moves than the store's `max_moves` (only possible with a
        user-supplied max_moves below the remaining plies) comes back with `length` clamped to what was recorded and
        `truncated` = True."""
        e = self.e
        n = int(self.fin_count.item())
        if n == 0:
            return []
        q = self.fin_queue[:n].cpu().numpy()
        slots = torch.as_tensor(q[:, 0].astype(np.int64), device=e.device)
        full_len = q[:, 2].copy()
        q[:, 2] = np.minimum(q[:, 2], self.max_moves)
        Tmax = int(q[:, 2].max())
        act = self.action[slots, :Tmax].cpu().numpy()
        val = self.value[slots, :Tmax].cpu().numpy()
        pol = self.policy[slots, :Tmax].cpu().numpy() if copy_policies else None
        sb = self.start_board[slots].cpu().numpy().view(np.uint64)
        si = self.start_info[slots].cpu().numpy()
        out = []
        for i in range(n):
            T = int(q[i, 2])
            bits = np.unpackbits(sb[i].view(np.uint8).reshape(2, 64), axis=1, bitorder="little")[:, :e.A]
            board = bits[0].astype(np.int8) - bits[1].astype(np.int8)
            out.append(dict(slot=int(q[i, 0]), game=int(q[i, 1]), length=T, winner=int(q[i, 3]), actions=act[i, :T].copy(),
                            values=val[i, :T].copy(), policies=None if pol is None else pol[i, :T].copy(),
                            start_board=board.reshape(e.N, e.N), start_player=int(si[i, 0]),
                            start_move_count=int(si[i, 1]), start_last_move=int(si[i, 2]),
                            truncated=bool(full_len[i] > self.max_moves)))
        self.fin_count.zero_()
        self.release(slots, unpark=unpark)
        return out

    def pack_finished(self, recycle=True):
        """Finished games since the last harvest / pack -> PackedGames on the DEVICE (None if there are none): one
        kernel expands every finished slot into fixed-stride move records (observations, policies, boards, final
        rewards, n-step value targets); nothing is computed per move on the host.  With `recycle` the slots go back
        on the free stack and parked games restart."""
        e = self.e
        n = int(self.fin_count.item())
        if n == 0:
            return None
        q = self.fin_queue[:n].cpu().numpy()
        lens = np.minimum(q[:, 2], self.max_moves).astype(np.int64)
        off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        stride = int(e.lib.gmz_move_record_bytes(e.N))
        # allocated in power-of-two buckets (>= 8192 records): chunks of similar size then reuse the caching allocator's
        # blocks (a fresh cudaMalloc of a few hundred MB costs ~100 ms, 300x the pack kernel itself)
        M = int(off[-1])
        rec = torch.empty((max(8192, 1 << (M - 1).bit_length()), stride), dtype=torch.uint8, device=e.device)[:M]
        off_d = torch.as_tensor(off[:-1].copy(), device=e.device)
        dpow = torch.tensor([config.DISCOUNT ** i for i in range(config.N_STEPS + 1)], dtype=torch.float64, device=e.device)
        check(e.lib.gmz_traj_pack(C.byref(self.c), e.N, self.fin_queue.data_ptr(), n, off_d.data_ptr(), dpow.data_ptr(),
                                  int(config.N_STEPS), rec.data_ptr(), e._stream()), "gmz_traj_pack")
        e.launches += 1
        self.fin_count.zero_()
        if recycle:
            self.release(torch.as_tensor(q[:, 0].astype(np.int32), device=e.device))
        return PackedGames(rec, q, off, e.N)

    def free_slots_left(self):
        return int(self.free_top.item())

    def release(self, slots, unpark=True):
        """Push slots back on the free stack and (unless unpark=False) restart every parked game that can get one --
        including games parked by play(restart=False)."""
        e = self.e
        slots = torch.as_tensor(slots, device=e.device).to(torch.int32).reshape(-1)
        n = int(slots.numel())
        if n == 0:
            return
        top = int(self.free_top.item())
        self.free_slots[top:top + n] = slots
        self.free_top.fill_(top + n)
        if unpark:
            check(e.lib.gmz_selfplay_unpark(e.handle, C.byref(self.c), e._stream()), "gmz_selfplay_unpark")
            e.launches += 1


def final_rewards(num_moves, winner):
    """workers.py:183-187: last mover +1, then -1, then r[i] = -r[i+2] backwards; zeros on a draw."""
    r = np.zeros(num_moves, dtype=np.float32)
    if winner != 0 and num_moves > 0:
        r[-1] = 1.0
        if num_moves > 1:
            r[-2] = -1.0
        for i in range(num_moves - 3, -1, -1):
            r[i] = -r[i + 2]
    return r


def compute_n_step_returns(rewards, values, discount, n_steps):
    """workers.py:144-152, same operand types: `rewards` a list of Python floats, values -> float32
    array (so the bootstrap product is float32), Python `sum` for the reward part."""
    T = len(rewards)
    returns = np.zeros(T, dtype=np.float32)
    v32 = np.array(values, dtype=np.float32)
    powers = [discount ** i for i in range(n_steps)]
    gamma_n = discount ** n_steps
    for t in range(T - 1, -1, -1):
        b = t + n_steps
        boot = v32[b] * gamma_n if b < len(v32) else 0.0
        acc = sum(powers[i] * rewards[t + i] for i in range(n_steps) if t + i < T)
        returns[t] = acc + boot
    return returns.tolist()


def build_game_record(rec, board_size=None):
    """One harvested game (from an empty start) -> GameRecord (workers.py:172-206)."""
    N = board_size or rec["start_board"].shape[0]
    T = rec["length"]
    board = rec["start_board"].astype(np.int8).copy()
    player, last = rec["start_player"], rec["start_last_move"]
    observations, board_states = [], []
    for t in range(T):
        obs = np.zeros((3, N, N), dtype=np.float32)
        obs[0][board == player] = 1.0
        obs[1][board == -player] = 1.0
        if last >= 0:
            obs[2, last // N, last % N] = 1.0
        observations.append(obs)
        board_states.append(board.copy())
        a = int(rec["actions"][t])
        board[a // N, a % N] = player
        player, last = -player, a
    rewards = final_rewards(T, rec["winner"]).tolist()
    values = [np.float64(v) for v in rec["values"]]
    targets = compute_n_step_returns(rewards, values, config.DISCOUNT, config.N_STEPS)
    policies = [rec["policies"][t] for t in range(T)]
    return GameRecord(observations, [int(a) for a in rec["actions"]], rewards, policies, targets, board_states)


def cut_training_slices(game_record):
    """workers.py:208-222: one slice per move, U unroll steps, padded with zeros / -1."""
    U = config.NUM_UNROLL_STEPS
    obs, acts, rews, pols, vals = (game_record.observations, game_record.actions, game_record.rewards,
                                   game_record.policies, game_record.values)
    T = len(acts)
    if T == 0:
        return []
    obs_p = np.concatenate([np.stack(obs), np.zeros((U + 1,) + obs[0].shape, obs[0].dtype)])
    act_p = np.array(list(acts) + [-1] * U, dtype=np.int32)
    rew_p = np.array(list(rews) + [0.0] * U, dtype=np.float32)
    pol_p = np.concatenate([np.stack(pols), np.zeros((U + 1,) + pols[0].shape, pols[0].dtype)])
    val_p = np.array(list(vals) + [0.0] * (U + 1), dtype=np.float32)
    return [TrainingSlice(obs_p[i:i + U + 1].copy(), act_p[i:i + U].copy(), rew_p[i:i + U].copy(),
                          pol_p[i:i + U + 1].copy(), val_p[i:i + U + 1].copy()) for i in range(T)]
