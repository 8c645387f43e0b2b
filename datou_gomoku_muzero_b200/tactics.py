"""Tactical move classifier on the device (reference workers.py:49-123) and the missed-win statistics
built on it (workers.py:191-203): per host GameRecord (`missed_win_stats`), and straight from the packed move
records of device self-play (`missed_win_counts`, `SelfPlayStats`)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check
from .config import config

FIVE, OPEN_FOUR, COMBO = 1, 2, 3


def classify_boards(boards, players, board_size=None, n_in_row=None, device=None):
    """boards int8 [B,N,N] or [B,A], players +-1 [B] -> int8 [B,A] classes (device tensor)."""
    if not torch.cuda.is_available():
        raise _lib.GmzError("classify_boards needs a CUDA device (there is no CPU fallback)")
    lib = _lib.load()
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    b = torch.as_tensor(boards).to(device=dev, dtype=torch.int8)
    B = b.shape[0]
    N = board_size or (b.shape[1] if b.dim() == 3 else int(round(b.shape[1] ** 0.5)))
    b = b.reshape(B, N * N).contiguous()
    p = torch.as_tensor(players).to(device=dev, dtype=torch.int8).reshape(B).contiguous()
    out = torch.empty((B, N * N), dtype=torch.int8, device=dev)
    check(lib.gmz_tactics_classify(C.c_void_p(b.data_ptr()), C.c_void_p(p.data_ptr()), B, N,
                                   int(config.N_IN_ROW if n_in_row is None else n_in_row), C.c_void_p(out.data_ptr()),
                                   C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "gmz_tactics_classify")
    return out


def find_winning_moves_rebuilt(board, player):
    """Same return shape as the reference: {'five': [(r,c)...], 'open_four': [...], 'combo': [...]}."""
    board = np.asarray(board)
    N = board.shape[0]
    cls = classify_boards(board[None], [player], N).cpu().numpy()[0]
    out = {"five": [], "open_four": [], "combo": []}
    for a in np.flatnonzero(cls):
        out[{FIVE: "five", OPEN_FOUR: "open_four", COMBO: "combo"}[int(cls[a])]].append((int(a) // N, int(a) % N))
    return out


def missed_win_stats(game_record, board_size=None):
    """(missed_fives, missed_totals) of one finished game, as workers.py:191-203 counts them."""
    T = len(game_record.actions)
    if T == 0:
        return 0, 0
    N = board_size or np.asarray(game_record.board_states[0]).shape[0]
    boards = np.stack([np.asarray(b, np.int8) for b in game_record.board_states[:T]])
    players = np.where(np.arange(T) % 2 == 0, 1, -1).astype(np.int8)
    cls = classify_boards(boards, players, N)
    acts = torch.as_tensor(np.asarray(game_record.actions[:T], dtype=np.int64), device=cls.device)
    any_win = (cls > 0).any(dim=1)
    played = cls.gather(1, acts.reshape(-1, 1)).reshape(-1)
    missed = any_win & (played == 0)
    has_five = (cls == FIVE).any(dim=1)
    return int((missed & has_five).sum().item()), int(missed.sum().item())


# Bits of the per-record flags gmz_records_tactics writes.
WIN_AVAILABLE, FIVE_AVAILABLE, PLAYED_WIN = 1, 2, 4


def record_flags(records, board_size, n_in_row=None):
    """Missed-win flags of packed move records, classified where they lie: `records` a uint8 device tensor
    [M, stride] (a trajectory.PackedGames block or a stretch of the DeviceReplayBuffer ring) -> uint8 [M] on the same
    device (bits WIN_AVAILABLE, FIVE_AVAILABLE, PLAYED_WIN for the side in each record's to_move)."""
    lib = _lib.load()
    N = int(board_size)
    stride = int(lib.gmz_move_record_bytes(N))
    if not torch.is_tensor(records) or records.device.type != "cuda":
        raise _lib.GmzError("record_flags needs the records in a CUDA tensor (there is no CPU fallback)")
    if records.dtype != torch.uint8 or records.dim() != 2 or records.shape[1] != stride or not records.is_contiguous():
        raise ValueError(f"records must be a contiguous uint8 tensor [M, {stride}] of {N}x{N} move records")
    M = int(records.shape[0])
    out = torch.empty(M, dtype=torch.uint8, device=records.device)
    if M == 0:
        return out
    with torch.cuda.device(records.device):
        check(lib.gmz_records_tactics(C.c_void_p(records.data_ptr()), M, N,
                                      int(config.N_IN_ROW if n_in_row is None else n_in_row), C.c_void_p(out.data_ptr()),
                                      C.c_void_p(torch.cuda.current_stream(records.device).cuda_stream)),
              "gmz_records_tactics")
    return out


def _missed(flags):
    """(missed five, missed win) bool masks: a win was available and the move played was not one; a missed five
    also had a five available."""
    return (flags & 7) == (WIN_AVAILABLE | FIVE_AVAILABLE), (flags & (WIN_AVAILABLE | PLAYED_WIN)) == WIN_AVAILABLE


def missed_win_counts(packed, n_in_row=None):
    """(missed_fives, missed_totals) of every game of a trajectory.PackedGames, in `packed.table` order: int64
    [len(packed), 2] on the device, the counts `missed_win_stats` gives for `packed.game_record(i)` (one kernel over all
    records and one reduction, no loop over games).  Records held on the host (e.g. gathered over gloo) are copied
    to the current device once."""
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    off = np.asarray(packed.offsets, np.int64)
    n, M = len(packed), int(off[-1] - off[0])
    rec = packed.records if torch.is_tensor(packed.records) else torch.from_numpy(np.ascontiguousarray(packed.records))
    if rec.device.type != "cuda":
        rec = rec.to(dev)
    rec = rec.reshape(-1, int(_lib.load().gmz_move_record_bytes(packed.N)))[int(off[0]):int(off[-1])]
    out = torch.zeros((n, 2), dtype=torch.int64, device=rec.device)
    if M == 0:
        return out
    fives, missed = _missed(record_flags(rec, packed.N, n_in_row))
    # record -> game from the offsets (the header's game_seq restarts on every rank, so it repeats after a gather)
    game = torch.repeat_interleave(torch.arange(n, device=rec.device), torch.as_tensor(np.diff(off), device=rec.device),
                                   output_size=M)
    out.index_add_(0, game, torch.stack([fives, missed], dim=1).to(torch.int64))
    return out


class SelfPlayStats:
    """Running self-play statistics of device self-play -- what universal_worker reports per game in
    SelfPlayStatus (workers.py:191-203, 235): games, moves, results, missed fives and missed wins.  Pass
    `add` to play() alongside the replay sink, `sink=lambda pg: (stats.add(pg), buf.add_packed(pg))`.
    Game / move / result counts come from the host-side game table; the missed counts stay in device counters, so
    `add` never waits for the GPU.  `summary()` reads them back once."""

    def __init__(self, n_in_row=None, device=None):
        if not torch.cuda.is_available():
            raise _lib.GmzError("SelfPlayStats needs a CUDA device (there is no CPU fallback)")
        self.n_in_row = n_in_row
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self._missed = torch.zeros(2, dtype=torch.int64, device=self.device)      # missed fives, missed wins
        self.reset()

    def reset(self):
        self.games = self.moves = self.wins_black = self.wins_white = self.draws = 0
        self._missed.zero_()

    def add(self, packed):
        """Count the games of a trajectory.PackedGames whose records are on this device.  Launches one kernel and a
        few reductions on the current stream; copies nothing between host and device."""
        M = packed.n_moves
        if M and not (torch.is_tensor(packed.records) and packed.records.device == self.device):
            raise ValueError(f"SelfPlayStats.add takes records on {self.device}; use missed_win_counts for host records")
        self.games += len(packed)
        self.moves += M
        if len(packed):
            w = np.asarray(packed.table)[:, 3]                 # winner: +1, -1, 0 = draw
            self.wins_black += int((w == 1).sum())
            self.wins_white += int((w == -1).sum())
            self.draws += int((w == 0).sum())
        if M == 0:
            return
        fives, missed = _missed(record_flags(packed.records[:M], packed.N, self.n_in_row))
        self._missed += torch.stack([fives.sum(), missed.sum()])

    def summary(self):
        """dict of the counts plus avg_game_length and per-game rates (one device -> host copy)."""
        fives, missed = (int(x) for x in self._missed.tolist())
        g = self.games
        return {"games": g, "moves": self.moves, "wins_black": self.wins_black, "wins_white": self.wins_white,
                "draws": self.draws, "missed_fives": fives, "missed_all_wins": missed,
                "avg_game_length": self.moves / g if g else 0.0,
                "missed_fives_per_game": fives / g if g else 0.0, "missed_all_wins_per_game": missed / g if g else 0.0}
