"""Tactical move classifier on the device (reference workers.py:49-123) and the missed-win statistics
built on it (workers.py:191-203): per host GameRecord (`missed_win_stats`), and straight from the packed move
records of device self-play (`missed_win_counts`, `SelfPlayStats`).  Forced wins beyond the next stone: the VCF
solver (`find_vcf`) and the missed-VCF statistics built on it (`vcf_record_flags`, `missed_vcf_counts`,
`SelfPlayStats(vcf_attacks=k)`), and the VCT solver through threats of three (`find_vct`, `vct_record_flags`,
`missed_vct_counts`) for offline use and samples."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check
from .config import config
from .trajectory import RECORD_HEADER

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
    rec, game = _game_records(packed)
    out = torch.zeros((len(packed), 2), dtype=torch.int64, device=rec.device)
    if rec.shape[0] == 0:
        return out
    fives, missed = _missed(record_flags(rec, packed.N, n_in_row))
    out.index_add_(0, game, torch.stack([fives, missed], dim=1).to(torch.int64))
    return out


def _game_records(packed):
    """(the records of every game of a trajectory.PackedGames on the current device -- host records are copied there
    once --, the game index of each record int64 [M])."""
    dev = torch.device(f"cuda:{torch.cuda.current_device()}")
    off = np.asarray(packed.offsets, np.int64)
    n, M = len(packed), int(off[-1] - off[0])
    rec = packed.records if torch.is_tensor(packed.records) else torch.from_numpy(np.ascontiguousarray(packed.records))
    if rec.device.type != "cuda":
        rec = rec.to(dev)
    rec = rec.reshape(-1, int(_lib.load().gmz_move_record_bytes(packed.N)))[int(off[0]):int(off[-1])]
    # record -> game from the offsets (the header's game_seq restarts on every rank, so it repeats after a gather)
    game = torch.repeat_interleave(torch.arange(n, device=rec.device), torch.as_tensor(np.diff(off), device=rec.device),
                                   output_size=M)
    return rec, game


# Forced wins: the VCF solver (include/gmz.h gmz_vcf_solve states the definition, the visiting order and the budget).
VCF_ATTACKS, VCF_BUDGET = 8, 20_000
# Bits of the per-record flags gmz_records_vcf writes.
VCF_AVAILABLE, PLAYED_VCF, VCF_UNKNOWN = 1, 2, 4


def _solve(entry, name, boards, players, max_attacks, node_budget, n_in_row, board_size, device):
    """gmz_vcf_solve / gmz_vct_solve on a batch -> device tensors (length int32 [B], first bool [B,A], nodes int32 [B])."""
    if not torch.cuda.is_available():
        raise _lib.GmzError(f"{name} needs a CUDA device (there is no CPU fallback)")
    lib = _lib.load()
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    b = torch.as_tensor(boards).to(device=dev, dtype=torch.int8)
    B = b.shape[0]
    N = board_size or (b.shape[1] if b.dim() == 3 else int(round(b.shape[1] ** 0.5)))
    A = N * N
    b = b.reshape(B, A).contiguous()
    p = torch.as_tensor(players).to(device=dev, dtype=torch.int8).reshape(B).contiguous()
    length = torch.empty(B, dtype=torch.int32, device=dev)
    nodes = torch.empty(B, dtype=torch.int32, device=dev)
    first = torch.empty((B, 6), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        check(getattr(lib, entry)(C.c_void_p(b.data_ptr()), C.c_void_p(p.data_ptr()), B, N,
                                  int(config.N_IN_ROW if n_in_row is None else n_in_row), int(max_attacks), int(node_budget),
                                  C.c_void_p(length.data_ptr()), C.c_void_p(first.data_ptr()), C.c_void_p(nodes.data_ptr()),
                                  C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), entry)
    bits = (first.unsqueeze(-1) >> torch.arange(64, device=dev)) & 1
    return length, bits.reshape(B, 6 * 64)[:, :A].bool(), nodes


def _solver_flags(entry, name, records, board_size, max_attacks, node_budget, n_in_row):
    """gmz_records_vcf / gmz_records_vct on packed move records where they lie -> uint8 [M] flags."""
    lib = _lib.load()
    N = int(board_size)
    stride = int(lib.gmz_move_record_bytes(N))
    if not torch.is_tensor(records) or records.device.type != "cuda":
        raise _lib.GmzError(f"{name} needs the records in a CUDA tensor (there is no CPU fallback)")
    if records.dtype != torch.uint8 or records.dim() != 2 or records.shape[1] != stride or not records.is_contiguous():
        raise ValueError(f"records must be a contiguous uint8 tensor [M, {stride}] of {N}x{N} move records")
    M = int(records.shape[0])
    out = torch.empty(M, dtype=torch.uint8, device=records.device)
    if M == 0:
        return out
    with torch.cuda.device(records.device):
        check(getattr(lib, entry)(C.c_void_p(records.data_ptr()), M, N, int(config.N_IN_ROW if n_in_row is None else n_in_row),
                                  int(max_attacks), int(node_budget), C.c_void_p(out.data_ptr()),
                                  C.c_void_p(torch.cuda.current_stream(records.device).cuda_stream)), entry)
    return out


def _missed_forced(flags_fn, packed, max_attacks, node_budget, n_in_row):
    """Per game of a PackedGames: the records whose flags have bit 0 (a forced win) without bit 1 (the move played
    starts one)."""
    rec, game = _game_records(packed)
    out = torch.zeros(len(packed), dtype=torch.int64, device=rec.device)
    if rec.shape[0] == 0:
        return out
    flags = flags_fn(rec, packed.N, max_attacks, node_budget, n_in_row)
    out.index_add_(0, game, ((flags & (VCF_AVAILABLE | PLAYED_VCF)) == VCF_AVAILABLE).to(torch.int64))
    return out


def find_vcf(boards, players, max_attacks=VCF_ATTACKS, node_budget=VCF_BUDGET, n_in_row=None, board_size=None,
             device=None):
    """Forced wins by continuous fours for the side to move.  boards int8 [B,N,N] or [B,A], players +-1 [B] -> device
    tensors (length int32 [B], first bool [B,A], nodes int32 [B]): the fewest attacker stones of a VCF of at most
    `max_attacks` stones (0: none, -1: the node budget ran out), every first move that starts one, and the positions
    expanded."""
    return _solve("gmz_vcf_solve", "find_vcf", boards, players, max_attacks, node_budget, n_in_row, board_size, device)


def vcf_record_flags(records, board_size, max_attacks=VCF_ATTACKS, node_budget=VCF_BUDGET, n_in_row=None):
    """The VCF twin of record_flags: packed move records (uint8 device tensor [M, stride], a trajectory.PackedGames
    block or a stretch of the DeviceReplayBuffer ring) solved where they lie for the side in each record's to_move ->
    uint8 [M] (bits VCF_AVAILABLE, PLAYED_VCF = the played action starts a VCF, VCF_UNKNOWN = the budget ran out)."""
    return _solver_flags("gmz_records_vcf", "vcf_record_flags", records, board_size, max_attacks, node_budget, n_in_row)


def missed_vcf_counts(packed, max_attacks=VCF_ATTACKS, node_budget=VCF_BUDGET, n_in_row=None):
    """Per game of a trajectory.PackedGames, in `packed.table` order: int64 [len(packed)] on the device, the moves at
    which the mover had a VCF of at most `max_attacks` stones and played a move that does not start one."""
    return _missed_forced(vcf_record_flags, packed, max_attacks, node_budget, n_in_row)


# Forced wins through threats of three: the VCT solver (include/gmz.h gmz_vct_solve).  Its flag bits are the VCF ones.
# Defaults from profiles/r12_vct.json (one B200, 1000 W limit), on 100,000 15x15 E0 self-play records: a 5,000-node
# budget cuts 22.0 % of them at 23.3 k positions/s, a 20,000-node budget still cuts 21.0 % at 6.2 k/s; max_attacks 16
# cuts more than 8 (22.7 % against 22.0 % at 5,000 nodes).
VCT_ATTACKS, VCT_BUDGET = 8, 5_000


def find_vct(boards, players, max_attacks=VCT_ATTACKS, node_budget=VCT_BUDGET, n_in_row=None, board_size=None,
             device=None):
    """Forced wins by threats of three or four (VCT) for the side to move, as find_vcf: device tensors (length int32
    [B], first bool [B,A], nodes int32 [B]) -- the fewest attacker stones, forced blocks included, of a VCT of at most
    `max_attacks` stones (0: none, -1: the node budget ran out), every first move that starts one, and the positions
    expanded.  Every VCF is a VCT, so it finds at least what find_vcf finds where neither is cut."""
    return _solve("gmz_vct_solve", "find_vct", boards, players, max_attacks, node_budget, n_in_row, board_size, device)


def vct_record_flags(records, board_size, max_attacks=VCT_ATTACKS, node_budget=VCT_BUDGET, n_in_row=None):
    """The VCT twin of vcf_record_flags -> uint8 [M] (bits VCF_AVAILABLE = the mover had a VCT, PLAYED_VCF = the played
    action starts one, VCF_UNKNOWN = the budget ran out)."""
    return _solver_flags("gmz_records_vct", "vct_record_flags", records, board_size, max_attacks, node_budget, n_in_row)


def missed_vct_counts(packed, max_attacks=VCT_ATTACKS, node_budget=VCT_BUDGET, n_in_row=None):
    """Per game of a trajectory.PackedGames, in `packed.table` order: int64 [len(packed)] on the device, the moves at
    which the mover had a VCT of at most `max_attacks` stones and played a move that does not start one."""
    return _missed_forced(vct_record_flags, packed, max_attacks, node_budget, n_in_row)


class SelfPlayStats:
    """Running self-play statistics of device self-play -- what universal_worker reports per game in
    SelfPlayStatus (workers.py:191-203, 235): games, moves, results, missed fives and missed wins.  Pass
    `add` to play() alongside the replay sink, `sink=lambda pg: (stats.add(pg), buf.add_packed(pg))`.
    Game / move / result counts come from the host-side game table; the missed counts stay in device counters, so
    `add` never waits for the GPU.  `summary()` reads them back once.

    n_openings = O > 0 also keeps, per opening of a self-play book (SearchEngine.set_openings), how often the side to
    move at the opening won, drew and lost, from each game's first record on the device; `by_opening()` reads them.
    Games without a label in [0, O) count in the totals only.

    vcf_attacks = k > 0 also solves every record for forced wins of at most k attacker stones (gmz_records_vcf, at most
    `vcf_budget` positions each) and adds to `summary()` the moves at which the mover had one (vcf_available), those
    at which it played a move that starts none (missed_vcf, and missed_vcf_per_game) and the records the budget left
    undecided (vcf_unknown).  0 leaves the statistics and the summary's keys as they are without it."""

    def __init__(self, n_in_row=None, device=None, n_openings=0, vcf_attacks=0, vcf_budget=VCF_BUDGET):
        if not torch.cuda.is_available():
            raise _lib.GmzError("SelfPlayStats needs a CUDA device (there is no CPU fallback)")
        self.n_in_row = n_in_row
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self._missed = torch.zeros(2, dtype=torch.int64, device=self.device)      # missed fives, missed wins
        self.n_openings = int(n_openings)
        self._by_opening = torch.zeros((self.n_openings, 3), dtype=torch.int64, device=self.device)
        self.vcf_attacks, self.vcf_budget = int(vcf_attacks), int(vcf_budget)
        if self.vcf_attacks < 0:
            raise ValueError("vcf_attacks must be >= 0")
        self._vcf = torch.zeros(3, dtype=torch.int64, device=self.device)        # available, missed, unknown
        self.reset()

    def reset(self):
        self.games = self.moves = self.wins_black = self.wins_white = self.draws = 0
        self._missed.zero_()
        self._by_opening.zero_()
        self._vcf.zero_()

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
        if self.vcf_attacks:
            f = vcf_record_flags(packed.records[:M], packed.N, self.vcf_attacks, self.vcf_budget, self.n_in_row)
            self._vcf += torch.stack([(f & VCF_AVAILABLE).bool().sum(), ((f & (VCF_AVAILABLE | PLAYED_VCF)) == VCF_AVAILABLE).sum(),
                                      (f & VCF_UNKNOWN).bool().sum()])
        if self.n_openings:
            # first record of each game: winner, to_move and opening label + 1, int32 columns of its header
            first = torch.as_tensor(np.asarray(packed.offsets[:-1], np.int64), device=self.device)
            hdr = packed.records[first, :RECORD_HEADER.itemsize].contiguous().view(torch.int32)
            winner, to_move, opening = (hdr[:, RECORD_HEADER.fields[f][1] // 4] for f in ("winner", "to_move", "opening"))
            label = opening.to(torch.int64) - 1
            outcome = torch.where(winner == 0, 1, torch.where(winner == to_move, 0, 2)).to(torch.int64)
            ok = (label >= 0) & (label < self.n_openings)
            self._by_opening.view(-1).index_add_(0, torch.where(ok, label * 3 + outcome, 0), ok.to(torch.int64))

    def by_opening(self):
        """int64 [n_openings, 3]: per opening, the games the side to move at the opening won, drew and lost (one device
        -> host copy)."""
        return self._by_opening.cpu().numpy()

    def summary(self):
        """dict of the counts plus avg_game_length and per-game rates (one device -> host copy)."""
        fives, missed = (int(x) for x in self._missed.tolist())
        g = self.games
        out = {"games": g, "moves": self.moves, "wins_black": self.wins_black, "wins_white": self.wins_white,
               "draws": self.draws, "missed_fives": fives, "missed_all_wins": missed,
               "avg_game_length": self.moves / g if g else 0.0,
               "missed_fives_per_game": fives / g if g else 0.0, "missed_all_wins_per_game": missed / g if g else 0.0}
        if self.vcf_attacks:
            available, missed_vcf, unknown = (int(x) for x in self._vcf.tolist())
            out.update(vcf_available=available, missed_vcf=missed_vcf, missed_vcf_per_game=missed_vcf / g if g else 0.0,
                       vcf_unknown=unknown)
        return out
