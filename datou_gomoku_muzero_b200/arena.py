"""Arena: two players play each other on the GPU -- new weights against old ones, a MuZero-mode net against an
AlphaZero-mode one, 800 simulations against 400 -- colour-paired from an opening book, with results and an Elo estimate.

A player is a SearchEngine plus any evaluator `mcts.resolve_searchers` accepts.  The two engines must agree on the
number of games G, the board size and n_in_row; everything else (S, K, mode, accum_dtype, c_visit, ...) may differ, and
every search is the one that player's engine runs on its own: a player's move is what its engine chooses at that root
with that noise.

    res = Arena(eA, eB, new_net, old_net).play(random_openings(200, 4, 15, seed=step))
    res.elo()

Each opening is played twice: ticket 2o with A moving first, ticket 2o + 1 with B moving first (the first mover takes
the opening's side to move).  The 2G games in flight sit in slot g of engine A (A to move) or of engine B (B to move)
and change engines after every ply (csrc/gmz_match.cu), so both engines search G real roots per ply until the opening
queues run dry.  The Gumbel noise of ply k of opening o is gmz_fill_gumbel's draw at counters (o*A + k)*A ... + A - 1
of the match seed, shared by both games of the pair and independent of G and of the order games finish in: the same
match with G = 8 or G = 4096 plays the same games, and a player against itself scores exactly 50 %.
"""
from __future__ import annotations

import ctypes as C
import math
from collections import namedtuple

import numpy as np
import torch

from ._lib import GMZ_WINNER_NONE, GmzMatch, check
from .game import GomokuGame

# An opening book of O positions: boards int8 [O, A] in {-1, 0, +1}, the side to move int8 [O] (+-1), the last move
# int32 [O] (action index, -1 = None) and the move count int32 [O].
Openings = namedtuple("Openings", "boards players last_moves move_counts")

_Z95 = 1.959963984540054      # two-sided 95 % quantile of the standard normal


def empty_opening(board_size):
    """The default book: one empty board, black to move."""
    A = int(board_size) ** 2
    return Openings(np.zeros((1, A), np.int8), np.ones(1, np.int8), np.full(1, -1, np.int32), np.zeros(1, np.int32))


def check_openings(openings, board_size, n_in_row):
    """The book as contiguous host arrays of the documented dtypes; ValueError for a position a match cannot start from:
    a value outside {-1, 0, 1}, a side to move that is not +-1, a bad shape or last move, no empty cell, a move count
    below the number of stones (a full board would then not be a draw), or a game that has already ended by
    get_game_ended's rules."""
    N = int(board_size)
    A = N * N
    if openings is None:
        return empty_opening(N)
    boards, players, last, mc = (np.asarray(x) for x in openings)
    if boards.ndim == 3 and boards.shape[1:] == (N, N):
        boards = boards.reshape(boards.shape[0], A)
    if boards.ndim != 2 or boards.shape[1] != A or boards.shape[0] < 1:
        raise ValueError(f"opening boards must be [O, {A}] or [O, {N}, {N}] with O >= 1, not {list(boards.shape)}")
    O = boards.shape[0]
    for name, x in (("players", players), ("last_moves", last), ("move_counts", mc)):
        if x.shape != (O,):
            raise ValueError(f"opening {name} must have shape [{O}], not {list(x.shape)}")
    if not np.isin(boards, (-1, 0, 1)).all():
        raise ValueError("opening boards hold values outside {-1, 0, 1}")
    if not np.isin(players, (-1, 1)).all():
        raise ValueError("the side to move of an opening must be +1 or -1")
    if ((last < -1) | (last >= A)).any():
        raise ValueError(f"opening last moves must be -1 (None) or an action index below {A}")
    stones = (boards != 0).sum(axis=1)
    if (stones == A).any():
        raise ValueError(f"opening {int(np.flatnonzero(stones == A)[0])} has no empty cell")
    if (mc < stones).any():
        raise ValueError(f"opening {int(np.flatnonzero(mc < stones)[0])} has a move count below its number of stones")
    g = GomokuGame(board_size=N, n_in_row=int(n_in_row))
    for o in range(O):
        g.board = boards[o].reshape(N, N).astype(np.int8)
        g.last_move = None if last[o] < 0 else divmod(int(last[o]), N)
        g.move_count = int(mc[o])
        if g.get_game_ended() is not None:
            raise ValueError(f"opening {o} has already ended")
    return Openings(np.ascontiguousarray(boards, np.int8), np.ascontiguousarray(players, np.int8),
                    np.ascontiguousarray(last, np.int32), np.ascontiguousarray(mc, np.int32))


def random_openings(n, stones, board_size=15, seed=0, n_in_row=5):
    """`n` openings of `stones` alternating stones (black first) on random cells of a square window around the centre,
    about four cells per stone; a position in which the game has already ended is drawn again.  The side to move is the
    next colour, so odd `stones` gives white-to-move openings."""
    N, stones = int(board_size), int(stones)
    A = N * N
    if not 0 <= stones < A:
        raise ValueError(f"stones must be in [0, {A})")
    w = min(N, max(3, math.ceil(math.sqrt(4 * stones)) + 1))
    lo = (N - w) // 2
    cells = np.array([r * N + c for r in range(lo, lo + w) for c in range(lo, lo + w)])
    if stones > cells.size:
        cells = np.arange(A)
    rs = np.random.RandomState(seed)
    boards = np.zeros((n, A), np.int8)
    g = GomokuGame(board_size=N, n_in_row=int(n_in_row))
    last = np.full(n, -1, np.int32)
    for o in range(n):
        while True:
            g.reset()
            for a in rs.choice(cells, stones, replace=False):
                g.do_move(int(a))
                if g.get_game_ended() is not None:
                    break
            else:
                break
        boards[o] = g.board.reshape(A)
        last[o] = -1 if g.last_move is None else g.last_move[0] * N + g.last_move[1]
    players = np.full(n, 1 if stones % 2 == 0 else -1, np.int8)
    return Openings(boards, players, last, np.full(n, stones, np.int32))


def _opening_lengths(solve, book, max_attacks, node_budget, n_in_row, board_size):
    """(mover [O], opponent [O]) int32: `solve`'s length for the side to move of each opening and for the other side."""
    boards, players = np.asarray(book.boards), np.asarray(book.players)
    O = boards.shape[0]
    N = int(board_size) if board_size else (boards.shape[1] if boards.ndim == 3 else int(round(math.sqrt(boards.shape[1]))))
    boards = np.ascontiguousarray(boards.reshape(O, N * N), np.int8)
    side = np.where(players >= 0, 1, -1).astype(np.int8)
    length, _, _ = solve(np.concatenate([boards, boards]), np.concatenate([side, -side]), max_attacks, node_budget,
                         n_in_row=n_in_row, board_size=N)
    length = length.cpu().numpy()
    return length[:O], length[O:]


def opening_vcf(book, max_attacks=8, node_budget=20_000, n_in_row=5, board_size=None):
    """Which openings of a book are already decided by a forced win (tactics.find_vcf on the GPU): int32 arrays
    (mover [O], opponent [O]) = the VCF length of the side to move, and the length the other side would have if it were
    to move (0: none within `max_attacks` stones, -1: the node budget ran out).  A balanced book keeps
    `(mover == 0) & (opponent == 0)`."""
    from .tactics import find_vcf
    return _opening_lengths(find_vcf, book, max_attacks, node_budget, n_in_row, board_size)


def opening_vct(book, max_attacks=None, node_budget=None, n_in_row=5, board_size=None):
    """opening_vcf through threats of three (tactics.find_vct, defaults VCT_ATTACKS / VCT_BUDGET): (mover [O],
    opponent [O]) VCT lengths, 0 none, -1 the budget ran out.  It flags every opening opening_vcf decides where neither
    search is cut, and the openings won by threes besides; a balanced book keeps `(mover == 0) & (opponent == 0)`."""
    from .tactics import VCT_ATTACKS, VCT_BUDGET, find_vct
    return _opening_lengths(find_vct, book, VCT_ATTACKS if max_attacks is None else max_attacks,
                            VCT_BUDGET if node_budget is None else node_budget, n_in_row, board_size)


def elo_of(score):
    """Elo difference of an expected score: -400 log10(1/s - 1), -inf / +inf at 0 / 1."""
    if score <= 0.0:
        return -math.inf
    if score >= 1.0:
        return math.inf
    return -400.0 * math.log10(1.0 / score - 1.0)


def elo_stats(pair_scores):
    """Score, Elo difference with a 95 % interval and the likelihood of superiority from per-pair scores (each the mean
    of the two games of an opening, in [0, 1]).  The interval and the LOS use the normal approximation with the variance
    of the pair scores, which counts the correlation of the two games of a pair (pentanomial model)."""
    x = np.asarray(pair_scores, dtype=np.float64)
    n = x.size
    if n == 0:
        return dict(pairs=0, score=math.nan, elo=math.nan, elo_lo=math.nan, elo_hi=math.nan, los=math.nan)
    s = float(x.mean())
    se = math.sqrt(float(((x - s) ** 2).mean()) / n)
    if se == 0.0:
        los = 0.5 if s == 0.5 else float(s > 0.5)
    else:
        los = 0.5 * (1.0 + math.erf((s - 0.5) / se / math.sqrt(2.0)))
    return dict(pairs=n, score=s, elo=elo_of(s), elo_lo=elo_of(s - _Z95 * se), elo_hi=elo_of(s + _Z95 * se), los=los)


class MatchResult:
    """The outcome of a match, on the host.  Per-game table over the 2O tickets (ticket 2o: opening o, A first; 2o + 1:
    B first): `opening`, `a_first`, `a_colour` (+-1), `winner` (+-1, 0 draw, 2 = unfinished), `length` (plies);
    `moves` int32 [2O, A] (-1 past the end).  Statistics count finished games only, and the pair statistics pairs whose
    two games both finished."""

    def __init__(self, results, moves, openings, board_size, n_in_row=5, plies=0):
        results = np.asarray(results, np.int32).reshape(-1, 4)
        self.openings = openings
        self.board_size, self.n_in_row, self.plies = int(board_size), int(n_in_row), int(plies)
        self.moves = np.asarray(moves, np.int32)
        self.winner, self.length = results[:, 0].copy(), results[:, 1].copy()
        self.a_first = (np.arange(results.shape[0]) % 2) == 0
        self.a_colour = results[:, 3].copy()
        self.opening = np.arange(results.shape[0]) // 2
        self.finished = self.winner != GMZ_WINNER_NONE
        # A's score per game: 1 win, 0.5 draw, 0 loss (nan: unfinished)
        self.a_score = np.where(self.finished, np.where(self.winner == 0, 0.5, (self.winner == self.a_colour) * 1.0), np.nan)

    def __len__(self):
        return int(self.finished.sum())

    def wdl(self, colour=None):
        """(wins, draws, losses) of player A over the finished games, or only those A played with `colour` (+-1)."""
        m = self.finished if colour is None else self.finished & (self.a_colour == colour)
        s = self.a_score[m]
        return int((s == 1.0).sum()), int((s == 0.5).sum()), int((s == 0.0).sum())

    def pair_scores(self):
        """A's mean score over the two games of every opening whose games both finished."""
        s = self.a_score.reshape(-1, 2)
        return s[~np.isnan(s).any(axis=1)].mean(axis=1)

    def pairs(self):
        """Pentanomial counts: openings where A scored 0, 0.5, 1, 1.5, 2 points over its two games."""
        return np.bincount(np.rint(self.pair_scores() * 4).astype(np.int64), minlength=5)[:5]

    def score(self):
        """A's mean score over the finished games."""
        return float(np.nanmean(self.a_score)) if len(self) else math.nan

    def elo(self):
        """dict(pairs, score, elo, elo_lo, elo_hi, los) of A against B from the pair scores (see elo_stats)."""
        return elo_stats(self.pair_scores())

    def game_record(self, i):
        """Ticket i as a host GameRecord, rebuilt by replaying its moves from its opening.  A match keeps moves only:
        each policy is the one-hot of the move played, and the value targets are the n-step returns of the game's
        rewards with no search value to bootstrap from."""
        from .trajectory import build_game_record
        N, A = self.board_size, self.board_size ** 2
        o, T = int(self.opening[i]), int(self.length[i])
        if not self.finished[i]:
            raise ValueError(f"game {i} has not finished")
        actions = self.moves[i, :T]
        pol = np.zeros((T, A), np.float64)
        pol[np.arange(T), actions] = 1.0
        rec = dict(start_board=self.openings.boards[o].reshape(N, N), length=T, start_player=int(self.openings.players[o]),
                   start_last_move=int(self.openings.last_moves[o]), actions=actions, winner=int(self.winner[i]),
                   values=np.zeros(T), policies=pol)
        return build_game_record(rec, N)


class Arena:
    """Player A = (engine_a, evaluator_a), player B = (engine_b, evaluator_b).  Evaluators are resolved once, here, by
    mcts.resolve_searchers; eval_seed / logit_div configure an "e0" evaluator (logit_div 0 = dense, or a power of two).
    `seed` is the match's noise seed.  Everything is checked before any kernel runs (ValueError)."""

    def __init__(self, engine_a, engine_b, evaluator_a="e0", evaluator_b="e0", *, eval_seed_a=0, eval_seed_b=0,
                 logit_div_a=16, logit_div_b=16, seed=0, check_every=4):
        from .mcts import resolve_searchers
        from .muzero import MuZeroDeviceSearch
        if engine_a is engine_b:
            raise ValueError("the two players need two different engines")
        for what, f in (("num_games", lambda e: e.G), ("board size", lambda e: e.N),
                        ("n_in_row", lambda e: e.cfg.n_in_row), ("device", lambda e: e.device)):
            if f(engine_a) != f(engine_b):
                raise ValueError(f"the engines differ in {what}: {f(engine_a)} vs {f(engine_b)}")
        self.engines = (engine_a, engine_b)
        self.searchers = (resolve_searchers([engine_a], evaluator_a, eval_seed_a, logit_div_a)[0],
                          resolve_searchers([engine_b], evaluator_b, eval_seed_b, logit_div_b)[0])
        self.seed, self.check_every = int(seed), max(1, int(check_every))
        G, A, dev = engine_a.G, engine_a.A, engine_a.device
        self.budgets = []
        for s in self.searchers:             # learned dynamics: every game gets the largest budget any root can need
            if isinstance(s, MuZeroDeviceSearch):
                most = int(s.budget_table().max())
                s.check_budget(most)
                rows = torch.full((G,), most, dtype=torch.int32, device=dev)
                self.budgets.append((rows, G * most, most - 1))
            else:
                self.budgets.append(None)
        self.gumbel = tuple(torch.zeros((G, A), dtype=torch.float64, device=dev) for _ in range(2))
        self.streams = tuple(torch.cuda.Stream(device=dev) for _ in range(2))
        self.lib = engine_a.lib
        self.plies = 0
        self._buf = None

    def _cur(self):
        return torch.cuda.current_stream(self.engines[0].device)

    def start(self, openings=None):
        """Load an opening book (None = one empty board) and deal the first games into both engines' slots."""
        a, b = self.engines
        op = check_openings(openings, a.N, a.cfg.n_in_row)
        O, G, A, dev = op.boards.shape[0], a.G, a.A, a.device
        results = torch.zeros((2 * O, 4), dtype=torch.int32)
        results[:, 0] = GMZ_WINNER_NONE
        bf = dict(boards=torch.from_numpy(op.boards).to(dev), players=torch.from_numpy(op.players).to(dev),
                  last=torch.from_numpy(op.last_moves).to(dev), mc=torch.from_numpy(op.move_counts).to(dev),
                  cursor=torch.zeros(2, dtype=torch.int32, device=dev),
                  slot_ticket=torch.full((2, G), -1, dtype=torch.int32, device=dev),
                  slot_ply=torch.zeros((2, G), dtype=torch.int32, device=dev), results=results.to(dev),
                  moves=torch.full((2 * O, A), -1, dtype=torch.int32, device=dev),
                  finished=torch.zeros(1, dtype=torch.int32, device=dev))
        p = {k: v.data_ptr() for k, v in bf.items()}
        self.c = GmzMatch(O, 0, p["boards"], p["players"], p["last"], p["mc"], p["cursor"], p["slot_ticket"], p["slot_ply"],
                          p["results"], p["moves"], p["finished"])
        self._buf, self.openings, self.plies = bf, op, 0
        check(self.lib.gmz_match_start(a.handle, b.handle, C.byref(self.c), C.c_void_p(self._cur().cuda_stream)),
              "gmz_match_start")

    @torch.no_grad()
    def ply(self):
        """One ply of every game in flight: both players' noise, each engine's search on its own stream (the two may
        overlap), both decisions, then gmz_match_step on the current stream.  Nothing is read back to the host."""
        if self._buf is None:
            raise RuntimeError("start() the match first")
        a, b = self.engines
        cur = self._cur()
        st = C.c_void_p(cur.cuda_stream)
        check(self.lib.gmz_match_noise(a.handle, b.handle, C.byref(self.c), C.c_uint64(self.seed & (2**64 - 1)),
                                       self.gumbel[0].data_ptr(), self.gumbel[1].data_ptr(), st), "gmz_match_noise")
        for i, eng in enumerate(self.engines):
            self.streams[i].wait_stream(cur)
            with torch.cuda.stream(self.streams[i]):
                self.searchers[i].search(self.gumbel[i], self.budgets[i])
                eng.finalize(want_visits=False)
        for s in self.streams:
            cur.wait_stream(s)
        check(self.lib.gmz_match_step(a.handle, b.handle, C.byref(self.c), a.action.data_ptr(), b.action.data_ptr(), st),
              "gmz_match_step")
        self.plies += 1

    def finished(self):
        """Games finished so far (reads one device counter)."""
        return int(self._buf["finished"].item())

    def play(self, openings=None, max_plies=None):
        """Play the whole book (each opening once with each player first) and return its MatchResult.  The finished
        counter is read every `check_every` plies; `max_plies` stops early (unfinished games are marked as such)."""
        self.start(openings)
        total = 2 * self.openings.boards.shape[0]
        while max_plies is None or self.plies < int(max_plies):
            self.ply()
            if self.plies % self.check_every == 0 and self.finished() >= total:
                break
        return self.result()

    def result(self):
        """The match so far as a MatchResult."""
        res = self._buf["results"].cpu().numpy()
        n = self.finished()
        if n != int((res[:, 0] != GMZ_WINNER_NONE).sum()):
            raise RuntimeError("a game in the match ended without a move from its player's search")
        a = self.engines[0]
        return MatchResult(res, self._buf["moves"].cpu().numpy(), self.openings, a.N, a.cfg.n_in_row, self.plies)
