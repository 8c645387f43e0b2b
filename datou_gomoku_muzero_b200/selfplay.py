"""Batched self-play driver: the device-resident replacement of the reference's per-process game
loop (workers.py:162-189): search -> record -> do_move -> get_game_ended -> restart, for G games
at once with no host round trip inside a move.
"""
from __future__ import annotations

import numpy as np
import torch

from .engine import SearchEngine


class SelfPlayEngine:
    """evaluator: "e0" (fixed deterministic evaluator, fused persistent-kernel search); a `GomokuNetEZ` module or a
    `network.NetworkSearch` (the production evaluator of universal_worker, workers.py:129-241: one CUDA graph per
    simulation step, select -> network -> expand/backup, bf16 NHWC observations written by the select); any callable
    `f(obs f32 [G,3,N,N]) -> (logits f32 [G,A], values f32/f64 [G])` run on the device (eager stepwise path); or --
    for an engine in MuZero mode -- a pair `(initial_fn, recurrent_fn)` / a `muzero.MuZeroDeviceSearch`
    (learned dynamics in the tree, hidden states in the device pool; MuZeroMCTS.search, mcts.py:288-362).  The evaluator
    is resolved by mcts.resolve_searchers, as for re-analysis."""

    def __init__(self, engine: SearchEngine, evaluator="e0", seed=0, logit_div=16, noise_seed=0):
        self.e = engine
        self.evaluator = evaluator
        self.seed, self.logit_div, self.noise_seed = int(seed), int(logit_div), int(noise_seed)
        G, A = engine.G, engine.A
        self.gumbel = torch.empty((G, A), dtype=torch.float64, device=engine.device)
        self.noise_counter = 0
        self.moves_played = 0
        self.games_finished = 0
        self.done_mask = torch.zeros(G, dtype=torch.uint8, device=engine.device)
        from .mcts import resolve_searchers
        from .muzero import MuZeroDeviceSearch
        from .network import NetworkSearch
        searcher = resolve_searchers([engine], evaluator)[0]
        self.ns = searcher if isinstance(searcher, NetworkSearch) else None
        self.mz = searcher if isinstance(searcher, MuZeroDeviceSearch) else None
        self._e0 = isinstance(evaluator, str)
        engine.reset_games()

    def search(self, gumbel=None):
        """One search for every game from its current root; returns finalize() outputs."""
        e = self.e
        if gumbel is None:
            e.fill_gumbel(self.gumbel, self.noise_seed, self.noise_counter)
            self.noise_counter += self.gumbel.numel()
            gumbel = self.gumbel
        if self._e0:
            e.search_e0(gumbel, self.seed, self.logit_div)
        elif self.ns is not None:
            self.ns.search(gumbel)
        elif self.mz is not None:
            self.mz.search(gumbel)
        else:
            obs = e.root_obs()
            lg, v = self.evaluator(obs)
            e.root_expand(lg, v, gumbel)
            for _ in range(e.S - 1):
                obs = e.select()
                lg, v = self.evaluator(obs)
                e.expand_backup(lg, v)
        return e.finalize(want_visits=False)

    def step(self, restart=True, traj=None):
        """One self-play move for all G games through the stepwise kernels (any evaluator): search,
        decision, trajectory record, do_move, end check, restart (workers.py:168-189).  Finished games
        are harvested from `traj` exactly as with play()."""
        e = self.e
        policy, value, action, _ = self.search()
        winner = e.selfplay_step(policy, value, action, traj, restart)
        self.moves_played += e.G
        return winner

    def play(self, moves_per_game=1, traj=None, restart=True, sink=None, chunk=None):
        """Self-play of G * moves_per_game moves.  Fixed evaluator: the persistent kernel, games advancing
        independently; any other evaluator: `moves_per_game` step() calls (all games move in lock-step, one
        network batch of G per simulation).  Without `sink` the caller harvests finished games from `traj`
        (games that finish when no trajectory slot is free park until slots are released).  With `sink` -- a
        callable taking a trajectory.PackedGames, e.g. `DeviceReplayBuffer.add_packed` -- the run is cut into
        pieces of `chunk` moves per game (default: what the store's spare slots absorb, at most 48; 1 for a network
        evaluator) and after
        each one the finished games are packed on the device, handed to the sink and their slots recycled, so a
        run of any length never parks a game."""
        e = self.e
        total = int(moves_per_game)

        def advance(n):
            if self._e0:
                e.selfplay_e0(e.G * n, self.seed, self.logit_div, self.noise_seed, traj, restart)
                self.moves_played += e.G * n
            else:
                for _ in range(n):
                    self.step(restart, traj)

        if sink is None or traj is None:
            advance(total)
            return
        if chunk is None and not self._e0:
            chunk = 1              # lock-step games finish in bursts and a move costs S network batches: pack after every move
        if chunk is None:          # a game ends about every A/3 moves at the earliest in practice; spare slots absorb the finishes
            spare = max(1, traj.n_slots - e.G)
            chunk = int(max(4, min(48, spare * (e.A // 3) // max(1, e.G))))
        done = 0
        while done < total:
            n = min(int(chunk), total - done)
            advance(n)
            done += n
            packed = traj.pack_finished(recycle=True)
            if packed is not None:
                sink(packed)
                self.games_finished += len(packed)

    def count_finished(self, winner):
        n = int((winner != 2).sum().item())
        self.games_finished += n
        return n
