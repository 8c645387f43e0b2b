"""AlphaZeroMCTS / MuZeroMCTS with the reference's class interface (mcts.py:50-64, 191-362),
backed by the CUDA engine.

Two ways in:
  * `AlphaZeroMCTS(worker_id, request_queue, result_queue).search(game)` -- the reference's
    constructor and call, batch of one, evaluator reached through the reference's queue protocol
    (mcts.py:73-85).  Same outputs `(policy float64[A], value, int action)`, same sentinel
    `(zeros, 0.0, -1)`, same request pattern (NUM_SIMULATIONS 'initial' requests in AlphaZero mode;
    one 'initial' + 'recurrent_batch' requests in MuZero mode), same use of `np.random.gumbel`.
    The tree arithmetic follows the dtype of the evaluator's value scalar exactly as the reference's
    does under NumPy >= 2 (SURVEY App. A.7): Python floats -> float64 engine; np.float32 (what the
    reference's inference server returns, workers.py:355,368) -> float32-accumulation engine, and the
    returned `value` is then an np.float32 as well.
  * `AlphaZeroMCTS.for_engine(engine, evaluator=...)` + `search_batch(...)` -- G searches at once
    from host buffers, evaluator on the device: any evaluator `resolve_searchers` accepts.
The tree itself (selection, expansion, backup, halving, decision) always runs in the kernels.
"""
from __future__ import annotations

import logging
from abc import ABC, abstractmethod
from queue import Empty

import numpy as np

from .config import config


class MCTS(ABC):
    def __init__(self, worker_id, request_queue, result_queue):
        self.worker_id = worker_id
        self.request_queue = request_queue
        self.result_queue = result_queue
        self.logger = logging.getLogger(f"MCTS-{self.__class__.__name__}-{worker_id}")

    @abstractmethod
    def search(self, game):
        """Run one search; returns (policy, value, action)."""


class _GumbelEngineMCTS(MCTS):
    MODE = "AlphaZero"

    def __init__(self, worker_id=0, request_queue=None, result_queue=None):
        super().__init__(worker_id, request_queue, result_queue)
        self._engines = {}
        self._batch = None
        self._last = None       # (engine, move) of the last search(game), for last_tree()

    # ------------------------------------------------------------------ queue protocol (mcts.py:73-85)
    def _remote_initial_inference(self, obs):
        self.request_queue.put((self.worker_id, "initial", obs))
        return self.result_queue.get(timeout=20)

    def _remote_recurrent_inference_batch(self, hidden_states_batch, actions_batch):
        if not actions_batch:
            return []
        self.request_queue.put((self.worker_id, "recurrent_batch",
                                (hidden_states_batch, np.array(actions_batch, dtype=np.int32))))
        try:
            p, v, h, r = self.result_queue.get(timeout=20)
            return [(p[i], v[i, 0], h[i:i + 1], r[i, 0]) for i in range(len(actions_batch))]
        except Empty:
            self.logger.warning(f"Worker {self.worker_id} timed out waiting for recurrent inference.")
            return []

    @staticmethod
    def _accum_of(value):
        """dtype the reference's value_sum takes from this evaluator scalar (0 + np.float32 stays float32)."""
        return "float32" if isinstance(value, np.float32) else "float64"

    def _engine_for_config(self, accum="float64"):
        from .engine import SearchEngine
        key = (config.BOARD_SIZE, config.N_IN_ROW, config.NUM_SIMULATIONS, config.NUM_TOP_ACTIONS, config.C_VISIT,
               config.C_SCALE, config.VALUE_MINMAX_DELTA, config.DISCOUNT, accum)
        eng = self._engines.get(key)
        if eng is None:
            eng = SearchEngine(1, board_size=config.BOARD_SIZE, n_in_row=config.N_IN_ROW,
                               num_simulations=config.NUM_SIMULATIONS, num_top_actions=config.NUM_TOP_ACTIONS,
                               mode=self.MODE, c_visit=config.C_VISIT, c_scale=config.C_SCALE,
                               minmax_delta=config.VALUE_MINMAX_DELTA, discount=config.DISCOUNT, accum_dtype=accum)
            self._engines = {key: eng}      # one live engine per instance
        return eng

    def _drain(self):
        try:
            while True:
                self.result_queue.get_nowait()
        except Empty:
            pass

    def _load_root(self, eng, game):
        n = config.BOARD_SIZE
        board = np.ascontiguousarray(game.board, dtype=np.int8).reshape(1, n * n)
        lm = -1 if game.last_move is None else int(game.last_move[0]) * n + int(game.last_move[1])
        eng.set_roots(board, np.array([game.current_player], np.int8), np.array([lm], np.int32),
                      np.array([game.move_count], np.int32))

    def _decision(self, eng):
        pol, val, act, _ = eng.finalize(want_visits=False)
        value = val[0].cpu().numpy()[()]
        if eng.accum_dtype == "float32":
            value = np.float32(value)          # root.get_value() is an np.float32 in this mode (exact: it was computed in float32)
        self._last = (eng, int(act[0].item()))
        return pol[0].cpu().numpy(), value, self._last[1]

    def last_tree(self):
        """The tree of the last `search(game)` as host numpy arrays (searchtree.SearchTrees.game), its principal variation
        starting with the move `search` returned: the expected line, every root move's visits / Q / prior and Gumbel
        fate, every node's statistics.  None if that search returned the sentinel (or none ran)."""
        if self._last is None:
            return None
        eng, action = self._last
        return eng.export_tree().game(0, first=action)

    # ------------------------------------------------------------------ batched entry
    @classmethod
    def for_engine(cls, engine, evaluator="e0", eval_seed=0, logit_div=16):
        """Batched searches on `engine` with any evaluator `resolve_searchers` accepts (resolved once, here)."""
        import torch
        searcher = resolve_searchers([engine], evaluator, eval_seed, logit_div)[0]
        self = cls(0, None, None)
        G, A = engine.G, engine.A
        pin = dict(pin_memory=True)
        self._batch = dict(
            engine=engine, searcher=searcher,
            h_rows=torch.empty(G, dtype=torch.int32, **pin), d_rows=torch.empty(G, dtype=torch.int32, device=engine.device),
            h_boards=torch.empty((G, A), dtype=torch.int8, **pin), h_players=torch.empty(G, dtype=torch.int8, **pin),
            h_last=torch.empty(G, dtype=torch.int32, **pin), h_mc=torch.empty(G, dtype=torch.int32, **pin),
            h_gumbel=torch.empty((G, A), dtype=torch.float64, **pin),
            d_boards=torch.empty((G, A), dtype=torch.int8, device=engine.device),
            d_players=torch.empty(G, dtype=torch.int8, device=engine.device),
            d_last=torch.empty(G, dtype=torch.int32, device=engine.device),
            d_mc=torch.empty(G, dtype=torch.int32, device=engine.device),
            d_gumbel=torch.empty((G, A), dtype=torch.float64, device=engine.device),
            o_policy=torch.empty((G, A), dtype=torch.float64, **pin), o_value=torch.empty(G, dtype=torch.float64, **pin),
            o_action=torch.empty(G, dtype=torch.int32, **pin))
        return self

    def search_batch(self, boards, players, last_moves, move_counts, gumbel=None):
        """G searches from HOST arrays: boards int8 [G,A|N,N], players +-1 [G], last_moves (action index or -1)
        [G], move_counts [G], gumbel float64 [G,A] (drawn with np.random.gumbel if omitted, like the reference).
        Returns host arrays (policy float64 [G,A], value float64 [G], action int32 [G])."""
        import torch
        self.enqueue_batch(boards, players, last_moves, move_counts, gumbel)
        torch.cuda.current_stream(self._batch["engine"].device).synchronize()
        b = self._batch
        return b["o_policy"].numpy(), b["o_value"].numpy(), b["o_action"].numpy()

    def enqueue_batch(self, boards, players, last_moves, move_counts, gumbel=None, device_noise=None):
        """Asynchronous half of search_batch: stages the inputs in pinned memory and enqueues H2D copies,
        the search, the decision and the D2H copies on the current stream.  The pinned output arrays
        (`_batch["o_*"]`) are valid once that stream has been synchronised.  device_noise = (seed, counter):
        draw the Gumbel noise on the device (gmz_fill_gumbel) instead of shipping a host array."""
        b = self._batch
        if b is None:
            raise RuntimeError("search_batch needs an instance made with for_engine()")
        eng = b["engine"]
        G, A = eng.G, eng.A
        if gumbel is None and device_noise is None:
            gumbel = np.random.gumbel(0, 1, (G, A))
        b["h_boards"].numpy()[...] = np.asarray(boards, dtype=np.int8).reshape(G, A)
        b["h_players"].numpy()[...] = np.asarray(players, dtype=np.int8)
        b["h_last"].numpy()[...] = np.asarray(last_moves, dtype=np.int32)
        b["h_mc"].numpy()[...] = np.asarray(move_counts, dtype=np.int32)
        keys = ("boards", "players", "last", "mc")
        if device_noise is None:
            b["h_gumbel"].numpy()[...] = np.asarray(gumbel, dtype=np.float64).reshape(G, A)
            keys += ("gumbel",)
        else:
            eng.fill_gumbel(b["d_gumbel"], int(device_noise[0]), int(device_noise[1]))
        from .muzero import MuZeroDeviceSearch
        searcher, budget = b["searcher"], None
        if isinstance(searcher, MuZeroDeviceSearch):      # per-game node budgets from the host boards
            rows = searcher.host_budgets(b["h_boards"].numpy())
            b["h_rows"].numpy()[...] = rows
            keys += ("rows",)
            budget = (b["d_rows"], int(rows.sum()), int(rows.max()) - 1)
        for k in keys:
            b["d_" + k].copy_(b["h_" + k], non_blocking=True)
        eng.set_roots(b["d_boards"], b["d_players"], b["d_last"], b["d_mc"])
        searcher.search(b["d_gumbel"], budget)
        pol, val, act, _ = eng.finalize(want_visits=False)
        b["o_policy"].copy_(pol, non_blocking=True)
        b["o_value"].copy_(val, non_blocking=True)
        b["o_action"].copy_(act, non_blocking=True)


class E0Search:
    """The fixed evaluator E0 in the fused search kernel (either engine mode): evaluator seed `seed`, logits divided by
    `logit_div` (0 = dense logits, else a power of two).  A searcher as resolve_searchers describes."""

    def __init__(self, engine, seed=0, logit_div=16):
        seed, logit_div = int(seed), int(logit_div)
        if logit_div < 0 or logit_div & (logit_div - 1):
            raise ValueError("an 'e0' evaluator needs logit_div 0 (dense) or a power of two")
        self.e, self.seed, self.logit_div = engine, seed, logit_div

    def search(self, gumbel, budget=None):
        self.e.search_e0(gumbel, self.seed, self.logit_div)


class StepwiseSearch:
    """An eager evaluator fn(obs f32 [G,3,N,N]) -> (logits f32 [G,A], values [G]) driving the stepwise kernels (AlphaZero
    mode): root_obs -> fn -> root_expand, then S - 1 rounds of select -> fn -> expand_backup.  A searcher as
    resolve_searchers describes."""

    def __init__(self, engine, fn):
        self.e, self.fn = engine, fn

    def search(self, gumbel, budget=None):
        e = self.e
        lg, v = self.fn(e.root_obs())
        e.root_expand(lg, v, gumbel)
        for _ in range(e.S - 1):
            lg, v = self.fn(e.select())
            e.expand_backup(lg, v)


def resolve_searchers(engines, evaluator, eval_seed=0, logit_div=16):
    """One searcher per engine for `evaluator`, checked before anything is enqueued (ValueError otherwise):
      "e0"                              -> an E0Search(engine, eval_seed, logit_div) per engine (either engine mode);
      callable f(obs f32 [G,3,N,N]) -> (logits f32 [G,A], values [G])
                                        -> a StepwiseSearch per engine: eager select -> f -> expand_backup (AlphaZero);
      torch.nn.Module (GomokuNetEZ)     -> a network.NetworkSearch per engine, bf16, one CUDA graph per step (AlphaZero);
      (initial_fn, recurrent_fn)        -> a muzero.MuZeroDeviceSearch(graph=True) per engine (MuZero mode);
      [searcher, ...]                   -> already-built searchers of those four types, one bound to each engine in
                                           order (reused across calls: no re-capture, update_weights swaps weights in
                                           place).
    A lone searcher stands for a one-element list.  Every searcher `s` has `s.e`, the engine it drives, and
    `s.search(gumbel, budget=None)`, which enqueues one search of every root loaded in that engine on the current stream
    (follow with engine.finalize()); `budget` = (rows int32 device [G], arena rows, steps) gives a MuZeroDeviceSearch
    per-game node budgets in its compact arena and its exact step count, and is unused by the others."""
    import torch
    from .muzero import MuZeroDeviceSearch
    from .network import NetworkSearch
    engines = list(engines)
    built = (E0Search, StepwiseSearch, NetworkSearch, MuZeroDeviceSearch)
    if isinstance(evaluator, built):
        evaluator = [evaluator]
    if isinstance(evaluator, (tuple, list)) and evaluator and all(isinstance(x, built) for x in evaluator):
        if len(evaluator) != len(engines):
            raise ValueError(f"{len(evaluator)} searchers for {len(engines)} engines: pass one per engine")
        for s, e in zip(evaluator, engines):
            kind = "MuZero" if isinstance(s, MuZeroDeviceSearch) else None if isinstance(s, E0Search) else "AlphaZero"
            if kind is not None and e.mode != kind:
                raise ValueError(f"a {type(s).__name__} needs a {kind}-mode engine, not a {e.mode}-mode one")
            if s.e is not e:
                raise ValueError(f"the {type(s).__name__} drives a different engine")
        return list(evaluator)
    if isinstance(evaluator, str):
        if evaluator != "e0":
            raise ValueError(f"unknown evaluator {evaluator!r}")
        return [E0Search(e, eval_seed, logit_div) for e in engines]
    pair = isinstance(evaluator, (tuple, list)) and len(evaluator) == 2 and all(callable(f) for f in evaluator)
    module = isinstance(evaluator, torch.nn.Module)
    for e in engines:
        if e.mode == "MuZero" and not pair:
            raise ValueError("a MuZero-mode engine needs evaluator='e0', (initial_fn, recurrent_fn) or a MuZeroDeviceSearch")
        if e.mode == "AlphaZero" and (pair or not callable(evaluator)):
            raise ValueError("an AlphaZero-mode engine needs evaluator='e0', a GomokuNetEZ module, a NetworkSearch or a "
                             "callable f(obs) -> (logits, values); (initial_fn, recurrent_fn) drives MuZero-mode engines")
    if pair:
        return [MuZeroDeviceSearch(e, evaluator[0], evaluator[1], graph=True) for e in engines]
    if module:
        return [NetworkSearch(e, evaluator) for e in engines]
    return [StepwiseSearch(e, evaluator) for e in engines]


def host_budgets(mz, boards):
    """mz.host_budgets(boards) for a MuZeroDeviceSearch `mz`, under the name callers of this module import."""
    return mz.host_budgets(boards)


class PipelinedBatchSearch:
    """Double-buffered `search_batch`: consecutive host batches alternate between engines (own node
    pools, own CUDA stream), so batch i+1's copies and the bulk of its search overlap the tail of
    batch i (per-search work is heavy tailed; a lone batch ends with a few slow games on an idle GPU).

        pipe = PipelinedBatchSearch([eng_a, eng_b], evaluator="e0", eval_seed=...)
        t0 = pipe.submit(boards0, ...); t1 = pipe.submit(boards1, ...)
        policy, value, action = pipe.result(t0)        # host arrays, valid until that lane is reused
    """

    def __init__(self, engines, cls=None, evaluator="e0", eval_seed=0, logit_div=16):
        import torch
        cls = cls or AlphaZeroMCTS
        searchers = resolve_searchers(engines, evaluator, eval_seed, logit_div)
        self.lanes = [cls.for_engine(e, s) for e, s in zip(engines, searchers)]
        self.streams = [torch.cuda.Stream(device=e.device) for e in engines]
        for e, s in zip(engines, self.streams):      # work already enqueued on the engines (e.g. a ring re-analysis) comes first
            s.wait_stream(torch.cuda.current_stream(e.device))
        self.events = [None] * len(engines)
        self.n = 0

    def submit(self, boards, players, last_moves, move_counts, gumbel=None, device_noise=None):
        import torch
        i = self.n % len(self.lanes)
        if self.events[i] is not None:
            self.events[i].synchronize()           # the lane's pinned buffers are about to be overwritten
        with torch.cuda.stream(self.streams[i]):
            self.lanes[i].enqueue_batch(boards, players, last_moves, move_counts, gumbel, device_noise)
            ev = torch.cuda.Event()
            ev.record(self.streams[i])
        self.events[i] = ev
        self.n += 1
        return i

    def result(self, ticket):
        self.events[ticket].synchronize()
        b = self.lanes[ticket]._batch
        return b["o_policy"].numpy(), b["o_value"].numpy(), b["o_action"].numpy()


class AlphaZeroMCTS(_GumbelEngineMCTS):
    """Search on real game states: every simulation evaluates the replayed board (mcts.py:191-280)."""
    MODE = "AlphaZero"

    def search(self, game):
        self._drain()
        self._last = None
        A = config.ACTION_SPACE_SIZE
        obs = game.get_board_state(game.current_player, game.last_move)
        try:
            policy_logits, value, _hidden = self._remote_initial_inference(obs)
        except Empty:
            self.logger.warning(f"Worker {self.worker_id} timed out on initial inference.")
            return np.zeros(A), 0.0, -1
        if not (np.asarray(game.board) == 0).any():
            return np.zeros(A), 0.0, -1
        vdt = np.float32 if isinstance(value, np.float32) else np.float64
        eng = self._engine_for_config(self._accum_of(value))
        self._load_root(eng, game)
        gumbel = np.random.gumbel(0, 1, A)
        eng.root_expand(np.asarray(policy_logits, np.float32).reshape(1, A), np.array([value], vdt), gumbel.reshape(1, A))
        sim_count = 1
        while sim_count < config.NUM_SIMULATIONS:
            leaf_obs = eng.select()[0].cpu().numpy()
            try:
                lg, v, _h = self._remote_initial_inference(leaf_obs)
            except Empty:
                self.logger.warning(f"Worker {self.worker_id} timed out during MCTS expansion.")
                continue
            eng.expand_backup(np.asarray(lg, np.float32).reshape(1, A), np.array([v], vdt))
            sim_count += 1
        return self._decision(eng)


class MuZeroMCTS(_GumbelEngineMCTS):
    """Search with the learned dynamics network: one 'initial' request at the root, then
    'recurrent_batch' requests of len(selected_children_actions) identical rows (mcts.py:283-362)."""
    MODE = "MuZero"

    def search(self, game):
        self._drain()
        self._last = None
        A = config.ACTION_SPACE_SIZE
        obs = game.get_board_state(game.current_player, game.last_move)
        try:
            policy_logits, value, hidden = self._remote_initial_inference(obs)
        except Empty:
            self.logger.warning(f"Worker {self.worker_id} timed out on initial inference.")
            return np.zeros(A), 0.0, -1
        if not (np.asarray(game.board) == 0).any():
            return np.zeros(A), 0.0, -1
        vdt = np.float32 if isinstance(value, np.float32) else np.float64
        eng = self._engine_for_config(self._accum_of(value))
        self._load_root(eng, game)
        gumbel = np.random.gumbel(0, 1, A)
        eng.root_expand(np.asarray(policy_logits, np.float32).reshape(1, A), np.array([value], vdt), gumbel.reshape(1, A))
        hidden_of = {0: hidden}
        while True:
            parent, action, child, _depth, reps = eng.select_mz(with_reps=True)
            parent, action, child, reps = int(parent[0].item()), int(action[0].item()), int(child[0].item()), int(reps[0].item())
            if parent < 0:
                break
            results = self._remote_recurrent_inference_batch(
                np.concatenate([hidden_of[parent]] * reps, axis=0), [action] * reps)
            if not results:
                continue
            lg, v, h, r = results[-1]
            hidden_of[child] = h
            eng.expand_backup(np.asarray(lg, np.float32).reshape(1, A), np.array([results[0][1]], vdt), np.array([r], vdt))
        return self._decision(eng)
