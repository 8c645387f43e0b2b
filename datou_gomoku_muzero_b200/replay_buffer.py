"""Prioritized replay with the SumTree resident on the GPU, API-compatible with the reference's
replay_buffer.py (SumTree :4-41, InMemoryReplayBuffer :43-106).  Sampling and priority updates are
CUDA kernels (csrc/gmz_per.cu) that keep the reference's sequential float64 semantics bit for bit.

Two buffers:
  * `InMemoryReplayBuffer` -- the reference's class: slices are host objects in `self.data` exactly as in
    the reference, only the tree lives on the device.
  * `DeviceReplayBuffer` -- the same ring + tree with the DATA on the device too: a ring of packed move
    records (csrc/gmz_records.cu) written by the self-play engine's trajectory hand-off.  `sample()` returns
    the trainer's batch tuple (workers.py:430-433) as device tensors; nothing touches the host between a
    finished game and a training batch.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check
from .config import config
from .trajectory import record_dtype


def _ptr(t):
    return C.c_void_p(t.data_ptr())


class SumTree:
    def __init__(self, capacity: int, device=None):
        if not torch.cuda.is_available():
            raise _lib.GmzError("SumTree needs a CUDA device (there is no CPU fallback)")
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.capacity = int(capacity)
        self.tree = torch.zeros(2 * self.capacity - 1, dtype=torch.float64, device=self.device)
        self.write_ptr = 0
        self.count = 0

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, x, dtype):
        """numpy / list / tensor -> contiguous device tensor of `dtype` (no copy if it already is one)."""
        if not torch.is_tensor(x):
            x = torch.as_tensor(np.ascontiguousarray(x))
        return x.to(device=self.device, dtype=dtype).contiguous()

    # ---- device-tensor entry points (no host round trip)
    def update_many(self, tree_idx, priorities):
        """Apply tree.update(idx_i, p_i) for i = 0..n-1 in order (replay_buffer.py:16-19)."""
        idx, pr = self._dev(tree_idx, torch.int64), self._dev(priorities, torch.float64)
        check(self.lib.gmz_per_update(_ptr(self.tree), self.capacity, _ptr(idx), _ptr(pr), int(idx.numel()),
                                      self._stream()), "gmz_per_update")

    def update(self, tree_idx, priority):
        self.update_many([int(tree_idx)], [float(priority)])

    def add_many(self, priorities):
        pr = self._dev(priorities, torch.float64)
        n = int(pr.numel())
        if n == 0:
            return
        scratch = torch.empty(n, dtype=torch.int64, device=self.device)
        check(self.lib.gmz_per_add(_ptr(self.tree), self.capacity, self.write_ptr, _ptr(pr), n, _ptr(scratch),
                                   self._stream()), "gmz_per_add")
        self.write_ptr = (self.write_ptr + n) % self.capacity
        self.count = min(self.capacity, self.count + n)

    def add(self, priority):
        self.add_many([float(priority)])

    def sample_device(self, u01, beta):
        """Stratified draw on the device: (tree_idx int64 [B], priority f64 [B], is_weights f32 [B]) device tensors."""
        u = self._dev(u01, torch.float64)
        B = int(u.numel())
        idx = torch.empty(B, dtype=torch.int64, device=self.device)
        pr = torch.empty(B, dtype=torch.float64, device=self.device)
        w = torch.empty(B, dtype=torch.float32, device=self.device)
        check(self.lib.gmz_per_sample(_ptr(self.tree), self.capacity, self.count, _ptr(u), B, float(beta),
                                      _ptr(idx), _ptr(pr), _ptr(w), self._stream()), "gmz_per_sample")
        return idx, pr, w

    def sample(self, u01, beta):
        """Host-facing form of sample_device (numpy results)."""
        idx, pr, w = self.sample_device(u01, beta)
        return idx.cpu().numpy(), pr.cpu().numpy(), w.cpu().numpy()

    def get_leaf(self, value):
        """SumTree.get_leaf (replay_buffer.py:27-38): the descent runs as tensor ops on the device, one
        synchronisation at the end (not one per level)."""
        tree, n = self.tree, self.tree.numel()
        parent = torch.zeros((), dtype=torch.int64, device=self.device)
        v = torch.tensor(float(value), dtype=torch.float64, device=self.device)
        levels = 0
        while (1 << levels) - 1 < n:        # deepest possible leaf level
            levels += 1
        for _ in range(levels):
            left = 2 * parent + 1
            inner = left < n
            lv = tree[left.clamp(max=n - 1)]
            go_left = v <= lv
            nxt = torch.where(go_left, left, left + 1)
            v = torch.where(inner & ~go_left, v - lv, v)
            parent = torch.where(inner, nxt, parent)
        return int(parent.item())

    def total_priority(self):
        return float(self.tree[0])


class InMemoryReplayBuffer:
    def __init__(self, capacity, device=None):
        self.capacity = capacity
        self.sum_tree = SumTree(capacity, device)
        self.data = [None] * capacity
        self.max_priority = 1.0

    def add(self, training_slice):
        self.data[self.sum_tree.write_ptr] = training_slice
        self.sum_tree.add(self.max_priority if config.ENABLE_PER else 1.0)

    def add_many(self, slices):
        """Batch form of add(): one kernel for the whole game's slices (workers.py:399-407 adds them in a loop)."""
        p = self.max_priority if config.ENABLE_PER else 1.0
        wp = self.sum_tree.write_ptr
        for i, s in enumerate(slices):
            self.data[(wp + i) % self.capacity] = s
        self.sum_tree.add_many([p] * len(slices))

    def sample(self, batch_size):
        if self.sum_tree.count < batch_size:
            return None, None, None
        if config.ENABLE_PER:
            u = np.random.random_sample(batch_size)      # the doubles np.random.uniform would consume
            idx, _, w = self.sum_tree.sample(u, config.PER_BETA)
            batch = [self.data[int(i) - self.capacity + 1] for i in idx]
            return batch, [int(i) for i in idx], w
        indices = np.random.choice(self.sum_tree.count, batch_size, replace=False)
        return [self.data[i] for i in indices], indices, np.ones(batch_size, dtype=np.float32)

    def update_priorities(self, tree_indices, td_errors):
        if not config.ENABLE_PER:
            return
        priorities = np.abs(td_errors) + config.PER_EPSILON      # keeps td_errors' dtype (float32 from the loss)
        if len(priorities) == 0:
            return
        self.max_priority = max(self.max_priority, priorities.max())
        self.sum_tree.update_many(np.asarray(tree_indices, dtype=np.int64), priorities.astype(np.float64))

    def __len__(self):
        return self.sum_tree.count


RING_STATE_FORMAT, RING_STATE_VERSION = "gmz_device_replay_ring", 1


def validate_ring_state(sd, board_size):
    """Host-side check of a DeviceReplayBuffer.state_dict() before anything of it goes to the device; raises ValueError
    naming the first thing that does not fit.  Checks the tag and version, the board size, every shape and dtype, count
    and write_ptr against the saved capacity, the tree length, the base boards' stone values and the header t chain:
    segments start exactly at k = 0 and wherever t = 0, t grows by 1 and length stays put inside a segment, 0 <= t <
    length, and every segment ends at its game's last move (games are appended whole)."""
    if not isinstance(sd, dict):
        raise ValueError("ring state must be a dict (DeviceReplayBuffer.state_dict())")
    if sd.get("format") != RING_STATE_FORMAT or sd.get("version") != RING_STATE_VERSION:
        raise ValueError(f"unknown ring state format {sd.get('format')!r} version {sd.get('version')!r} "
                         f"(expected {RING_STATE_FORMAT!r} version {RING_STATE_VERSION})")
    for key in ("board_size", "capacity", "count", "write_ptr"):
        if not isinstance(sd.get(key), int) or isinstance(sd.get(key), bool):
            raise ValueError(f"ring state {key} must be an int")
    N, cap, n, wp = sd["board_size"], sd["capacity"], sd["count"], sd["write_ptr"]
    if N != int(board_size):
        raise ValueError(f"ring state board size {N} differs from the buffer's {int(board_size)}")
    A = N * N
    if cap < 1:
        raise ValueError(f"ring state capacity {cap} must be >= 1")
    if not 0 <= n <= cap:
        raise ValueError(f"ring state count {n} outside 0..capacity ({cap})")
    if not 0 <= wp < cap or (n < cap and wp != n):
        raise ValueError(f"ring state write_ptr {wp} outside the saved ring (capacity {cap}, count {n})")

    def tensor(key, dtype, shape):
        t = sd.get(key)
        if not torch.is_tensor(t) or t.device.type != "cpu" or t.dtype != dtype or tuple(t.shape) != shape:
            got = f"{t.dtype} {tuple(t.shape)} on {t.device}" if torch.is_tensor(t) else type(t).__name__
            raise ValueError(f"ring state {key} must be a CPU {dtype} tensor of shape {shape}, got {got}")
        return t
    seg = sd.get("seg_start")
    n_seg = int(seg.shape[0]) if torch.is_tensor(seg) and seg.dim() == 1 else -1
    headers = tensor("headers", torch.uint8, (n, 64))
    tensor("policies", torch.float64, (n, A))
    seg = tensor("seg_start", torch.int64, (max(n_seg, 0),))
    base = tensor("base_boards", torch.int8, (max(n_seg, 0), A))
    tensor("tree", torch.float64, (2 * cap - 1,))
    tensor("max_priority", torch.float64, ())
    if base.numel() and (base.min() < -1 or base.max() > 1):
        raise ValueError("ring state base_boards hold a value outside {-1, 0, 1}")
    h = headers.numpy().view(np.int32)                  # gmz_move_record: game_seq, t, length, ...
    t, T = h[:, 1].astype(np.int64), h[:, 2].astype(np.int64)
    k = np.arange(n)
    starts = (k == 0) | (t == 0)
    if not np.array_equal(seg.numpy(), np.flatnonzero(starts)):
        raise ValueError("ring state seg_start does not match the header t chain (segments start at k = 0 and where t = 0)")
    if n and not ((t >= 0) & (t < T)).all():
        raise ValueError(f"ring state header t outside 0..length-1 at record {int(np.flatnonzero((t < 0) | (t >= T))[0])}")
    inner = ~starts[1:]
    broken = inner & ((t[1:] != t[:-1] + 1) | (T[1:] != T[:-1]))
    if broken.any():
        raise ValueError(f"ring state header t chain broken inside a segment at record {int(np.flatnonzero(broken)[0]) + 1}")
    ends = np.append(starts[1:], True) if n else starts
    if n and (t[ends] != T[ends] - 1).any():
        raise ValueError("ring state holds a game cut before its last move")
    return n_seg


class DeviceReplayBuffer:
    """The reference's InMemoryReplayBuffer (replay_buffer.py:43-106) with tree AND data on the device.

    data ring : `capacity` packed move records (include/gmz.h gmz_move_record); record i is the TrainingSlice the
                reference would have stored at data[i] -- a slice is that record plus the next U of the same game, which
                follow it in the ring (games are appended whole, in move order; a ring overwrites oldest first, so the
                successors of a live record are live).
    add_packed(games)  = `for s in slices: buffer.add(s)` for every game of a trajectory.PackedGames (workers.py:399-407)
    sample(B)          -> ((obs, act, rew, pi, val), tree_indices, is_weights), all device tensors: the tuple
                          data_loader_worker stacks (workers.py:430-433); rot_k / flip apply the trainer's D4
                          augmentation while gathering (loss.py:37-51)
    update_priorities  = replay_buffer.py:98-103 on device tensors (td_errors float32, as the loss returns them)
    rewrite_targets    = the re-analysis write-back (db_manager.py:189-214) for records in the ring
    reanalyse(engines) = Surge re-analysis (workers.py:243-305) of the records in the ring, in place, on the device
    state_dict() / load_state_dict(sd) = checkpoint and restore of ring, tree, write_ptr, count and max_priority in a
                          compact form (headers, policies, one board per segment), rebuilt on the device
    """

    def __init__(self, capacity, board_size, device=None, unroll_steps=None):
        self.sum_tree = SumTree(capacity, device)
        self.capacity, self.N, self.A = int(capacity), int(board_size), int(board_size) ** 2
        self.device, self.lib = self.sum_tree.device, self.sum_tree.lib
        self.stride = int(self.lib.gmz_move_record_bytes(self.N))
        # byte range of each record field within a ring row (policy, board, header scalars, ...)
        self._field = {name: slice(off, off + dt.itemsize) for name, (dt, off) in record_dtype(self.N).fields.items()}
        self.ring = torch.zeros((self.capacity, self.stride), dtype=torch.uint8, device=self.device)
        self.max_priority = torch.ones((), dtype=torch.float64, device=self.device)
        self.unroll = int(config.NUM_UNROLL_STEPS if unroll_steps is None else unroll_steps)

    def add_packed(self, games):
        rec = games.records
        if rec.device != self.device:
            rec = rec.to(self.device)
        total = int(rec.shape[0])
        for s0 in range(0, total, self.capacity):        # more records than the ring holds: wrap exactly like sequential add()s
            part = rec[s0:s0 + self.capacity]
            M = int(part.shape[0])
            wp = self.sum_tree.write_ptr
            first = min(M, self.capacity - wp)
            self.ring[wp:wp + first].copy_(part[:first])
            if first < M:
                self.ring[:M - first].copy_(part[first:])
            pr = (self.max_priority if config.ENABLE_PER else torch.ones_like(self.max_priority)).expand(M)
            self.sum_tree.add_many(pr)

    def sample(self, batch_size, u01=None, rot_k=0, flip=False):
        if self.sum_tree.count < batch_size:
            return None, None, None
        B = int(batch_size)
        if config.ENABLE_PER:
            u = torch.rand(B, dtype=torch.float64, device=self.device) if u01 is None else u01
            idx, _, w = self.sum_tree.sample_device(u, config.PER_BETA)
            pos = idx - (self.capacity - 1)
        else:
            pos = torch.randperm(self.sum_tree.count, device=self.device)[:B]
            idx, w = pos, torch.ones(B, dtype=torch.float32, device=self.device)
        return self.batch(pos, rot_k, flip), idx, w

    def batch(self, positions, rot_k=0, flip=False):
        """Trainer tuple for the slices stored at ring `positions` (int64 device tensor)."""
        pos = self.sum_tree._dev(positions, torch.int64)
        B, U, N, A, dev = int(pos.numel()), self.unroll, self.N, self.A, self.device
        obs = torch.empty((B, U + 1, 3, N, N), dtype=torch.float32, device=dev)
        act = torch.empty((B, U), dtype=torch.int32, device=dev)
        rew = torch.empty((B, U), dtype=torch.float32, device=dev)
        pi = torch.empty((B, U + 1, A), dtype=torch.float64, device=dev)
        val = torch.empty((B, U + 1), dtype=torch.float32, device=dev)
        check(self.lib.gmz_records_batch(_ptr(self.ring), self.capacity, N, _ptr(pos), B, U, int(rot_k) % 4, 1 if flip else 0,
                                         _ptr(obs), _ptr(act), _ptr(rew), _ptr(pi), _ptr(val), self.sum_tree._stream()),
              "gmz_records_batch")
        return obs, act, rew, pi, val

    def rewrite_targets(self, positions, policies, value_targets):
        """Re-analysis write-back (db_manager.py:189-214) for records resident in the ring: the policy and the value
        target of the move stored at each ring position are replaced; every slice that covers the move -- slices are
        assembled from consecutive records when a batch is built -- then carries the new window.  positions int64 [M],
        policies float64 [M, A], value_targets float32 [M] (host or device)."""
        pos = self.sum_tree._dev(positions, torch.int64).reshape(-1)
        pol = self.sum_tree._dev(policies, torch.float64).reshape(pos.numel(), self.A).contiguous()
        val = self.sum_tree._dev(value_targets, torch.float32).reshape(pos.numel()).contiguous()
        if pos.numel() == 0:
            return
        if int(pos.min()) < 0 or int(pos.max()) >= self.capacity:
            raise ValueError("ring position out of range")
        self.ring[pos, self._field["policy"]] = pol.view(torch.uint8).reshape(pos.numel(), 8 * self.A)
        self.ring[pos, self._field["value_target"]] = val.view(torch.uint8).reshape(pos.numel(), 4)

    def reanalyse(self, engines, first=None, count=None, evaluator="e0", eval_seed=0, logit_div=16, noise_seed=0):
        """Surge re-analysis (workers.py:243-305) of the records in the ring, in place: every position is searched again
        with the latest evaluator, its policy and root search value are replaced, and the n-step value targets of the
        stretch are recomputed from the new root values (re-analysis arithmetic: float32 rewards, workers.py:291-292).
        Observations, boards, actions, rewards and the PER tree are left as they are.

        Which records: by default every live record, oldest first.  An explicit stretch (`first` = a ring position,
        `count` records; either may be omitted: from the oldest live record / up to the newest) is widened to whole
        games, as far as those games are still live -- the reference re-analyses whole GameRecords.  A stretch that
        reaches outside the live records raises ValueError.  Returns the widened (first, count).

        engines: SearchEngines of the buffer's board size.  The stretch goes through them G records per batch, batches
        alternating between the engines, each on a stream of its own; the caller's current stream waits for all of them
        and then runs the target recomputation, so later add_packed / batch / sample calls see the new bytes.  Loading the
        roots overwrites an engine's games: do not pass the engine that is running self-play.
        evaluator: whatever SelfPlayEngine takes, resolved to one searcher per engine by mcts.resolve_searchers -- "e0"
        (the fixed evaluator, either engine mode; eval_seed / logit_div as SearchEngine.search_e0); a callable
        f(obs f32 [G,3,N,N]) -> (logits, values) (eager, AlphaZero mode); a GomokuNetEZ module (a bf16 NetworkSearch per
        engine, AlphaZero mode); a pair (initial_fn, recurrent_fn) (a MuZeroDeviceSearch(graph=True) per engine, MuZero
        mode); or a list of already-built NetworkSearch / MuZeroDeviceSearch objects, one bound to each engine, which keep
        their captured graphs from call to call.  Anything else raises ValueError before any kernel is enqueued.
        Noise is drawn on the device: record k of the widened stretch uses Gumbel counters k*A .. k*A + A-1 of
        `noise_seed`, as reanalyse_positions gives its position k.

        MuZero searchers keep hidden states in a compact arena: a record with k = min(K, empty cells) root survivors gets
        the root plus muzero.evals_per_search(S, K, k) rows, so the arena holds what the batch can use, not G * S rows.
        One device pass over the stretch counts the empty cells; one small read brings every batch's row total and step
        count to the host before any search is enqueued (ValueError, nothing touched, if a searcher's nodes_per_game is
        below a record's budget), and each batch then runs its exact step count without reading anything back.

        Policies and values never go to the host; the only host reads are that budget read (MuZero searchers) and the two
        boundary headers of an explicit stretch."""
        from .mcts import check_budget, resolve_searchers, search_roots
        from .muzero import MuZeroDeviceSearch
        engines = list(engines)
        if isinstance(evaluator, str) and evaluator != "e0":
            raise ValueError(f"unknown evaluator {evaluator!r}")
        if not engines:
            raise ValueError("reanalyse needs at least one engine")
        for e in engines:
            if e.N != self.N:
                raise ValueError(f"engine board size {e.N} differs from the buffer's {self.N}")
            if e.device != self.device:
                raise ValueError(f"engine on {e.device}, buffer on {self.device}")
        searchers = resolve_searchers(engines, evaluator)
        cap, live = self.capacity, self.sum_tree.count
        oldest = self.sum_tree.write_ptr if live == cap else 0
        if first is not None and not 0 <= int(first) < cap:
            raise ValueError(f"first={first} is not a ring position (capacity {cap})")
        rel = 0 if first is None else (int(first) - oldest) % cap          # offset from the oldest live record
        n = live - rel if count is None else int(count)
        if (first is not None and rel >= live) or n < 0 or rel + n > live:
            raise ValueError(f"stretch first={first}, count={count} reaches outside the {live} live records")
        if n > 0 and (first is not None or count is not None):
            ends = torch.tensor([(oldest + rel) % cap, (oldest + rel + n - 1) % cap], device=self.device)
            h = torch.cat([self.ring[ends, self._field["t"]], self.ring[ends, self._field["length"]]], 1)
            h = h.cpu().numpy().view(np.int32)                             # (t, length) of both ends
            end = rel + n + int(h[1, 1]) - 1 - int(h[1, 0])
            rel = max(0, rel - int(h[0, 0]))                               # a cut oldest game: its live suffix
            if end > live:
                raise RuntimeError("ring records do not hold whole games")
            n = end - rel
        start = (oldest + rel) % cap
        if n == 0:
            return start, 0
        batches, s0 = [], 0                                   # (engine, first record of the stretch, records)
        while s0 < n:
            i = len(batches) % len(engines)
            batches.append((i, s0, min(engines[i].G, n - s0)))
            s0 += batches[-1][2]
        budgets = self._mz_budgets(start, n, batches, engines, searchers) \
            if any(isinstance(x, MuZeroDeviceSearch) for x in searchers) else None
        if budgets is not None:
            rows, total, steps = budgets
            for b, (i, _, _) in enumerate(batches):
                if isinstance(searchers[i], MuZeroDeviceSearch):
                    check_budget(searchers[i], steps[b] + 1)
            arena = [max((total[b] for b, x in enumerate(batches) if x[0] == i), default=0) for i in range(len(engines))]
        cur = torch.cuda.current_stream(self.device)
        streams = [torch.cuda.Stream(device=self.device) for _ in engines]
        gumbel = [torch.empty((e.G, self.A), dtype=torch.float64, device=self.device) for e in engines]
        for s in streams:
            s.wait_stream(cur)
        for b, (i, s0, k) in enumerate(batches):
            e = engines[i]
            pos = (start + s0) % cap
            with torch.cuda.stream(streams[i]):
                e.set_roots_from_records(self.ring, cap, pos, k)
                e.fill_gumbel(gumbel[i], noise_seed, s0 * self.A)
                budget = None
                if isinstance(searchers[i], MuZeroDeviceSearch):      # padding games: inactive roots, one row each
                    budget = (rows[s0:s0 + k] if k == e.G else torch.cat((rows[s0:s0 + k], rows.new_ones(e.G - k))),
                              arena[i], steps[b])
                search_roots(e, gumbel[i], searchers[i], eval_seed, logit_div, budget)
                pol, val, _, _ = e.finalize(want_visits=False)
                check(self.lib.gmz_records_writeback(_ptr(self.ring), cap, self.N, pos, k, _ptr(pol), _ptr(val), e._stream()),
                      "gmz_records_writeback")
        for s in streams:
            cur.wait_stream(s)
        dpow = torch.tensor([config.DISCOUNT ** i for i in range(config.N_STEPS + 1)], dtype=torch.float64).pin_memory()
        dpow = dpow.to(self.device, non_blocking=True)      # no host synchronisation
        check(self.lib.gmz_records_retarget(_ptr(self.ring), cap, self.N, start, n, _ptr(dpow), int(config.N_STEPS),
                                            self.sum_tree._stream()), "gmz_records_retarget")
        return start, n

    def _mz_budgets(self, start, n, batches, engines, searchers):
        """Per-record node budgets of a re-analysis stretch for MuZeroDeviceSearch engines (others: 1), from each record's
        empty-cell count on the device.  Returns (rows int32 device [n], per-batch arena rows incl. one per padding game,
        per-batch step counts) -- the two lists from one device-to-host copy."""
        from .muzero import MuZeroDeviceSearch
        dev, m = self.device, len(engines)
        K = max(e.K for e in engines)
        table = np.ones((m, K + 1), np.int32)                 # [engine, k] -> rows; clamped to each engine's own K below
        kmax = np.array([e.K for e in engines], np.int64)
        for i, x in enumerate(searchers):
            if isinstance(x, MuZeroDeviceSearch):
                t = x.budget_table()
                table[i] = t[np.minimum(np.arange(K + 1), engines[i].K)]
        first = np.array([s0 for _, s0, _ in batches], np.int64)
        host = torch.from_numpy(np.concatenate([first, kmax, table.reshape(-1).astype(np.int64)])).pin_memory()
        dv = host.to(dev, non_blocking=True)
        nb = len(batches)
        d_first, d_kmax, d_table = dv[:nb], dv[nb:nb + m], dv[nb + m:].reshape(m, K + 1)
        idx = (start + torch.arange(n, device=dev)) % self.capacity
        empty = (self.ring[idx, self._field["board"]] == 0).sum(1)
        batch = torch.searchsorted(d_first, torch.arange(n, device=dev), right=True) - 1
        eng = batch % m
        rows = d_table[eng, torch.minimum(empty, d_kmax[eng])]
        out = torch.zeros((2, nb), dtype=torch.int64, device=dev)
        out[0].scatter_add_(0, batch, rows)
        out[1].scatter_reduce_(0, batch, rows - 1, "amax")
        total, steps = out.cpu().tolist()                     # the one host read
        total = [t + engines[i].G - k for t, (i, _, k) in zip(total, batches)]
        return rows.to(torch.int32), total, steps

    def update_priorities(self, tree_indices, td_errors):
        if not config.ENABLE_PER:
            return
        td = self.sum_tree._dev(td_errors, torch.float32)
        if td.numel() == 0:
            return
        pr = (td.abs() + np.float32(config.PER_EPSILON)).double()        # float32 arithmetic like the reference, then widened
        self.max_priority = torch.maximum(self.max_priority, pr.max())
        self.sum_tree.update_many(tree_indices, pr)

    def state_dict(self):
        """The buffer's state as a dict of CPU tensors, ints and strs, for torch.save next to the network (loads with
        torch.load(weights_only=True)).  Records are kept in compact form, oldest first: headers u8 [count, 64] and
        policies f64 [count, A] verbatim, plus seg_start int64 [n_seg] (the first record of each segment: the oldest live
        record and every game start) and base_boards int8 [n_seg, A] (their boards).  Boards and observation planes of
        the other records are rebuilt by load_state_dict.  tree, write_ptr, count and max_priority are saved verbatim.

        Runs on the current stream after any pending add_packed / reanalyse / update_priorities and synchronises with
        the host (the result is host memory).  Extra device memory: the compact size of the live records.  Raises
        ValueError, leaving the buffer as it is, if a live record's board or observation planes are not what its
        predecessor and header imply (gmz_records_compact bit 1: such a record cannot be rebuilt)."""
        cap, n, wp, A, dev = self.capacity, self.sum_tree.count, self.sum_tree.write_ptr, self.A, self.device
        oldest = wp if n == cap else 0
        headers = torch.empty((n, 64), dtype=torch.uint8, device=dev)
        policies = torch.empty((n, A), dtype=torch.float64, device=dev)
        seg = torch.empty(0, dtype=torch.int64, device=dev)
        if n > 0:
            flags = torch.empty(n, dtype=torch.uint8, device=dev)
            check(self.lib.gmz_records_compact(_ptr(self.ring), cap, self.N, oldest, n, _ptr(headers), _ptr(policies),
                                               _ptr(flags), self.sum_tree._stream()), "gmz_records_compact")
            bad = (flags & 2) != 0
            n_bad, k_bad = (int(x) for x in torch.stack([bad.sum(), bad.int().argmax()]).cpu())
            if n_bad:
                raise ValueError(f"{n_bad} live ring records cannot be rebuilt from their predecessor and header (board or "
                                 f"observation planes altered); the first is at ring position {(oldest + k_bad) % cap}")
            seg = (flags & 1).nonzero().reshape(-1)
        base = self.ring[(oldest + seg) % cap, self._field["board"]].view(torch.int8)
        return {"format": RING_STATE_FORMAT, "version": RING_STATE_VERSION, "board_size": self.N, "capacity": cap,
                "count": n, "write_ptr": wp, "headers": headers.cpu(), "policies": policies.cpu(), "seg_start": seg.cpu(),
                "base_boards": base.cpu(), "tree": self.sum_tree.tree.cpu(), "max_priority": self.max_priority.cpu()}

    def load_state_dict(self, sd):
        """Restore a state_dict() (validated on the host first: validate_ring_state; ValueError before any device work).

        Same capacity: the state bit for bit -- record k of the saved order at ring position (oldest + k) % capacity, tree,
        write_ptr, count and max_priority verbatim (ring positions holding no live record are zeroed, as in a new buffer;
        the tail padding of each record is zero).  Later sample / batch / add_packed / reanalyse calls behave as on the
        saved buffer.
        Different capacity: the newest min(count, capacity) records, oldest first, at positions 0.. (a cut may fall inside
        the oldest kept game), write_ptr and count to match, and the tree rebuilt by SumTree.add_many from the kept
        records' saved leaf priorities in order -- equal to sequential add()s of them, not bit-equal to the old internal
        sums.  max_priority is kept.
        Value targets are restored as saved, whatever config.N_STEPS / DISCOUNT say now."""
        n_seg = validate_ring_state(sd, self.N)
        cap, dev, st = self.capacity, self.device, self.sum_tree
        scap, n, swp = sd["capacity"], sd["count"], sd["write_ptr"]
        kept = min(n, cap)
        skip = n - kept
        if kept > 0:
            headers, policies, seg, base = (sd[key].to(dev).contiguous() for key in ("headers", "policies", "seg_start", "base_boards"))
            first = (swp if n == cap else 0) if scap == cap else 0
            check(self.lib.gmz_records_expand(_ptr(headers), _ptr(policies), n, _ptr(seg), _ptr(base), n_seg, skip, self.N,
                                              _ptr(self.ring), cap, first, st._stream()), "gmz_records_expand")
        if kept < cap:
            self.ring[kept:].zero_()
        if scap == cap:
            st.tree.copy_(sd["tree"])
            st.write_ptr, st.count = swp, n
        else:
            soldest = swp if n == scap else 0
            leaf = (soldest + torch.arange(skip, n, dtype=torch.int64)) % scap + (scap - 1)
            st.tree.zero_()
            st.write_ptr, st.count = 0, 0
            st.add_many(sd["tree"][leaf])
        self.max_priority = sd["max_priority"].to(dev)

    def __len__(self):
        return self.sum_tree.count
