"""SearchEngine: G concurrent Gumbel-MCTS game trees resident on one GPU.

Thin host layer over the C ABI (include/gmz.h -> libgmz.so).  PyTorch is used for device
memory, streams and the evaluator network only; every tree operation is a hand-written
sm_100a kernel.  One engine = one process = one GPU (multi-GPU = one engine per rank).

The engine replaces, for a whole batch of games at once, what the reference does per game in
Python: `AlphaZeroMCTS.search` / `MuZeroMCTS.search` (mcts.py:197-362) and the self-play
move loop around it (workers.py:162-181).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import (GMZ_ACCUM_F32, GMZ_ACCUM_F64, GMZ_BF16, GMZ_F32, GMZ_F64, GMZ_MODE_ALPHAZERO, GMZ_MODE_MUZERO, GmzConfig,
                   GmzOpenings, check)


def _ptr(t):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


class SearchEngine:
    """accum_dtype: the dtype the reference's tree arithmetic runs in, which follows the evaluator's value
    scalars (SURVEY.md App. A.7).  "float64": the evaluator hands Python floats (the upstream test mock,
    tests/test_mcts_logic.py:43).  "float32": it hands np.float32 scalars -- the reference's inference server
    (workers.py:355,368) -- so under NumPy >= 2 value_sum, the backed-up value, Q and the MinMaxStats bounds
    are float32; use this mode behind a real network to reproduce the reference's visit counts."""

    def __init__(self, num_games, board_size=15, n_in_row=5, num_simulations=400, num_top_actions=16,
                 mode="AlphaZero", c_visit=30, c_scale=1.0, minmax_delta=1e-3, discount=0.997, device=None,
                 accum_dtype="float64"):
        if not torch.cuda.is_available():
            raise _lib.GmzError("SearchEngine needs a CUDA device (there is no CPU fallback)")
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if mode not in ("AlphaZero", "MuZero"):
            raise ValueError(f"Unknown MCTS implementation in config: '{mode}'")   # workers.py:142
        self.mode = mode
        name = getattr(accum_dtype, "__name__", str(accum_dtype)).replace("torch.", "")     # "float32", np.float32, torch.float32
        acc = {"float64": GMZ_ACCUM_F64, "f64": GMZ_ACCUM_F64, "float32": GMZ_ACCUM_F32, "f32": GMZ_ACCUM_F32}.get(name)
        if acc is None:
            raise ValueError(f"accum_dtype must be 'float64' or 'float32', not {accum_dtype!r}")
        self.accum_dtype = "float32" if acc == GMZ_ACCUM_F32 else "float64"
        self.G, self.N, self.A = int(num_games), int(board_size), int(board_size) ** 2
        self.S, self.K = int(num_simulations), int(num_top_actions)
        self.cfg = GmzConfig(self.N, int(n_in_row), self.S, self.K,
                             GMZ_MODE_ALPHAZERO if mode == "AlphaZero" else GMZ_MODE_MUZERO, self.G, 0, acc,
                             float(c_visit), float(c_scale), float(minmax_delta), float(discount))
        nbytes = self.lib.gmz_workspace_bytes(C.byref(self.cfg))
        if nbytes == 0:
            raise _lib.GmzError("gmz_workspace_bytes: " + self.lib.gmz_last_error().decode())
        with torch.cuda.device(self.device):
            self.workspace = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)
            off = (-self.workspace.data_ptr()) % 256
            self._ws_ptr = self.workspace.data_ptr() + off
            handle = C.c_void_p()
            check(self.lib.gmz_create(C.byref(self.cfg), C.c_void_p(self._ws_ptr), nbytes, self._stream(),
                                      C.byref(handle)), "gmz_create")
        self.handle = handle
        self.workspace_bytes = int(nbytes)
        G, A, N = self.G, self.A, self.N
        dev = self.device
        self.leaf_obs = torch.zeros((G, 3, N, N), dtype=torch.float32, device=dev)
        self.policy = torch.zeros((G, A), dtype=torch.float64, device=dev)
        self.value = torch.zeros(G, dtype=torch.float64, device=dev)
        self.action = torch.zeros(G, dtype=torch.int32, device=dev)
        self.visits = torch.zeros((G, A), dtype=torch.int32, device=dev)
        self.winner = torch.zeros(G, dtype=torch.int32, device=dev)
        self.leaf_action = torch.zeros(G, dtype=torch.int32, device=dev)
        self.leaf_depth = torch.zeros(G, dtype=torch.int32, device=dev)
        self.launches = 0   # kernels of ours launched through this engine
        self._book = None   # device copies of the bound opening book

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.gmz_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def _dev(self, x, dtype):
        t = torch.as_tensor(x)
        if t.dtype != dtype or t.device != self.device or not t.is_contiguous():
            t = t.to(device=self.device, dtype=dtype).contiguous()
        return t

    # ------------------------------------------------------------------ roots
    def set_roots(self, boards, players, last_moves, move_counts):
        """boards int8 [G,N,N] or [G,A]; players +-1 [G]; last_moves action index or -1 [G]; move_counts [G]."""
        b = self._dev(boards, torch.int8).reshape(self.G, self.A)
        pl = self._dev(players, torch.int8).reshape(self.G)
        lm = self._dev(last_moves, torch.int32).reshape(self.G)
        mc = self._dev(move_counts, torch.int32).reshape(self.G)
        check(self.lib.gmz_set_roots(self.handle, _ptr(b), _ptr(pl), _ptr(lm), _ptr(mc), self._stream()), "gmz_set_roots")
        self.launches += 1

    def set_roots_from_records(self, ring, capacity, first, n):
        """Roots from `n` <= G packed move records of a ring (uint8 device tensor [capacity, stride]): game k takes the
        record at ring position (first + k) % capacity -- its board, and from its header the side to move, last move and
        move count; games n..G-1 become inactive.  Nothing is copied to or from the host."""
        check(self.lib.gmz_set_roots_from_records(self.handle, _ptr(ring), int(capacity), int(first), int(n), self._stream()),
              "gmz_set_roots_from_records")
        self.launches += 1

    def reset_games(self, mask=None):
        m = None if mask is None else self._dev(mask, torch.uint8).reshape(self.G)
        check(self.lib.gmz_games_reset(self.handle, _ptr(m), self._stream()), "gmz_games_reset")
        self.launches += 1

    def set_openings(self, openings):
        """Bind an opening book (arena.Openings, or any 4-tuple of boards [O,A] or [O,N,N], players, last moves, move
        counts) that every later self-play deal of this engine takes its position from: the k-th deal of game g since
        this call takes opening (k*G + g) mod O.  None unbinds (deals are empty boards again).  Games in flight continue
        unchanged.  The book is checked first (arena.check_openings, ValueError) and nothing is launched if it fails."""
        if openings is None:
            check(self.lib.gmz_set_openings(self.handle, None, self._stream()), "gmz_set_openings")
            self._book = None
            return
        from .arena import check_openings
        op = check_openings(openings, self.N, self.cfg.n_in_row)
        book = [torch.from_numpy(x).to(self.device) for x in op]
        c = GmzOpenings(op.boards.shape[0], 0, *(t.data_ptr() for t in book))
        check(self.lib.gmz_set_openings(self.handle, C.byref(c), self._stream()), "gmz_set_openings")
        self._book = book

    def get_roots(self):
        b = torch.empty((self.G, self.N, self.N), dtype=torch.int8, device=self.device)
        pl = torch.empty(self.G, dtype=torch.int8, device=self.device)
        lm = torch.empty(self.G, dtype=torch.int32, device=self.device)
        mc = torch.empty(self.G, dtype=torch.int32, device=self.device)
        check(self.lib.gmz_get_roots(self.handle, _ptr(b), _ptr(pl), _ptr(lm), _ptr(mc), self._stream()), "gmz_get_roots")
        self.launches += 1
        return b, pl, lm, mc

    def obs_buffer_bf16(self):
        """An observation buffer the kernels can fill directly in the network's input format: bfloat16, logical
        shape [G,3,N,N] with channels_last strides (memory [G,N,N,3])."""
        return torch.zeros((self.G, self.N, self.N, 3), dtype=torch.bfloat16, device=self.device).permute(0, 3, 1, 2)

    def _obs_kind(self, out):
        if out.dtype == torch.float32 and out.is_contiguous():
            return GMZ_F32
        if out.dtype == torch.bfloat16 and out.permute(0, 2, 3, 1).is_contiguous():
            return GMZ_BF16
        raise TypeError("observation buffer must be contiguous float32 [G,3,N,N] or channels_last bfloat16 [G,3,N,N]")

    def root_obs(self, out=None):
        out = self.leaf_obs if out is None else out
        check(self.lib.gmz_root_obs(self.handle, _ptr(out), self._obs_kind(out), self._stream()), "gmz_root_obs")
        self.launches += 1
        return out

    # ------------------------------------------------------------------ stepwise search
    @staticmethod
    def _vdtype(values):
        if values.dtype == torch.float64:
            return GMZ_F64
        if values.dtype == torch.float32:
            return GMZ_F32
        raise TypeError("values must be float32 or float64")

    def root_expand(self, logits, values, gumbel):
        lg = self._dev(logits, torch.float32).reshape(self.G, self.A)
        v = torch.as_tensor(values)
        v = self._dev(v, v.dtype if v.dtype in (torch.float32, torch.float64) else torch.float64).reshape(self.G)
        gm = self._dev(gumbel, torch.float64).reshape(self.G, self.A)
        check(self.lib.gmz_root_expand(self.handle, _ptr(lg), _ptr(v), self._vdtype(v), _ptr(gm), self._stream()),
              "gmz_root_expand")
        self.launches += 1

    def select(self, trace=False, out=None):
        """AlphaZero mode: returns the leaf observations [G,3,N,N] (engine-owned float32 buffer, or `out`: a float32
        NCHW or channels_last bfloat16 buffer, see obs_buffer_bf16)."""
        out = self.leaf_obs if out is None else out
        check(self.lib.gmz_select(self.handle, _ptr(out), self._obs_kind(out),
                                  _ptr(self.leaf_action) if trace else None,
                                  _ptr(self.leaf_depth) if trace else None, self._stream()), "gmz_select")
        self.launches += 1
        return out

    def select_mz(self, with_reps=False):
        """MuZero mode: (parent_slot, action, child_slot, depth[, reps]) int32 [G]; -1 where nothing to evaluate."""
        if not hasattr(self, "_mz_out"):
            self._mz_out = [torch.zeros(self.G, dtype=torch.int32, device=self.device) for _ in range(5)]
        a, b, c, d, r = self._mz_out
        check(self.lib.gmz_select_mz(self.handle, _ptr(a), _ptr(b), _ptr(c), _ptr(d), _ptr(r), self._stream()),
              "gmz_select_mz")
        self.launches += 1
        return (a, b, c, d, r) if with_reps else (a, b, c, d)

    def expand_backup(self, logits, values, rewards=None):
        lg = self._dev(logits, torch.float32).reshape(self.G, self.A)
        v = torch.as_tensor(values)
        v = self._dev(v, v.dtype if v.dtype in (torch.float32, torch.float64) else torch.float64).reshape(self.G)
        r = None if rewards is None else self._dev(rewards, v.dtype).reshape(self.G)
        check(self.lib.gmz_expand_backup(self.handle, _ptr(lg), _ptr(v), _ptr(r), self._vdtype(v), self._stream()),
              "gmz_expand_backup")
        self.launches += 1

    def finalize(self, want_visits=True):
        """Decision phase: (policy f64 [G,A], value f64 [G], action i32 [G], visits i32 [G,A])."""
        check(self.lib.gmz_finalize(self.handle, _ptr(self.policy), _ptr(self.value), _ptr(self.action),
                                    _ptr(self.visits) if want_visits else None, self._stream()), "gmz_finalize")
        self.launches += 1
        return self.policy, self.value, self.action, self.visits

    # ------------------------------------------------------------------ E0 / fused paths
    def e0_eval(self, obs, seed, logit_div=16, logits=None, values=None):
        obs = self._dev(obs, torch.float32)
        B = obs.shape[0]
        logits = torch.empty((B, self.A), dtype=torch.float32, device=self.device) if logits is None else logits
        values = torch.empty(B, dtype=torch.float64, device=self.device) if values is None else values
        check(self.lib.gmz_e0_eval_obs(_ptr(obs), B, self.N, C.c_uint64(seed & (2**64 - 1)), int(logit_div),
                                       _ptr(logits), _ptr(values), self._stream()), "gmz_e0_eval_obs")
        self.launches += 1
        return logits, values

    def search_e0(self, gumbel, seed, logit_div=16, trace=False):
        """Whole AlphaZero-mode search with the fixed evaluator in one persistent kernel."""
        gm = self._dev(gumbel, torch.float64).reshape(self.G, self.A)
        ta = td = None
        if trace:
            ta = torch.full((self.G, self.S), -1, dtype=torch.int32, device=self.device)
            td = torch.full((self.G, self.S), -1, dtype=torch.int32, device=self.device)
        check(self.lib.gmz_search_e0(self.handle, _ptr(gm), C.c_uint64(seed & (2**64 - 1)), int(logit_div),
                                     _ptr(ta), _ptr(td), self._stream()), "gmz_search_e0")
        self.launches += 1
        return ta, td

    def selfplay_e0(self, total_moves, eval_seed, logit_div=16, noise_seed=0, traj=None, restart=True):
        """Persistent self-play kernel: `total_moves` moves (search + decision + do_move + end check)
        handed out to the G games by a ticket counter; finished games restart in-kernel."""
        check(self.lib.gmz_selfplay_e0(self.handle, C.byref(traj.c) if traj is not None else None,
                                       C.c_uint64(eval_seed & (2**64 - 1)), int(logit_div),
                                       C.c_uint64(noise_seed & (2**64 - 1)), int(total_moves), int(bool(restart)),
                                       self._stream()), "gmz_selfplay_e0")
        self.launches += 1

    def selfplay_step(self, policy, value, action, traj=None, restart=True):
        """Stepwise-path move bookkeeping: record into the trajectory store, do_move, end check, restart."""
        check(self.lib.gmz_selfplay_step(self.handle, C.byref(traj.c) if traj is not None else None, _ptr(policy),
                                         _ptr(value), _ptr(action), int(bool(restart)), _ptr(self.winner), self._stream()),
              "gmz_selfplay_step")
        self.launches += 1
        return self.winner

    def play_counters(self):
        """(moves played, games finished) by the persistent kernel since the engine was created."""
        out = torch.zeros(4, dtype=torch.int64, device=self.device)
        check(self.lib.gmz_play_counters(self.handle, _ptr(out), self._stream()), "gmz_play_counters")
        m, f, unserved, idle = out.cpu().tolist()
        self.tickets_unserved, self.tickets_idle = int(unserved), int(idle)
        return int(m), int(f)

    def select_counters(self):
        """(fallbacks, certified, mismatches): interior selects handed to the exact path since the engine was
        created; the last two are only counted by -DGMZ_VERIFY_FAST builds of the library."""
        out = torch.zeros(3, dtype=torch.int64, device=self.device)
        check(self.lib.gmz_select_counters(self.handle, _ptr(out), self._stream()), "gmz_select_counters")
        return tuple(int(x) for x in out.cpu().tolist())

    def fill_gumbel(self, out, seed, offset=0):
        check(self.lib.gmz_fill_gumbel(_ptr(out), out.numel(), C.c_uint64(seed & (2**64 - 1)),
                                       C.c_uint64(offset), self._stream()), "gmz_fill_gumbel")
        self.launches += 1
        return out

    def search_stepwise_e0(self, gumbel, seed, logit_div=16, trace=False):
        """Same search through the stepwise kernels + the stand-alone E0 evaluator kernel
        (the path an external network takes).  Returns per-evaluation traces if asked."""
        obs = self.root_obs()
        lg, v = self.e0_eval(obs, seed, logit_div)
        self.root_expand(lg, v, gumbel)
        tr_a, tr_d = [], []
        for _ in range(self.S - 1):
            obs = self.select(trace=trace)
            if trace:
                tr_a.append(self.leaf_action.clone()); tr_d.append(self.leaf_depth.clone())
            self.e0_eval(obs, seed, logit_div, lg, v)
            self.expand_backup(lg, v)
        if trace:
            return torch.stack(tr_a, 1) if tr_a else None, torch.stack(tr_d, 1) if tr_d else None
        return None, None

    # ------------------------------------------------------------------ inspection
    def export_tree(self, out=None):
        """Every game's current search tree, the root's Gumbel top-k and halving rounds, as device tensors
        (searchtree.SearchTrees; one kernel on the current stream, no host read).  `out`: a previous export to refill."""
        from .searchtree import export_tree
        return export_tree(self, out)

    # ------------------------------------------------------------------ game step
    def game_step(self, actions):
        a = self._dev(actions, torch.int32).reshape(self.G)
        check(self.lib.gmz_game_step(self.handle, _ptr(a), _ptr(self.winner), self._stream()), "gmz_game_step")
        self.launches += 1
        return self.winner
