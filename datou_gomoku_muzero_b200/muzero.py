"""Device-resident MuZero-mode search (reference MuZeroMCTS.search, mcts.py:288-362) for G games.

The tree lives in the engine (gmz_select_mz / gmz_expand_backup); hidden states live in a pool on the
device, one row per tree node, addressed by the slots the select kernel emits -- the reference instead
pickles every hidden state through two mp.Queue hops per batch (mcts.py:77-85, workers.py:357-369).
One loop iteration = one of the reference's batches: the len(survivors) identical selections are
deduplicated to one evaluation, the kernel applies that many backups (SURVEY App. A.6).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from ._lib import check
from .network import GomokuNetEZ, GraphStepSearch, _fold, _fold_heads, _support_scalar

_M64 = (1 << 64) - 1


def evals_per_search(num_simulations, num_top_actions, n_survivors):
    """Number of recurrent evaluations one search performs when the initial survivor list has
    `n_survivors` entries: the halving state machine of mcts.py:158-181 driven with sim_count += k."""
    S, K = int(num_simulations), int(num_top_actions)
    lg2 = np.log2(K) if K > 1 else 0.0
    nxt = S if (K <= 1 or lg2 <= 0) else int(min(np.floor(S / (lg2 * K)) * K, S))
    m, used, sims, k, evals = K, 0.0, 1, int(n_survivors), 0
    while sims < S and k > 0:
        sims += k
        evals += 1
        if sims >= nxt:
            m //= 2
            if m >= 1:
                extra = (S - used) if (m <= 1 or lg2 <= 0) else np.floor(S / (lg2 * m)) * m
                used += extra
                nxt = min(nxt + int(extra), S)
                k = min(m, k)
    return evals


class MuZeroDeviceSearch(GraphStepSearch):
    """initial_fn(obs f32 [G,3,N,N]) -> (logits f32 [G,A], values [G], hidden [G, ...])
    recurrent_fn(hidden [G, ...], actions int64 [G]) -> (logits, values, rewards [G], next_hidden [G, ...])
    Hidden rows may be any dtype / shape (4-byte multiples); the pool is allocated from the first
    initial_fn result.  A 4-D hidden state [G,C,N,N] is stored NHWC (one row = N*N cells x C channels), so
    the gathered batch is a channels_last tensor without a copy.

    Pool layouts: by default game g owns rows g*nodes_per_game .. g*nodes_per_game + nodes_per_game - 1.  A search given
    per-game budgets (`budget`, re-analysis) uses one compact arena instead: game g owns rows base[g] .. base[g] + rows[g] - 1,
    base the exclusive prefix sum of the budgets; a node at or beyond its game's budget is not stored (skip slot) and is counted
    in `overflow` (int64 device scalar).  `nodes_per_game` then caps the budget a game may ask for.

    One simulation step = gmz_select_mz -> gmz_hidden_gather -> recurrent_fn -> gmz_hidden_scatter ->
    gmz_expand_backup, all on the device.  If recurrent_fn has `embed` ([E] action-embedding vector) and
    `forward_fused(x)` (x = [G, C+E, N, N] channels_last: hidden state and one-hot action embedding already
    concatenated, network.py:70-73), the gather writes that concatenated input directly.  With `graph=True`
    the step is captured in a CUDA graph after `graph_warmup` eager steps and replayed from then on."""

    def __init__(self, engine, initial_fn, recurrent_fn, nodes_per_game=None, graph=False, graph_warmup=3):
        if engine.mode != "MuZero":
            raise ValueError("MuZeroDeviceSearch needs an engine created with mode='MuZero'")
        super().__init__(engine, graph, graph_warmup)
        self.initial_fn, self.recurrent_fn = initial_fn, recurrent_fn
        self.nodes = int(nodes_per_game) if nodes_per_game else engine.S
        self.pool = None
        self.evaluations = 0
        self.fused = hasattr(recurrent_fn, "forward_fused") and getattr(recurrent_fn, "embed", None) is not None
        self._root_slot = (torch.arange(engine.G, dtype=torch.int32, device=engine.device) * engine.S).contiguous()
        self.arena = False                              # pool layout: g * nodes + node (False) or base[g] + node (True)
        self._budget = torch.zeros(engine.G, dtype=torch.int32, device=engine.device)
        self._base = torch.zeros(engine.G, dtype=torch.int32, device=engine.device)
        self.overflow = torch.zeros((), dtype=torch.int64, device=engine.device)

    def set_recurrent_fn(self, recurrent_fn):
        """Swap the dynamics evaluator (e.g. after a model update that built a new FoldedRecurrentInference): the
        captured CUDA graph holds the old one's weight pointers, so it is dropped and re-captured on the next search.
        (FoldedRecurrentInference.update_weights refreshes the weights in place instead and needs no re-capture.)"""
        self.recurrent_fn = recurrent_fn
        self.fused = hasattr(recurrent_fn, "forward_fused") and getattr(recurrent_fn, "embed", None) is not None
        self.graph = None
        if self.pool is not None:                       # same hidden-state shape assumed: keep the pool, refresh the embedding
            had = self.embed is not None
            if self.fused and len(self.hshape) == 3:
                self.embed = recurrent_fn.embed.detach().to(self.pool.dtype).to(self.pool.device).contiguous()
            else:
                self.embed = None
            if had != (self.embed is not None):
                self.pool = None                        # the gathered batch changes width: start over

    # ---- pool layout
    @staticmethod
    def _rows(h):
        """hidden [G, ...] -> [G, row] view in pool order (NHWC for 4-D), copying only if the layout differs."""
        if h.dim() == 4:
            return h.permute(0, 2, 3, 1).contiguous().reshape(h.shape[0], -1)
        return h.contiguous().reshape(h.shape[0], -1)

    def _ensure_pool(self, hidden, arena_rows=None):
        e = self.e
        rows = self._rows(hidden)
        arena = arena_rows is not None
        shape = (int(arena_rows) if arena else e.G * self.nodes, rows.shape[1])
        if arena and self.pool is not None and self.arena and self.pool.shape[0] >= shape[0]:
            shape = tuple(self.pool.shape)              # the arena only grows
        if self.pool is None or self.pool.shape != shape or self.pool.dtype != hidden.dtype or self.arena != arena:
            self.pool = None                            # free the old pool first
            self.pool = torch.empty(shape, dtype=hidden.dtype, device=hidden.device)
            self.arena = arena
            self.hshape = tuple(hidden.shape[1:])
            self.row_bytes = rows.shape[1] * hidden.element_size()
            if self.row_bytes % 4:
                raise ValueError("hidden-state rows must be a multiple of 4 bytes")
            if hidden.dim() == 4:
                C_, n1, n2 = self.hshape
                self.positions, self.pos_bytes = n1 * n2, C_ * hidden.element_size()
            else:
                self.positions, self.pos_bytes = 1, self.row_bytes
            self.embed = None
            if self.fused and hidden.dim() == 4:
                self.embed = self.recurrent_fn.embed.detach().to(hidden.dtype).to(hidden.device).contiguous()
            E = 0 if self.embed is None else self.embed.numel()
            self.embed_bytes = E * hidden.element_size()
            per_pos = (self.pos_bytes + self.embed_bytes) // hidden.element_size()
            self.x = torch.zeros((e.G, self.positions * per_pos), dtype=hidden.dtype, device=hidden.device)
            self.graph = None
        return rows

    def _gather(self, slot, action):
        e = self.e
        S, nodes = (1, 1) if self.arena else (e.S, self.nodes)         # arena: slots are already pool rows
        check(e.lib.gmz_hidden_gather(self.pool.data_ptr(), slot.data_ptr(), action.data_ptr(), e.G, S, nodes,
                                      self.positions, self.pos_bytes,
                                      None if self.embed is None else self.embed.data_ptr(), self.embed_bytes,
                                      self.x.data_ptr(), e._stream()), "gmz_hidden_gather")
        e.launches += 1

    def _scatter(self, slot, rows):
        e = self.e
        if rows.dtype != self.pool.dtype or rows.shape[1] != self.pool.shape[1]:
            raise ValueError("recurrent_fn returned a hidden state of a different dtype / shape than initial_fn")
        S, nodes = (1, 1) if self.arena else (e.S, self.nodes)
        check(e.lib.gmz_hidden_scatter(self.pool.data_ptr(), slot.data_ptr(), e.G, S, nodes, self.row_bytes,
                                       rows.data_ptr(), e._stream()), "gmz_hidden_scatter")
        e.launches += 1

    def _x_view(self):
        """The gathered batch in the shape recurrent_fn expects."""
        e = self.e
        if len(self.hshape) == 3:
            C_, n1, n2 = self.hshape
            E = 0 if self.embed is None else self.embed.numel()
            return self.x.view(e.G, n1, n2, C_ + E).permute(0, 3, 1, 2)           # channels_last [G, C+E, N, N]
        return self.x.view((e.G,) + self.hshape)

    def _arena_row(self, slot, count=False):
        """Engine slot g*S + node -> arena row base[g] + node, or -1 (skip) for node >= rows[g]; with `count`, such nodes
        are added to `overflow`.  Device tensor ops only (captured with the step)."""
        node = slot - self._root_slot
        live = slot >= 0
        ok = live & (node < self._budget)
        if count:
            self.overflow.add_((live & ~ok).sum())
        return torch.where(ok, self._base + node, -1).to(torch.int32)

    def _step(self):
        e = self.e
        parent, action, child, depth = e.select_mz()
        if self.arena:
            parent, child = self._arena_row(parent), self._arena_row(child, count=True)
        self._gather(parent, action)
        if self.embed is not None:
            lg, v, r, h_out = self.recurrent_fn.forward_fused(self._x_view())
        else:
            lg, v, r, h_out = self.recurrent_fn(self._x_view(), action.long().clamp_min(0))
        self._scatter(child, self._rows(h_out))
        e.expand_backup(lg, v, r)

    def budget_table(self):
        """Tree nodes a search can create, by the number of root survivors k = min(K, empty cells) = 0..K: the root plus
        one node per recurrent evaluation (int64 numpy [K+1])."""
        e = self.e
        return np.array([evals_per_search(e.S, e.K, k) + 1 for k in range(e.K + 1)], dtype=np.int64)

    def host_budgets(self, boards):
        """Per-game node budgets (int32 [G]) for roots given as host boards int8 [G, A]: the root plus one node per
        recurrent evaluation, for k = min(K, empty cells) root survivors (ValueError if one exceeds nodes_per_game)."""
        k = np.minimum((np.asarray(boards) == 0).sum(axis=1), self.e.K)
        rows = self.budget_table()[k].astype(np.int32)
        self.check_budget(int(rows.max()))
        return rows

    def check_budget(self, most_rows):
        if most_rows > self.nodes:
            raise ValueError(f"the MuZeroDeviceSearch holds {self.nodes} tree nodes per game (nodes_per_game); a root here "
                             f"needs {most_rows}")

    @torch.no_grad()
    def search(self, gumbel, budget=None, max_steps=None):
        """Runs one search for every game from the engine's current roots; call engine.finalize() after.

        budget = (rows, arena_rows, steps): rows (int32 device tensor [G]) / arena_rows (host int >= rows.sum()) are per-game
        node budgets in one compact arena of at least `arena_rows` rows (grown, and the graph re-captured, only when that is
        more than the arena has).  The search then runs exactly `steps` steps (the largest evaluation count of the batch)
        and reads nothing back to the host; steps after a game has finished evaluate nothing for it.  Without a budget,
        `max_steps` (if given and non-zero) caps the number of steps."""
        e = self.e
        rows, arena_rows = None, None
        if budget is not None:
            rows, arena_rows, max_steps = budget
        arena = rows is not None
        lg, v, h = self.initial_fn(e.root_obs())
        pool_rows = self._ensure_pool(h, arena_rows if arena else None)
        root = self._root_slot
        if arena:
            self._budget.copy_(rows)
            torch.cumsum(self._budget, 0, dtype=torch.int32, out=self._base)
            self._base.sub_(self._budget)
            root = self._arena_row(root, count=True)
        self._scatter(root, pool_rows)
        e.root_expand(lg, v, gumbel)
        steps, limit = 0, int(max_steps) if max_steps is not None and (arena or max_steps) else e.S - 1   # at most S-1 evaluations
        while steps < limit:
            if not arena and steps + 2 > self.nodes:          # this step may create node id steps + 1
                raise RuntimeError("hidden-state pool too small: pass a larger nodes_per_game")
            self._advance(steps)
            steps += 1
            self.evaluations += 1
            if not arena and steps % 8 == 0 and steps < limit and int(e._mz_out[0].max().item()) < 0:   # every game is done
                self.evaluations -= 1           # the last step evaluated nothing
                steps -= 1
                break
        return steps


class TorchE0:
    """The fixed evaluator E0 in MuZero mode, as torch integer ops on the device (hidden state = the
    64-bit hash, one int64 per node).  Same integers as the CUDA E0 (csrc/gmz_common.cuh) and
    tests/golden/e0_py.py; logit_div = 0 selects the dense (unquantised) heads."""

    GOLD, CV, CA = 0x9E3779B97F4A7C15, 0xD1B54A32D192ED03, 0x8CB92BA72F3D8DD7
    K1, K2 = 0xBF58476D1CE4E5B9, 0x94D049BB133111EB
    GOLD32, M1 = 0x9E3779B1, 0x7FEB352D

    def __init__(self, board_size, seed=0, logit_div=16, device="cuda"):
        self.N, self.A = board_size, board_size * board_size
        self.seed, self.div, self.device = int(seed), int(logit_div), device
        self.a1 = self._c((np.arange(1, self.A + 1, dtype=np.int64) * self.GOLD32) & 0xFFFFFFFF)     # (a + 1) * GOLD32 mod 2^32
        self.h0 = self._s(self.mix_int(self.seed ^ self.GOLD))

    def _c(self, x):
        return torch.as_tensor(x, dtype=torch.int64, device=self.device)

    @staticmethod
    def _s(v):          # python int (unsigned 64) -> signed int64 value
        v &= _M64
        return v - (1 << 64) if v >= (1 << 63) else v

    @staticmethod
    def _shr(z, k):     # logical right shift on int64
        return (z >> k) & ((1 << (64 - k)) - 1)

    def mix(self, z):
        z = z ^ self._shr(z, 30)
        z = z * self._s(self.K1)
        z = z ^ self._shr(z, 27)
        z = z * self._s(self.K2)
        return z ^ self._shr(z, 31)

    def heads(self, h, with_reward=False):
        m32 = 0xFFFFFFFF
        s = (h & m32) ^ self._shr(h, 32)                           # 32-bit arithmetic carried in int64 lanes
        x = (s[:, None] + self.a1[None, :]) & m32
        x = x ^ (x >> 16)
        x = (x * self.M1) & m32
        vk = self._shr(h, 40) & 0xFFFFFF
        rk = self._shr(h, 16) & 0xFFFFFF
        if self.div > 0:
            logits = ((x >> 26) - 32).to(torch.float32) / float(self.div)
            value = ((vk % 33) - 16).to(torch.float64) / 16.0
            reward = ((rk % 5) - 2).to(torch.float64) / 16.0
        else:
            logits = ((x >> 8) - (1 << 23)).to(torch.float32) * (2.0 ** -21)
            value = (vk - (1 << 23)).to(torch.float64) * (2.0 ** -23)
            reward = (rk - (1 << 23)).to(torch.float64) * (2.0 ** -25)
        return (logits, value, reward) if with_reward else (logits, value)

    def initial(self, obs):
        B, A = obs.shape[0], self.A
        nw = (A + 63) // 64
        planes = (obs.reshape(B, 3, A) > 0.5)
        weights = torch.zeros((nw, A), dtype=torch.int64, device=obs.device)
        idx = torch.arange(A, device=obs.device)
        bit = torch.ones(A, dtype=torch.int64, device=obs.device) << (idx % 64)      # bit 63 wraps to the sign bit
        weights[idx // 64, idx] = bit
        own = (planes[:, 0, None, :].long() * weights[None]).sum(-1)                # disjoint bits: sum == or
        opp = (planes[:, 1, None, :].long() * weights[None]).sum(-1)
        has_last = planes[:, 2].any(dim=1)
        last = torch.where(has_last, planes[:, 2].float().argmax(dim=1), torch.full((B,), -1, device=obs.device))
        acc = torch.zeros((B,), dtype=torch.int64, device=obs.device)
        for w in range(nw):
            acc = acc ^ (((own[:, w] ^ self.h0) + self._s((2 * w + 1) * self.GOLD)) * self._s(self.K1))
            b = ((opp[:, w] ^ self.h0) + self._s((2 * w + 2) * self.GOLD)) * self._s(self.K2)
            acc = acc ^ ((b << 32) | self._shr(b, 32))
        h = self.mix(acc + (last + 1) * self._s(self.CV))
        lg, v = self.heads(h)
        return lg, v, h

    @staticmethod
    def mix_int(z):
        z &= _M64
        z ^= z >> 30; z = (z * 0xBF58476D1CE4E5B9) & _M64
        z ^= z >> 27; z = (z * 0x94D049BB133111EB) & _M64
        return z ^ (z >> 31)

    def recurrent(self, h_parent, actions):
        hc = self.mix(h_parent + (actions + 1) * self._s(self.CA))
        lg, v, r = self.heads(hc, with_reward=True)
        return lg, v, r, hc


class FoldedRecurrentInference:
    """`recurrent_inference` (network.py:145-152) for the engine: BatchNorm folded, cuDNN fused
    conv+bias(+residual)+ReLU, channels_last bf16 hidden states, reward head weights permuted to the
    NHWC flatten order so the [B, C*N*N] view of the hidden state is free.  Library kernels."""

    def __init__(self, net: GomokuNetEZ, dtype=torch.bfloat16):
        self.dtype = dtype
        self.fused = True
        self._fold_from(net)
        self.v_sup, self.r_sup = net.v_sup, net.r_sup
        self.n = net.board_size
        try:        # the fused cuDNN entry points do not cover every dtype / build: fall back to conv2d + relu
            dev = self.stem[0].device
            self._cr(torch.zeros((1, self.stem[0].shape[1], self.n, self.n), dtype=dtype, device=dev)
                     .contiguous(memory_format=torch.channels_last), self.stem, 1)
        except RuntimeError:
            self.fused = False

    def _tensors(self):
        return [self.stem, *sum(([a, b] for a, b in self.blocks), []), self.r1, self.r2, self.pv, self.policy_fc,
                self.value_fc1, self.value_fc2]

    def update_weights(self, net: GomokuNetEZ):
        """Refold from `net` (fp32 weights) INTO the existing tensors, so a CUDA graph captured over this object
        (MuZeroDeviceSearch) keeps replaying against the same buffers -- the MuZero-mode counterpart of
        DeviceEvaluator.update_weights (ModelWeightsUpdate, workers.py:331-335)."""
        old = self._tensors(); old_embed = self.embed
        self._fold_from(net)
        new = self._tensors()
        with torch.no_grad():
            for (ow, ob), (nw, nb) in zip(old, new):
                ow.copy_(nw); ob.copy_(nb)
            old_embed.copy_(self.embed)
        self.embed = old_embed
        (self.stem, *rest) = old
        nb = len(self.blocks)
        self.blocks = [(rest[2 * i], rest[2 * i + 1]) for i in range(nb)]
        self.r1, self.r2, self.pv, self.policy_fc, self.value_fc1, self.value_fc2 = rest[2 * nb:]

    def _fold_from(self, net):
        d, p = net.dynamics_net, net.prediction_net
        dtype = self.dtype
        self.embed = d.action_embed_conv.weight.detach().to(dtype).reshape(-1).clone()           # [16]
        self.stem = _fold(d.conv, d.bn, dtype)
        self.blocks = [(_fold(b.conv1, b.bn1, dtype), _fold(b.conv2, b.bn2, dtype)) for b in d.resblocks]
        n, C = net.board_size, d.conv.out_channels
        w1 = d.reward_fc[0].weight.detach()                                                # [hid, C*n*n] in CHW order
        self.r1 = (w1.reshape(-1, C, n, n).permute(0, 2, 3, 1).reshape(w1.shape[0], -1).to(dtype).contiguous(), None)
        own = lambda t: t.detach().to(dtype).clone()      # never alias the module's parameters (update_weights writes in place)
        self.r1 = (self.r1[0], own(d.reward_fc[0].bias))
        self.r2 = (own(d.reward_fc[2].weight), own(d.reward_fc[2].bias))
        self.pv = _fold_heads(p, dtype)
        self.policy_fc = (own(p.policy_fc.weight), own(p.policy_fc.bias))
        self.value_fc1 = (own(p.value_fc1.weight), own(p.value_fc1.bias))
        self.value_fc2 = (own(p.value_fc2.weight), own(p.value_fc2.bias))

    def _cr(self, x, wb, pad):
        if self.fused:
            return torch.cudnn_convolution_relu(x, wb[0], wb[1], (1, 1), (pad, pad), (1, 1), 1)
        return F.relu(F.conv2d(x, wb[0], wb[1], padding=pad))

    def _car(self, x, wb, z):
        if self.fused:
            return torch.cudnn_convolution_add_relu(x, wb[0], z, 1.0, wb[1], (1, 1), (1, 1), (1, 1), 1)
        return F.relu(F.conv2d(x, wb[0], wb[1], padding=1) + z)

    @torch.no_grad()
    def __call__(self, hidden, actions):
        B, n = hidden.shape[0], self.n
        plane = F.one_hot(actions, n * n).to(self.dtype).reshape(B, 1, n, n)
        emb = plane * self.embed.reshape(1, -1, 1, 1)                                      # 1x1 conv of a one-hot plane
        return self.forward_fused(torch.cat((hidden, emb), dim=1).contiguous(memory_format=torch.channels_last))

    @torch.no_grad()
    def forward_fused(self, x):
        """x [B, C+16, n, n] channels_last: hidden state and action embedding already concatenated
        (what gmz_hidden_gather writes)."""
        B = x.shape[0]
        h = self._cr(x, self.stem, 1)
        for c1, c2 in self.blocks:
            h = self._car(self._cr(h, c1, 1), c2, h)
        flat = h.permute(0, 2, 3, 1).reshape(B, -1)
        rew = _support_scalar(F.linear(F.relu(F.linear(flat, *self.r1)), *self.r2).float(), *self.r_sup)
        pv = self._cr(h, self.pv, 0)
        pl, vl = pv[:, :2].reshape(B, -1), pv[:, 2].reshape(B, -1)
        logits = F.linear(pl, *self.policy_fc).float()
        value = _support_scalar(F.linear(F.relu(F.linear(vl, *self.value_fc1)), *self.value_fc2).float(), *self.v_sup)
        return logits.contiguous(), value.reshape(-1), rew.reshape(-1), h
