"""Search inspection: what an engine's searches hold, as device tensors.

`SearchEngine.export_tree()` copies every game's tree out of the engine's workspace with one kernel (gmz_tree_export):
node statistics as stored, the edges, the MinMax bounds, and the root's Gumbel top-k in sequential-halving order with
the round each entry was eliminated in.  `SearchTrees` then answers the questions a user asks of a search without
re-running it -- the expected line (`pv`), each root move's visits, Q, prior and Gumbel fate (`root_table`) -- for all
G games at once in torch, or for one game as numpy arrays (`game`).  This is the reference's web-UI view of a search
(webui.py /api/mcts_test) for every evaluator the engine runs, the bf16 network and learned dynamics included.

A game's tree is current from its root expansion until its root changes (set_roots, game_step, self-play, matches);
a game without one exports 0 nodes.  Node 0 is the root and node k the k-th node created.
"""
from __future__ import annotations

import ctypes as C

import torch

from ._lib import GmzTreeOut, check

# field -> (dtype, shape kind): "g" [G], "g3" [G,3], "g2" [G,2], "k" [G,K], "a" [G,A], "s" [G,S]
_FIELDS = {
    "num_nodes": (torch.int32, "g"), "sim_count": (torch.int32, "g"), "root": (torch.int32, "g3"),
    "minmax": (torch.float64, "g2"), "halving": (torch.int32, "g3"),
    "topk_action": (torch.int32, "k"), "topk_gumbel": (torch.float64, "k"), "topk_logit": (torch.float32, "k"),
    "topk_round": (torch.int32, "k"), "root_logits": (torch.float32, "a"),
    "parent": (torch.int32, "s"), "action": (torch.int32, "s"), "depth": (torch.int32, "s"), "visits": (torch.int32, "s"),
    "value_sum": (torch.float64, "s"), "reward": (torch.float64, "s"), "prior_logit": (torch.float32, "s"),
}


class SearchTrees:
    """Every game's search tree, device tensors (G games, S node slots, K top-k slots, A actions):
      per node [G,S]: parent, action (-1 for the root), depth, visits, value_sum, reward, prior_logit (the parent's
        logit at `action`, NaN for the root); entries past num_nodes are -1 / 0;
      per game: num_nodes, sim_count, to_move, last_move, move_count [G]; minmax [G,2] = (minimum, maximum);
        phase, n_surv, n_init [G]; topk_action, topk_gumbel, topk_logit, topk_round [G,K] (halving order: survivors
        first; topk_round = the round that eliminated the entry, `phase` for survivors, -1 past n_init);
        root_logits [G,A].
    `discount` and `accum_dtype` are the engine's."""

    def __init__(self, tensors, discount, accum_dtype, A):
        self.__dict__.update(tensors)
        self.discount, self.accum_dtype, self.A = float(discount), accum_dtype, int(A)
        self.G, self.S = self.parent.shape

    @property
    def to_move(self):
        return self.root[:, 0]

    @property
    def last_move(self):
        return self.root[:, 1]

    @property
    def move_count(self):
        return self.root[:, 2]

    @property
    def phase(self):
        return self.halving[:, 0]

    @property
    def n_surv(self):
        return self.halving[:, 1]

    @property
    def n_init(self):
        return self.halving[:, 2]

    def _exists(self):
        return torch.arange(self.S, device=self.parent.device)[None, :] < self.num_nodes[:, None]

    def q(self):
        """[G,S] the reference's get_qsa of each node's edge, reward + discount * value_sum / visits (mcts.py:32-38), in
        the engine's accumulation dtype; float32 mode computes every operation in float32 as Node.get_value / get_qsa do
        on np.float32 values.  NaN for the root, unvisited nodes and entries past num_nodes."""
        ok = self._exists() & (self.parent >= 0) & (self.visits > 0)
        n = self.visits.clamp(min=1)
        if self.accum_dtype == "float32":
            disc = torch.tensor(self.discount, dtype=torch.float32, device=self.parent.device)
            q = self.reward.float() + disc * (self.value_sum.float() / n.float())
        else:
            q = self.reward + self.discount * (self.value_sum / n.double())
        return torch.where(ok, q, torch.full_like(q, float("nan")))

    def _best_child(self):
        """[G,S] node id of each node's most-visited child (ties: lowest action), -1 for nodes without children."""
        G, S, A = self.G, self.S, self.A
        child = self._exists() & (self.parent >= 0)
        key = torch.where(child, self.visits.long() * (A + 1) + (A - self.action.long()), torch.full_like(self.visits, -1, dtype=torch.long))
        par = torch.where(child, self.parent.long(), torch.zeros_like(self.parent, dtype=torch.long))
        best = torch.full((G, S), -1, dtype=torch.long, device=key.device).scatter_reduce(1, par, key, "amax", include_self=True)
        win = child & (key == best.gather(1, par))
        ids = torch.arange(S, device=key.device).expand(G, S)
        out = torch.full((G, S), -1, dtype=torch.long, device=key.device)
        return out.scatter_reduce(1, torch.where(win, par, torch.zeros_like(par)), torch.where(win, ids, torch.full_like(ids, -1)),
                                  "amax", include_self=True)

    def _root_children(self):
        """[G,A] node id of each root action's child, -1 where there is none."""
        G, S, A = self.G, self.S, self.A
        rc = self._exists() & (self.parent == 0)
        a = torch.where(rc, self.action.long(), torch.zeros_like(self.action, dtype=torch.long))
        ids = torch.arange(S, device=a.device).expand(G, S)
        out = torch.full((G, A), -1, dtype=torch.long, device=a.device)
        return out.scatter_reduce(1, a, torch.where(rc, ids, torch.full_like(ids, -1)), "amax", include_self=True)

    def pv(self, first=None, max_depth=None):
        """Principal variation: (actions int32, visits int32, q) [G,D], -1 / -1 / NaN past its end.  Ply 0 is `first`
        (int32 [G], e.g. finalize's action; -1 = none) or, with first=None, the most-visited root child (lowest action
        among ties -- the decision's move unless its maximum is tied); every later ply the most-visited child, lowest
        action among ties.  D = max_depth, or the deepest tree's depth (one device-to-host read)."""
        dev = self.parent.device
        if max_depth is None:
            max_depth = int((torch.where(self._exists(), self.depth, torch.zeros_like(self.depth))).max().item()) if self.S else 0
        D = max(1, int(max_depth))
        gi = torch.arange(self.G, device=dev)
        best = self._best_child()
        q = self.q()
        if first is None:
            node = best[:, 0]
            act0 = torch.where(node >= 0, self.action.long().gather(1, node.clamp(min=0)[:, None])[:, 0], torch.full_like(node, -1))
        else:
            act0 = torch.as_tensor(first, device=dev).long().reshape(self.G)
            valid = (act0 >= 0) & (act0 < self.A) & (self.num_nodes > 0)
            node = torch.where(valid, self._root_children()[gi, act0.clamp(0, self.A - 1)], torch.full_like(act0, -1))
            act0 = torch.where(valid, act0, torch.full_like(act0, -1))
        acts = torch.full((self.G, D), -1, dtype=torch.int32, device=dev)
        vis = torch.full((self.G, D), -1, dtype=torch.int32, device=dev)
        qs = torch.full((self.G, D), float("nan"), dtype=q.dtype, device=dev)
        acts[:, 0] = act0.int()
        has = node >= 0
        nc = node.clamp(min=0)
        vis[:, 0] = torch.where(act0 >= 0, torch.where(has, self.visits[gi, nc], torch.zeros_like(self.visits[gi, nc])), vis[:, 0])
        qs[:, 0] = torch.where(has, q[gi, nc], qs[:, 0])
        for d in range(1, D):
            node = torch.where(has, best[gi, nc], torch.full_like(node, -1))
            has = node >= 0
            nc = node.clamp(min=0)
            acts[:, d] = torch.where(has, self.action[gi, nc], acts[:, d])
            vis[:, d] = torch.where(has, self.visits[gi, nc], vis[:, d])
            qs[:, d] = torch.where(has, q[gi, nc], qs[:, d])
        return acts, vis, qs

    def root_table(self):
        """Per root action [G,A]: prior_logit, visits, q (NaN if unvisited), topk_rank (position in the initial Gumbel
        top-k, -1 if not in it), gumbel (NaN if not in the top-k), eliminated_in (-1 if not in the top-k, `phase` for
        survivors).  A dict of device tensors."""
        G, A, K = self.G, self.A, self.topk_action.shape[1]
        dev = self.parent.device
        gi = torch.arange(G, device=dev)[:, None]
        rc = self._root_children()
        has = rc >= 0
        rcc = rc.clamp(min=0)
        visits = torch.where(has, self.visits.gather(1, rcc), torch.zeros_like(rc, dtype=torch.int32))
        q = self.q().gather(1, rcc)
        q = torch.where(has & (visits > 0), q, torch.full_like(q, float("nan")))
        ink = self.topk_action >= 0
        ka = torch.where(ink, self.topk_action.long(), torch.full_like(self.topk_action, A, dtype=torch.long))   # A = a spill column
        rank = torch.full((G, A + 1), -1, dtype=torch.int32, device=dev)
        rank[gi, ka] = torch.arange(K, dtype=torch.int32, device=dev).expand(G, K)
        gum = torch.full((G, A + 1), float("nan"), dtype=torch.float64, device=dev)
        gum[gi, ka] = self.topk_gumbel
        elim = torch.full((G, A + 1), -1, dtype=torch.int32, device=dev)
        elim[gi, ka] = self.topk_round
        return dict(prior_logit=self.root_logits, visits=visits, q=q, topk_rank=rank[:, :A], gumbel=gum[:, :A],
                    eliminated_in=elim[:, :A])

    def game(self, g, first=None):
        """Game g's tree as host numpy arrays: the per-node arrays cut to num_nodes, the per-game fields, the root table,
        q, and the principal variation (`pv_actions`, `pv_visits`, `pv_q`, cut at its end) started from `first` (an int
        action, or None for the most-visited root child)."""
        g = int(g)
        n = int(self.num_nodes[g].item())
        out = {f: getattr(self, f)[g, :n].cpu().numpy() for f in
               ("parent", "action", "depth", "visits", "value_sum", "reward", "prior_logit")}
        out["q"] = self.q()[g, :n].cpu().numpy()
        k = int(self.n_init[g].item())
        for f in ("topk_action", "topk_gumbel", "topk_logit", "topk_round"):
            out[f] = getattr(self, f)[g, :k].cpu().numpy()
        for f in ("num_nodes", "sim_count", "to_move", "last_move", "move_count", "phase", "n_surv", "n_init"):
            out[f] = int(getattr(self, f)[g].item())
        out["minmax"] = self.minmax[g].cpu().numpy()
        sub = self._one(g)
        out["root"] = {f: t[0].cpu().numpy() for f, t in sub.root_table().items()}
        fa = None if first is None else torch.tensor([int(first)], dtype=torch.int32, device=self.parent.device)
        a, v, q = (t[0].cpu().numpy() for t in sub.pv(fa))
        end = int((a >= 0).sum())
        out["pv_actions"], out["pv_visits"], out["pv_q"] = a[:end], v[:end], q[:end]
        return out

    def _one(self, g):
        return SearchTrees({f: getattr(self, f)[g:g + 1] for f in _FIELDS}, self.discount, self.accum_dtype, self.A)

    @classmethod
    def from_tensors(cls, tensors, discount, accum_dtype, A):
        """A SearchTrees over given tensors (any device), e.g. a hand-built tree: every key of the export's fields."""
        missing = set(_FIELDS) - set(tensors)
        if missing:
            raise ValueError(f"missing fields: {sorted(missing)}")
        return cls(dict(tensors), discount, accum_dtype, A)


def export_tree(engine, out: SearchTrees | None = None) -> SearchTrees:
    """Copy every game's tree out of `engine` (one gmz_tree_export on the current stream, no host read).  `out`: a
    SearchTrees of this engine to refill instead of allocating new tensors."""
    G, S, K, A = engine.G, engine.S, engine.K, engine.A
    shapes = {"g": (G,), "g2": (G, 2), "g3": (G, 3), "k": (G, K), "a": (G, A), "s": (G, S)}
    if out is None:
        t = {f: torch.empty(shapes[kind], dtype=dt, device=engine.device) for f, (dt, kind) in _FIELDS.items()}
        out = SearchTrees(t, engine.cfg.discount, engine.accum_dtype, A)
    c = GmzTreeOut(*[getattr(out, f).data_ptr() for f, _ in GmzTreeOut._fields_])
    check(engine.lib.gmz_tree_export(engine.handle, C.byref(c), engine._stream()), "gmz_tree_export")
    engine.launches += 1
    return out
