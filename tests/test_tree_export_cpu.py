"""Search inspection without a GPU: the oracle search that keeps its whole tree (tests/_tree_oracle.py, the unchanged
oracle with orc_search's driver loop restated) is the same search as oracle.search and the reference goldens, and SearchTrees' principal variation, Q and root table -- torch over all games
at once -- equal a plain recursive restatement on hand-built trees (ties, an empty tree, a lone root) and oracle trees."""
import math

import numpy as np
import pytest
import torch

from _golden_util import load_search_cases
from _tree_oracle import search_tree
from oracle import oracle as O


def _cfg(c):
    return O.make_config(board_size=c["N"], n_in_row=c["n_in_row"], num_simulations=c["S"], num_top_actions=c["K"],
                         mode=0 if c["mode"] == "az" else 1, eval_kind=c["kind"], logit_div=c["logit_div"],
                         c_visit=c["c_visit"], c_scale=c["c_scale"], minmax_delta=c["delta"], discount=c["discount"],
                         const_value=c["const_value"], const_reward=c["const_reward"], eval_seed=c["seed"],
                         accum_dtype=c["vdtype"])


def _check_structure(t, tag, mz):
    n = t["num_nodes"]
    par, act, dep, vis = t["parent"], t["node_action"], t["depth"], t["node_visits"]
    assert par[0] == -1 and act[0] == -1 and dep[0] == 0 and math.isnan(t["prior_logit"][0]), tag
    assert (par[1:] < np.arange(1, n)).all() and (par[1:] >= 0).all(), tag            # parents precede children
    assert np.array_equal(dep[1:], dep[par[1:]] + 1), tag
    child_sum = np.zeros(n, np.int64)
    np.add.at(child_sum, par[1:], vis[1:])
    own = vis - child_sum                                                              # backups received as a new leaf
    assert own[0] == 1 and (own[1:] >= 1).all() and (mz or (own[1:] == 1).all()), tag
    assert vis[0] == t["sim_count"], tag
    assert t["n_surv"] <= t["n_init"] and len(set(t["topk_action"].tolist())) == t["n_init"], tag
    assert (t["topk_round"][:t["n_surv"]] == t["phase"]).all(), tag
    assert (np.diff(t["topk_round"][t["n_surv"]:]) <= 0).all(), tag                   # later rounds sit nearer the front


@pytest.mark.parametrize("mode", ["az", "mz"])
@pytest.mark.parametrize("N", [6, 9, 15, 19])
def test_search_tree_is_the_search(mode, N):
    """search_tree runs the very search oracle.search runs (pinned to the reference goldens) and reports its tree."""
    for c in load_search_cases(mode, N):
        cfg = _cfg(c)
        tag = f"{mode} N={N} case {c['idx']}"
        t = search_tree(cfg, c["board"], c["player"], c["last_move"], c["move_count"], c["gumbel"])
        r = O.search(cfg, c["board"], c["player"], c["last_move"], c["move_count"], c["gumbel"], trace=True)
        assert np.array_equal(t["visits"], c["visits"]) and t["action"] == c["action"] and t["value"] == c["value"], tag
        assert np.array_equal(t["policy"], r["policy"]), tag
        assert np.array_equal(t["leaf_actions"], r["leaf_actions"]) and np.array_equal(t["leaf_depths"], r["leaf_depths"]), tag
        assert t["num_nodes"] == r["n_nodes"] and t["sim_count"] == r["sim_count"], tag
        assert t["minmax"].tobytes() == r["minmax"].tobytes(), tag
        assert t["node_visits"][0] == c["root_n"] and t["value_sum"][0] == c["root_w"], tag
        assert t["depth"].max() == r["max_depth"], tag
        root_kids = t["parent"] == 0
        vis = np.zeros(N * N, np.int64)
        vis[t["node_action"][root_kids]] = t["node_visits"][root_kids]
        assert np.array_equal(vis, c["visits"]), tag
        _check_structure(t, tag, mode == "mz")


# ---------------------------------------------------------------------------------------------------------------------
# SearchTrees on CPU tensors against a plain restatement

def _trees(games, S, K, A, discount=0.997, accum="float64"):
    """A SearchTrees over G hand-described games: dicts of per-node lists (parent, action, visits, value_sum, reward,
    prior_logit), root_logits [A] and top-k lists (topk_action, topk_gumbel, topk_round)."""
    from datou_gomoku_muzero_b200.searchtree import SearchTrees
    G = len(games)
    t = dict(num_nodes=torch.zeros(G, dtype=torch.int32), sim_count=torch.zeros(G, dtype=torch.int32),
             root=torch.zeros((G, 3), dtype=torch.int32), minmax=torch.zeros((G, 2), dtype=torch.float64),
             halving=torch.zeros((G, 3), dtype=torch.int32),
             topk_action=torch.full((G, K), -1, dtype=torch.int32), topk_gumbel=torch.zeros((G, K), dtype=torch.float64),
             topk_logit=torch.zeros((G, K), dtype=torch.float32), topk_round=torch.full((G, K), -1, dtype=torch.int32),
             root_logits=torch.full((G, A), float("nan"), dtype=torch.float32),
             parent=torch.full((G, S), -1, dtype=torch.int32), action=torch.full((G, S), -1, dtype=torch.int32),
             depth=torch.full((G, S), -1, dtype=torch.int32), visits=torch.full((G, S), -1, dtype=torch.int32),
             value_sum=torch.zeros((G, S), dtype=torch.float64), reward=torch.zeros((G, S), dtype=torch.float64),
             prior_logit=torch.zeros((G, S), dtype=torch.float32))
    for g, d in enumerate(games):
        n = len(d["parent"])
        t["num_nodes"][g] = n
        t["sim_count"][g] = d["visits"][0] if n else 0
        for f in ("parent", "action", "visits", "value_sum", "reward", "prior_logit"):
            if n:
                t[f][g, :n] = torch.tensor(d[f], dtype=t[f].dtype)
        dep = []
        for k in range(n):
            dep.append(0 if d["parent"][k] < 0 else dep[d["parent"][k]] + 1)
        if n:
            t["depth"][g, :n] = torch.tensor(dep, dtype=torch.int32)
            t["root_logits"][g] = torch.tensor(d["root_logits"], dtype=torch.float32)
        k = len(d.get("topk_action", []))
        t["halving"][g] = torch.tensor([d.get("phase", 0), d.get("n_surv", 0), k], dtype=torch.int32)
        if k:
            t["topk_action"][g, :k] = torch.tensor(d["topk_action"], dtype=torch.int32)
            t["topk_gumbel"][g, :k] = torch.tensor(d["topk_gumbel"], dtype=torch.float64)
            t["topk_round"][g, :k] = torch.tensor(d["topk_round"], dtype=torch.int32)
    return SearchTrees.from_tensors(t, discount, accum, A)


def _ref_q(d, k, discount, accum):
    if d["parent"][k] < 0 or d["visits"][k] <= 0:
        return float("nan")
    if accum == "float32":
        f = np.float32
        return float(f(d["reward"][k]) + f(discount) * (f(d["value_sum"][k]) / f(d["visits"][k])))
    return d["reward"][k] + discount * (d["value_sum"][k] / d["visits"][k])


def _ref_pv(d, first, discount, accum):
    """(actions, visits, q) of the principal variation, recursively: the most-visited child, lowest action among ties."""
    n = len(d["parent"])
    kids = {k: [c for c in range(1, n) if d["parent"][c] == k] for k in range(n)}

    def best(k):
        return max(kids[k], key=lambda c: (d["visits"][c], -d["action"][c])) if kids.get(k) else None

    def line(k):
        return [] if k is None else [(d["action"][k], d["visits"][k], _ref_q(d, k, discount, accum))] + line(best(k))

    if n == 0:
        return []
    if first is None:
        return line(best(0))
    node = next((c for c in kids[0] if d["action"][c] == first), None)
    if node is None:
        return [(first, 0, float("nan"))]
    return line(node)


def _ref_path(d, k):
    return [] if d["parent"][k] < 0 else _ref_path(d, d["parent"][k]) + [d["action"][k]]


def _ref_root_table(d, A, discount, accum):
    n = len(d["parent"])
    tab = dict(visits=[0] * A, q=[float("nan")] * A, topk_rank=[-1] * A, gumbel=[float("nan")] * A, eliminated_in=[-1] * A)
    for c in range(1, n):
        if d["parent"][c] == 0:
            tab["visits"][d["action"][c]] = d["visits"][c]
            tab["q"][d["action"][c]] = _ref_q(d, c, discount, accum)
    for i, a in enumerate(d.get("topk_action", [])):
        tab["topk_rank"][a] = i
        tab["gumbel"][a] = d["topk_gumbel"][i]
        tab["eliminated_in"][a] = d["topk_round"][i]
    return tab


def _same(x, y):
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    return x.shape == y.shape and np.array_equal(np.isnan(x), np.isnan(y)) and np.array_equal(x[~np.isnan(x)], y[~np.isnan(y)])


def _check_against_ref(games, S, K, A, discount, accum, firsts):
    trees = _trees(games, S, K, A, discount, accum)
    q = trees.q()
    assert q.dtype == (torch.float32 if accum == "float32" else torch.float64)
    for g, d in enumerate(games):
        n = len(d["parent"])
        assert _same(q[g, :n].numpy(), [_ref_q(d, k, discount, accum) for k in range(n)]), g
        assert torch.isnan(q[g, n:]).all()
    D = max([0] + [len(_ref_pv(d, None, discount, accum)) for d in games]) + 2
    for first in (None, firsts):
        f = None if first is None else torch.tensor(first, dtype=torch.int32)
        acts, vis, qs = trees.pv(f, max_depth=D)
        assert acts.shape == (len(games), D)
        for g, d in enumerate(games):
            ref = _ref_pv(d, None if first is None else first[g], discount, accum)
            m = len(ref)
            assert acts[g, :m].tolist() == [r[0] for r in ref] and (acts[g, m:] == -1).all(), (g, first)
            assert vis[g, :m].tolist() == [r[1] for r in ref] and (vis[g, m:] == -1).all(), (g, first)
            assert _same(qs[g, :m].numpy(), [r[2] for r in ref]) and torch.isnan(qs[g, m:]).all(), (g, first)
    a_auto, _, _ = trees.pv()                            # default length: the deepest node's depth
    depth = [max([0] + [len(_ref_path(d, k)) for k in range(len(d["parent"]))]) for d in games]
    assert a_auto.shape[1] == max(1, max(depth))
    tab = trees.root_table()
    for g, d in enumerate(games):
        ref = _ref_root_table(d, A, discount, accum)
        for f in ("visits", "topk_rank", "eliminated_in"):
            assert tab[f][g].tolist() == ref[f], (g, f)
        assert _same(tab["q"][g].numpy(), ref["q"]) and _same(tab["gumbel"][g].numpy(), ref["gumbel"]), g
        if len(d["parent"]):
            assert tab["prior_logit"][g].tolist() == torch.tensor(d["root_logits"], dtype=torch.float32).tolist()
    for g, d in enumerate(games):
        one = trees.game(g, first=None if firsts[g] < 0 else firsts[g])
        ref = _ref_pv(d, None if firsts[g] < 0 else firsts[g], discount, accum)
        assert one["pv_actions"].tolist() == [r[0] for r in ref] and one["num_nodes"] == len(d["parent"]), g
        assert one["parent"].tolist() == list(d["parent"]), g


def _hand_games(A):
    lg = [0.25 * (a % 5) - 0.5 for a in range(A)]
    tied = dict(   # root children 5 and 2 tie at 3 visits (2 wins); below 2, children 7 and 4 tie at 1 (4 wins), below 5 1 and 0
        parent=[-1, 0, 0, 2, 2, 0, 1, 1], action=[-1, 5, 2, 7, 4, 8, 1, 0], visits=[8, 3, 3, 1, 1, 1, 1, 1],
        value_sum=[0.5, -0.75, 1.25, 0.5, -0.5, 0.125, 0.25, 0.375],
        reward=[0.0, 0.0625, -0.125, 0.0, 0.25, 0.0, -0.0625, 0.0],
        prior_logit=[float("nan"), lg[5], lg[2], lg[7], lg[4], lg[8], lg[1], lg[0]], root_logits=lg,
        topk_action=[2, 5, 8, 0], topk_gumbel=[0.5, -0.25, 1.5, 0.0], topk_round=[2, 2, 1, 1], phase=2, n_surv=2)
    chain = dict(  # a deep line: 0 -> 3 -> 6 -> 1 -> 0
        parent=[-1, 0, 1, 2, 3, 0], action=[-1, 3, 6, 1, 0, 4], visits=[6, 4, 3, 2, 1, 1],
        value_sum=[1.0, -0.3, 0.7, -0.2, 0.9, 0.1], reward=[0.0] * 6, prior_logit=[float("nan")] + [lg[a] for a in (3, 6, 1, 0, 4)],
        root_logits=lg, topk_action=[3, 4], topk_gumbel=[0.1, 0.2], topk_round=[1, 1], phase=1, n_surv=1)
    empty = dict(parent=[], action=[], visits=[], value_sum=[], reward=[], prior_logit=[], root_logits=lg)
    lone = dict(parent=[-1], action=[-1], visits=[1], value_sum=[0.5], reward=[0.0], prior_logit=[float("nan")],
                root_logits=lg, topk_action=[4, 1], topk_gumbel=[0.3, -0.1], topk_round=[0, 0], phase=0, n_surv=2)
    return [tied, chain, empty, lone]


@pytest.mark.parametrize("accum", ["float64", "float32"])
def test_searchtrees_hand_built(accum):
    A, S, K = 9, 8, 4
    games = _hand_games(A)
    firsts = [5, 3, 2, 4]      # a tied-but-not-lowest root move, the PV's own move, an empty tree, an unexpanded move
    _check_against_ref(games, S, K, A, 0.997, accum, firsts)
    trees = _trees(games, S, K, A, 0.997, accum)
    acts, _, _ = trees.pv(max_depth=4)
    assert acts[0, :3].tolist() == [2, 4, -1] and trees.pv(torch.tensor([5, -1, -1, -1], dtype=torch.int32))[0][0, :2].tolist() == [5, 0] and acts[2].tolist() == [-1] * 4 and acts[3].tolist() == [-1] * 4


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("accum", [0, 1])
def test_searchtrees_on_oracle_trees(mode, accum):
    N, S, K, seed = 7, 60, 8, 5
    A = N * N
    rs = np.random.RandomState(10 + 2 * mode + accum)
    cfg = O.make_config(board_size=N, num_simulations=S, num_top_actions=K, mode=mode, eval_seed=seed, logit_div=0,
                        accum_dtype=accum)
    games, firsts = [], []
    for g in range(5):
        b = np.zeros(A, np.int8)
        p, last = 1, -1
        for a in rs.permutation(A)[:rs.randint(0, 12)]:
            b[a] = p; last = int(a); p = -p
        gum = rs.gumbel(0, 1, A)
        t = search_tree(cfg, b, p, last, int((b != 0).sum()), gum)
        lg, _, _ = O.e0_initial(cfg, b, p, last)
        games.append(dict(parent=t["parent"].tolist(), action=t["node_action"].tolist(), visits=t["node_visits"].tolist(),
                          value_sum=t["value_sum"].tolist(), reward=t["reward"].tolist(),
                          prior_logit=t["prior_logit"].tolist(), root_logits=lg.tolist(),
                          topk_action=t["topk_action"].tolist(), topk_gumbel=t["topk_gumbel"].tolist(),
                          topk_round=t["topk_round"].tolist(), phase=t["phase"], n_surv=t["n_surv"]))
        firsts.append(t["action"])
    _check_against_ref(games, S, K, A, 0.997, "float32" if accum else "float64", firsts)
    trees = _trees(games, S, K, A, 0.997, "float32" if accum else "float64")
    acts, _, _ = trees.pv(torch.tensor(firsts, dtype=torch.int32))
    assert acts[:, 0].tolist() == firsts                 # the PV starts with the move the search plays
