"""gmz_tree_export on the device: every exported tree equals the CPU oracle's node for node (parent, action, depth,
visits, and the bits of value_sum, reward, prior_logit and the MinMax bounds; sim_count, the Gumbel top-k in halving
order and the round that eliminated each entry) in both modes, both accumulation dtypes, dense and quantised logits,
through the fused, the stepwise and the learned-dynamics search; the export reads the workspace and writes nothing into
it; stale trees export as empty; a network search's tree has the structure every search has; bad handles fail cleanly."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _roots(N, G, rs, full_first=True):
    """Game 0 the full board (inactive), game 1 the empty board, the rest random mid-game positions."""
    A = N * N
    boards = np.zeros((G, A), np.int8)
    players = np.ones(G, np.int8); last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    for g in range(G):
        k = A if (g == 0 and full_first) else 0 if g == 1 else int(rs.randint(1, max(2, A * 2 // 3)))
        p = 1
        for a in rs.permutation(A)[:k]:
            boards[g, a] = p; last[g] = int(a); p = -p
        players[g] = p; mc[g] = k
    return boards, players, last, mc


def _bits(x):
    return np.ascontiguousarray(x).tobytes()


def _compare(tag, tr, want, roots):
    """tr: SearchTrees; want: list of _tree_oracle.search_tree dicts, one per game."""
    h = {f: getattr(tr, f).cpu().numpy() for f in ("num_nodes", "sim_count", "root", "minmax", "halving", "topk_action",
                                                  "topk_gumbel", "topk_logit", "topk_round", "parent", "action", "depth",
                                                  "visits", "value_sum", "reward", "prior_logit")}
    boards, players, last, mc = roots
    for g, w in enumerate(want):
        t = f"{tag} game {g}"
        n = w["num_nodes"]
        assert h["num_nodes"][g] == n and h["sim_count"][g] == w["sim_count"], f"{t}: num_nodes / sim_count"
        assert list(h["root"][g]) == [players[g], last[g], mc[g]], f"{t}: root"
        assert _bits(h["minmax"][g]) == _bits(w["minmax"]), f"{t}: minmax {h['minmax'][g]} vs {w['minmax']}"
        assert list(h["halving"][g]) == [w["phase"], w["n_surv"], w["n_init"]], f"{t}: halving {h['halving'][g]}"
        k = w["n_init"]
        assert np.array_equal(h["topk_action"][g, :k], w["topk_action"]), f"{t}: top-k order"
        assert _bits(h["topk_gumbel"][g, :k]) == _bits(w["topk_gumbel"]), f"{t}: top-k gumbel"
        assert _bits(h["topk_logit"][g, :k]) == _bits(w["topk_logit"]), f"{t}: top-k logit"
        assert np.array_equal(h["topk_round"][g, :k], w["topk_round"]), f"{t}: rounds {h['topk_round'][g, :k]} vs {w['topk_round']}"
        assert (h["topk_action"][g, k:] == -1).all() and (h["topk_round"][g, k:] == -1).all(), t
        for f, o in (("parent", "parent"), ("action", "node_action"), ("depth", "depth"), ("visits", "node_visits")):
            assert np.array_equal(h[f][g, :n], w[o]), f"{t}: {f}"
            assert (h[f][g, n:] == -1).all(), f"{t}: {f} past the end"
        for f in ("value_sum", "reward", "prior_logit"):
            assert _bits(h[f][g, :n]) == _bits(w[f]), f"{t}: {f} bits"
            assert (h[f][g, n:] == 0).all(), f"{t}: {f} past the end"


def _oracle(cfg, roots, gumbel):
    from _tree_oracle import search_tree
    boards, players, last, mc = roots
    return [search_tree(cfg, boards[g], players[g], last[g], mc[g], gumbel[g]) for g in range(len(boards))]


def _check_decision(tag, eng, tr):
    """Root visits of the export = finalize's; pv(first=action) starts with the action, and so does pv() unless the
    maximum is tied."""
    _, _, act, vis = (t.clone() for t in eng.finalize(want_visits=True))
    tab = tr.root_table()
    assert torch.equal(tab["visits"], vis), f"{tag}: root visits vs finalize"
    a, _, _ = tr.pv(act)
    assert torch.equal(a[:, 0], act), f"{tag}: pv(first=action)"
    vmax = vis.max(1, keepdim=True).values
    untied = ((vis == vmax).sum(1) == 1) & (act >= 0)
    a0, _, _ = tr.pv()
    assert torch.equal(a0[untied, 0], act[untied]), f"{tag}: pv() without ties"


CONFIGS = [(6, 50), (9, 100), (15, 400), (19, 200)]


@pytest.mark.parametrize("N,S", CONFIGS)
def test_export_matches_oracle(N, S):
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    G, seed = 6, 17
    A = N * N
    rs = np.random.RandomState(1000 + N)
    for K in (1, 16, 32):
        for accum in ("float64", "float32"):
            for div in (16, 0):
                for mode in ("AlphaZero", "MuZero"):
                    roots = _roots(N, G, rs)
                    gumbel = rs.gumbel(0, 1, (G, A))
                    cfg = oracle.make_config(board_size=N, num_simulations=S, num_top_actions=K, eval_seed=seed, logit_div=div,
                                             accum_dtype=int(accum == "float32"), mode=int(mode == "MuZero"))
                    want = _oracle(cfg, roots, gumbel)
                    eng = SearchEngine(G, board_size=N, num_simulations=S, num_top_actions=K, mode=mode, accum_dtype=accum)
                    paths = [("fused", eng.search_e0)] + ([("stepwise", eng.search_stepwise_e0)] if mode == "AlphaZero" else [])
                    for path, run in paths:
                        tag = f"N={N} S={S} K={K} {accum} div={div} {mode} {path}"
                        eng.set_roots(*roots)
                        run(torch.from_numpy(gumbel).cuda(), seed, div)
                        tr = eng.export_tree()
                        _compare(tag, tr, want, roots)
                        _check_decision(tag, eng, tr)
                    del eng


@pytest.mark.parametrize("N", [7, 11, 13, 17])
def test_export_matches_oracle_lane_chunks(N):
    """Boards of one, two and three lane chunks (odd N: a centre cell), both modes."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    G, S, K, seed = 8, 64, 16, 29
    A = N * N
    rs = np.random.RandomState(2000 + N)
    for accum, div in (("float32", 0), ("float64", 16)):
        for mode in ("AlphaZero", "MuZero"):
            roots = _roots(N, G, rs)
            gumbel = rs.gumbel(0, 1, (G, A))
            cfg = oracle.make_config(board_size=N, num_simulations=S, num_top_actions=K, eval_seed=seed, logit_div=div,
                                     accum_dtype=int(accum == "float32"), mode=int(mode == "MuZero"))
            eng = SearchEngine(G, board_size=N, num_simulations=S, num_top_actions=K, mode=mode, accum_dtype=accum)
            eng.set_roots(*roots)
            eng.search_e0(torch.from_numpy(gumbel).cuda(), seed, div)
            tag = f"N={N} {accum} div={div} {mode}"
            tr = eng.export_tree()
            _compare(tag, tr, _oracle(cfg, roots, gumbel), roots)
            _check_decision(tag, eng, tr)


@pytest.mark.parametrize("N", [8, 17])
def test_export_muzero_device_search(N):
    """MuZero mode through the hidden-state pool with TorchE0, set up as test_shapes_gpu's device-search test."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.muzero import MuZeroDeviceSearch, TorchE0
    from oracle import oracle
    A, S, G, seed = N * N, 32, 10, 41
    rs = np.random.RandomState(200 + N)
    roots = _roots(N, G, rs)
    gumbel = rs.gumbel(0, 1, (G, A))
    eng = SearchEngine(G, board_size=N, num_simulations=S, mode="MuZero")
    eng.set_roots(*roots)
    e0 = TorchE0(N, seed=seed)
    MuZeroDeviceSearch(eng, e0.initial, e0.recurrent).search(torch.from_numpy(gumbel).cuda())
    cfg = oracle.make_config(board_size=N, num_simulations=S, mode=1, eval_seed=seed)
    tr = eng.export_tree()
    _compare(f"N={N} MuZeroDeviceSearch", tr, _oracle(cfg, roots, gumbel), roots)
    _check_decision(f"N={N} MuZeroDeviceSearch", eng, tr)


def test_export_is_read_only_and_changes_no_search():
    """The workspace is bit-identical across an export, and a stepwise search exported after every step (its partial
    trees) decides exactly as one that is never exported."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    N, S, K, G, seed = 9, 48, 16, 8, 3
    A = N * N
    rs = np.random.RandomState(7)
    roots = _roots(N, G, rs)
    gumbel = torch.from_numpy(rs.gumbel(0, 1, (G, A))).cuda()
    cfg = oracle.make_config(board_size=N, num_simulations=S, num_top_actions=K, eval_seed=seed, accum_dtype=1, logit_div=0)
    want = _oracle(cfg, roots, gumbel.cpu().numpy())
    outs = []
    for exporting in (False, True):
        eng = SearchEngine(G, board_size=N, num_simulations=S, num_top_actions=K, accum_dtype="float32")
        eng.set_roots(*roots)
        obs = eng.root_obs()
        lg, v = eng.e0_eval(obs, seed, 0)
        eng.root_expand(lg, v, gumbel)
        tr = None
        for step in range(S - 1):
            if exporting:
                before = eng.workspace.clone()
                tr = eng.export_tree(out=tr)
                torch.cuda.synchronize()
                assert torch.equal(before, eng.workspace), f"step {step}: the export wrote into the workspace"
                nn = tr.num_nodes.cpu().numpy()
                live = np.array([w["num_nodes"] > 0 for w in want])
                assert (nn[live] == step + 1).all() and (nn[~live] == 0).all(), f"step {step}: partial tree sizes {nn}"
                par = tr.parent.cpu().numpy()
                for g in np.flatnonzero(live):       # the partial tree is the oracle's first step + 1 nodes
                    assert np.array_equal(par[g, :step + 1], want[g]["parent"][:step + 1]), f"step {step} game {g}"
            obs = eng.select()
            eng.e0_eval(obs, seed, 0, lg, v)
            eng.expand_backup(lg, v)
        outs.append([t.clone().cpu().numpy() for t in eng.finalize(want_visits=True)])
        if exporting:
            _compare("stepwise, exported every step", eng.export_tree(), want, roots)
    for a, b in zip(*outs):
        assert _bits(a) == _bits(b), "a search with exports in between decided differently"


def test_stale_trees_export_empty():
    """After game_step, set_roots or a self-play launch every game exports 0 nodes; the full-board root never has a tree."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    N, S, G, seed = 9, 32, 12, 5
    A = N * N
    rs = np.random.RandomState(11)
    roots = _roots(N, G, rs)
    gumbel = torch.from_numpy(rs.gumbel(0, 1, (G, A))).cuda()
    eng = SearchEngine(G, board_size=N, num_simulations=S)

    def searched():
        eng.set_roots(*roots)
        eng.search_e0(gumbel, seed)
        n = eng.export_tree().num_nodes.cpu().numpy()
        assert n[0] == 0 and (n[1:] == S).all(), n
        return eng.finalize()[2].clone()

    act = searched()
    eng.game_step(act)
    assert (eng.export_tree().num_nodes == 0).all(), "after game_step"
    searched()
    eng.set_roots(*roots)
    assert (eng.export_tree().num_nodes == 0).all(), "after set_roots"
    searched()
    eng.selfplay_e0(4 * G, seed, noise_seed=1)
    tr = eng.export_tree()
    assert (tr.num_nodes == 0).all() and (tr.halving == 0).all() and (tr.topk_action == -1).all(), "after selfplay_e0"
    assert torch.isnan(tr.root_logits).all() and (tr.parent == -1).all() and (tr.visits == -1).all()
    mm = tr.minmax.cpu().numpy()
    assert (mm[:, 0] == np.inf).all() and (mm[:, 1] == -np.inf).all()


def _check_invariants(tag, tr, mz, K):
    h = {f: getattr(tr, f).cpu().numpy() for f in ("num_nodes", "sim_count", "parent", "depth", "visits")}
    for g in range(tr.G):
        n = int(h["num_nodes"][g])
        if n == 0:
            continue
        par, dep, vis = h["parent"][g, :n], h["depth"][g, :n], h["visits"][g, :n]
        assert par[0] == -1 and (par[1:] >= 0).all() and (par[1:] < np.arange(1, n)).all(), f"{tag} {g}: parents first"
        assert dep[0] == 0 and np.array_equal(dep[1:], dep[par[1:]] + 1), f"{tag} {g}: depth"
        kids = np.zeros(n, np.int64)
        np.add.at(kids, par[1:], vis[1:])
        own = vis - kids
        assert vis[0] == h["sim_count"][g] and own[0] == 1, f"{tag} {g}: root visits"
        assert (own[1:] == 1).all() if not mz else ((own[1:] >= 1) & (own[1:] <= K)).all(), f"{tag} {g}: backups"


def test_network_search_tree_structure():
    """A seeded GomokuNetEZ through NetworkSearch (bf16, CUDA graph; AlphaZero mode) and its folded heads through
    MuZeroDeviceSearch (learned dynamics): every tree has the structure of a search."""
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.muzero import FoldedRecurrentInference, MuZeroDeviceSearch
    from datou_gomoku_muzero_b200.network import FoldedInitialInference, GomokuNetEZ, NetworkSearch
    N, S, K, G = 9, 40, 16, 16
    A = N * N
    torch.manual_seed(0)
    net = GomokuNetEZ(Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=A, NUM_RES_BLOCKS=1, NUM_FILTERS=16, HEAD_HIDDEN_DIM=8)).cuda().eval()
    rs = np.random.RandomState(3)
    roots = _roots(N, G, rs)
    gumbel = torch.from_numpy(rs.gumbel(0, 1, (G, A))).cuda()
    eng = SearchEngine(G, board_size=N, num_simulations=S, num_top_actions=K, accum_dtype="float32")
    eng.set_roots(*roots)
    with torch.no_grad():
        NetworkSearch(eng, net).search(gumbel)
    tr = eng.export_tree()
    _check_invariants("NetworkSearch", tr, False, K)
    _check_decision("NetworkSearch", eng, tr)
    assert (tr.num_nodes[1:] == S).all()

    fi, fr = FoldedInitialInference(net, torch.bfloat16), FoldedRecurrentInference(net, torch.bfloat16)

    def initial(obs):
        p, v, h = fi(obs.to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
        return p.float().contiguous(), v.reshape(-1).float(), h
    mz = SearchEngine(G, board_size=N, num_simulations=S, num_top_actions=K, mode="MuZero", accum_dtype="float32")
    mz.set_roots(*roots)
    with torch.no_grad():
        MuZeroDeviceSearch(mz, initial, fr, graph=True).search(gumbel)
    tr = mz.export_tree()
    _check_invariants("MuZeroDeviceSearch", tr, True, K)
    _check_decision("MuZeroDeviceSearch", mz, tr)


def test_bad_arguments():
    """A destroyed handle and a NULL `out` are errors with a message; nothing is launched."""
    from datou_gomoku_muzero_b200 import _lib
    from datou_gomoku_muzero_b200.engine import SearchEngine
    eng = SearchEngine(2, board_size=6, num_simulations=8)
    lib = eng.lib
    tr = eng.export_tree()
    c = _lib.GmzTreeOut(*[getattr(tr, f).data_ptr() for f, _ in _lib.GmzTreeOut._fields_])
    assert lib.gmz_tree_export(eng.handle, None, eng._stream()) != 0 and b"null out" in lib.gmz_last_error()
    handle = eng.handle
    lib.gmz_destroy(handle)
    eng.handle = None
    before = tr.parent.clone()
    tr.parent.fill_(7)
    assert lib.gmz_tree_export(handle, C.byref(c), None) != 0 and b"destroyed" in lib.gmz_last_error()
    torch.cuda.synchronize()
    assert (tr.parent == 7).all(), "a rejected call launched work"
    assert before.shape == tr.parent.shape


def test_last_tree_starts_with_the_move_played():
    """AlphaZeroMCTS(...).search(game) then last_tree(): the PV starts with the returned move."""
    import queue
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.game import GomokuGame
    from datou_gomoku_muzero_b200.mcts import AlphaZeroMCTS
    from oracle import oracle
    N, S, K, seed = 6, 24, 8, 9
    old = (config.BOARD_SIZE, config.ACTION_SPACE_SIZE, config.NUM_SIMULATIONS, config.NUM_TOP_ACTIONS, config.N_IN_ROW)
    config.BOARD_SIZE, config.ACTION_SPACE_SIZE, config.NUM_SIMULATIONS, config.NUM_TOP_ACTIONS, config.N_IN_ROW = N, N * N, S, K, 4
    try:
        ocfg = oracle.make_config(board_size=N, num_simulations=S, num_top_actions=K, eval_seed=seed)

        class Server:          # answers 'initial' requests with E0, as the reference's inference server answers them
            def __init__(self):
                self.q = queue.Queue()

            def put(self, item):
                _, kind, obs = item
                own, opp, lastp = np.asarray(obs)
                board = (own - opp).astype(np.int8)              # relative to the player to move (+1)
                last = int(np.flatnonzero(lastp.reshape(-1))[0]) if lastp.any() else -1
                lg, v, _ = oracle.e0_initial(ocfg, board.reshape(-1), 1, last)
                self.q.put((lg, v, None))

        srv = Server()
        mcts = AlphaZeroMCTS(0, srv, srv.q)
        game = GomokuGame(board_size=N, n_in_row=4)
        for a in (14, 15, 21):
            game.do_move(a)
        np.random.seed(4)
        _, _, action = mcts.search(game)
        t = mcts.last_tree()
        assert action >= 0 and t["pv_actions"][0] == action and t["num_nodes"] == S and t["sim_count"] == S
        assert t["root"]["visits"][action] == t["pv_visits"][0] == t["root"]["visits"].max()
        assert t["parent"][0] == -1 and len(t["parent"]) == S
    finally:
        config.BOARD_SIZE, config.ACTION_SPACE_SIZE, config.NUM_SIMULATIONS, config.NUM_TOP_ACTIONS, config.N_IN_ROW = old
