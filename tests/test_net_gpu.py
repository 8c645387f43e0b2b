"""Network evaluator on the device: folded/fused inference equals the plain module, weight hot-swap
keeps a captured CUDA graph valid, and a stepwise search driven by the network matches a search whose
evaluator outputs are replayed through the oracle-checked constant path."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _net(seed, n=9, blocks=2, ch=32):
    import torch
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.network import GomokuNetEZ
    torch.manual_seed(seed)
    net = GomokuNetEZ(Config(BOARD_SIZE=n, ACTION_SPACE_SIZE=n * n, NUM_RES_BLOCKS=blocks, NUM_FILTERS=ch, HEAD_HIDDEN_DIM=16))
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.2); m.running_var.uniform_(0.5, 1.5); m.weight.normal_(1, 0.2); m.bias.normal_(0, 0.2)
    return net


def test_device_evaluator_and_weight_hot_swap():
    import torch
    from datou_gomoku_muzero_b200.network import DeviceEvaluator
    net_a, net_b = _net(0), _net(1)
    obs = (torch.rand(64, 3, 9, 9, device="cuda") < 0.3).float()
    ev = DeviceEvaluator(net_a, obs, dtype=torch.float32, graph=True)
    lg, v = ev(obs)
    p, val, _ = net_a.cuda().eval().initial_inference(obs)
    torch.testing.assert_close(lg, p, rtol=1e-3, atol=1e-3)
    torch.testing.assert_close(v, val.reshape(-1), rtol=1e-3, atol=1e-3)
    ev.update_weights(net_b.state_dict())                   # ModelWeightsUpdate (workers.py:331-335)
    lg2, v2 = ev(obs)
    p2, val2, _ = net_b.cuda().eval().initial_inference(obs)
    torch.testing.assert_close(lg2, p2, rtol=1e-3, atol=1e-3)
    torch.testing.assert_close(v2, val2.reshape(-1), rtol=1e-3, atol=1e-3)
    assert (p - p2).abs().max() > 1e-2


@pytest.mark.parametrize("accum", ["float32", "float64"])
def test_network_driven_search_replayed_through_the_oracle(accum):
    """Stepwise search with a real network (continuous float32 logits and values): record every
    (observation -> logits, value) the network produced, then run the CPU oracle's tree logic with a table
    evaluator returning exactly those numbers -> same visit counts, moves, root values.  accum = float32 is the
    production dtype (the reference's inference server returns np.float32 scalars, workers.py:355)."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.network import DeviceEvaluator
    from oracle import oracle
    N, S, G = 9, 64, 12
    A = N * N
    rs = np.random.RandomState(5)
    boards = np.zeros((G, A), np.int8); players = np.ones(G, np.int8)
    last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    for g in range(G):
        p = 1
        for a in rs.permutation(A)[: 3 * g]:
            boards[g, a] = p; last[g] = a; p = -p; mc[g] += 1
        players[g] = p
    eng = SearchEngine(G, board_size=N, num_simulations=S, accum_dtype=accum)
    eng.set_roots(boards, players, last, mc)
    ev = DeviceEvaluator(_net(3), eng.leaf_obs, dtype=torch.float32, graph=False)
    gum_h = rs.gumbel(0, 1, (G, A))
    gum = torch.from_numpy(gum_h).cuda()
    table = {}

    def record(obs, lg, v):
        o, l, vv = obs.cpu().numpy(), lg.cpu().numpy(), v.cpu().numpy()
        for g in range(G):                                  # the evaluator is a pure function of the observation
            key = o[g].tobytes()
            cur = (l[g].copy(), float(vv[g]))
            if key in table:
                assert np.array_equal(table[key][0], cur[0]) and table[key][1] == cur[1]
            table[key] = cur

    def net_values(v):
        return v if accum == "float32" else v.double()       # float64 mode: the same numbers handed over as Python floats
    obs = eng.root_obs(); lg, v = ev(obs); record(obs, lg, v); eng.root_expand(lg, net_values(v), gum)
    for _ in range(S - 1):
        obs = eng.select()
        lg, v = ev(obs)
        record(obs, lg, v)
        eng.expand_backup(lg, net_values(v))
    pol, val, act, vis = (t.cpu().numpy() for t in eng.finalize())
    assert (vis.sum(1) == S - 1).all() and np.allclose(pol.sum(1), 1.0) and (np.abs(val) <= 1).all()

    def table_eval(board, player, last_move):               # what game.get_board_state would build (game.py:12-17)
        o = np.zeros((3, N, N), np.float32)
        o[0] = board == player; o[1] = board == -player
        if last_move >= 0:
            o[2, last_move // N, last_move % N] = 1.0
        return table[o.tobytes()]
    oracle.set_eval_callback(table_eval)
    try:
        cfg = oracle.make_config(board_size=N, num_simulations=S, eval_kind=3, accum_dtype=int(accum == "float32"))
        for g in range(G):
            r = oracle.search(cfg, boards[g], players[g], last[g], mc[g], gum_h[g])
            assert np.array_equal(vis[g], r["visits"]), (accum, g)
            assert act[g] == r["action"] and val[g] == r["value"], (accum, g)
            np.testing.assert_allclose(pol[g], r["policy"], rtol=1e-12, atol=1e-15)
    finally:
        oracle.set_eval_callback(None)


def test_network_search_one_graph_per_step_equals_eager_steps():
    """NetworkSearch: the captured {select -> network -> expand/backup} graph and bf16 NHWC observations written by the
    select give exactly what the eager float32-observation path gives (same folded network, same visit counts)."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.network import DeviceEvaluator, NetworkSearch
    N, S, G = 9, 48, 32
    A = N * N
    rs = np.random.RandomState(11)
    boards = np.zeros((G, A), np.int8); players = np.ones(G, np.int8)
    last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    for g in range(G):
        p = 1
        for a in rs.permutation(A)[: 2 * g]:
            boards[g, a] = p; last[g] = a; p = -p; mc[g] += 1
        players[g] = p
    gum = torch.from_numpy(rs.gumbel(0, 1, (G, A))).cuda()
    net = _net(7)
    out = {}
    for name in ("graph", "eager", "f32obs"):
        eng = SearchEngine(G, board_size=N, num_simulations=S, accum_dtype="float32")
        eng.set_roots(boards, players, last, mc)
        if name == "f32obs":                                  # round 1's path: float32 NCHW observations, cast by torch
            ev = DeviceEvaluator(net, eng.leaf_obs, dtype=torch.bfloat16, graph=False)
            lg, v = ev(eng.root_obs()); eng.root_expand(lg, v, gum)
            for _ in range(S - 1):
                lg, v = ev(eng.select()); eng.expand_backup(lg, v)
        else:
            ns = NetworkSearch(eng, net, dtype=torch.bfloat16, graph=(name == "graph"))
            assert ns.obs.dtype == torch.bfloat16 and ns.obs.is_contiguous(memory_format=torch.channels_last)
            assert ns.search(gum) == S - 1
            if name == "graph":
                assert ns.graph is not None
        pol, val, act, vis = (t.cpu().numpy().copy() for t in eng.finalize())
        out[name] = (vis, act, val)
        assert (vis.sum(1) == S - 1).all()
    for name in ("eager", "f32obs"):
        assert np.array_equal(out["graph"][0], out[name][0]) and np.array_equal(out["graph"][1], out[name][1]), name
        assert np.array_equal(out["graph"][2], out[name][2]), name
    # the bf16 NHWC observation the kernels write == the float32 planes, re-laid out
    eng = SearchEngine(G, board_size=N, num_simulations=S)
    eng.set_roots(boards, players, last, mc)
    o16 = eng.root_obs(eng.obs_buffer_bf16())
    assert torch.equal(o16.float(), eng.root_obs().clone())


def test_bf16_network_against_fp32_network_at_8x128():
    """The bench's network legs run the 8x128 GomokuNetEZ in bf16; the reference's server runs it in fp32
    (workers.py:318).  Bound the difference on 15x15 positions: logits, softmax policy, value -- and what it does
    to the searches (same noise, same roots): agreement of the chosen moves and of the visit distributions.  The
    measured numbers go to gpurun_out/bf16_vs_fp32.json (copied to profiles/ by hand)."""
    import json
    import os
    import torch
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.network import GomokuNetEZ, NetworkSearch
    N, S, G = 15, 64, 256
    A = N * N
    torch.manual_seed(0)
    net = GomokuNetEZ(Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=A, NUM_RES_BLOCKS=8, NUM_FILTERS=128, HEAD_HIDDEN_DIM=64))
    with torch.no_grad():                                     # trained-like statistics: non-trivial BN, non-zero residual gains
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.1); m.running_var.uniform_(0.8, 1.2); m.weight.normal_(0.5, 0.1); m.bias.normal_(0, 0.1)
    rs = np.random.RandomState(2)
    boards = np.zeros((G, A), np.int8); players = np.ones(G, np.int8)
    last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    for g in range(G):
        k = int(rs.randint(0, 120)); p = 1
        for a in rs.permutation(A)[:k]:
            boards[g, a] = p; last[g] = a; p = -p
        players[g] = p; mc[g] = k
    gum = torch.from_numpy(rs.gumbel(0, 1, (G, A))).cuda()
    res = {}
    saved = torch.backends.cudnn.allow_tf32
    try:
        for name, dt, tf32 in (("fp32", torch.float32, False), ("tf32", torch.float32, True), ("bf16", torch.bfloat16, True)):
            torch.backends.cudnn.allow_tf32 = tf32
            eng = SearchEngine(G, board_size=N, num_simulations=S, accum_dtype="float32")
            eng.set_roots(boards, players, last, mc)
            ns = NetworkSearch(eng, net, dtype=dt, graph=False)
            eng.root_obs(ns.obs); ns.ev._forward()
            lg0, v0 = ns.ev.logits.clone(), ns.ev.values.clone()
            ns.search(gum)
            pol, val, act, vis = (t.cpu().numpy().copy() for t in eng.finalize())
            res[name] = dict(logits=lg0.cpu().numpy(), values=v0.cpu().numpy(), act=act, vis=vis)
    finally:
        torch.backends.cudnn.allow_tf32 = saved
    valid = boards == 0

    def softmax(l):
        l = np.where(valid, l, -np.inf); e = np.exp(l - l.max(1, keepdims=True)); return e / e.sum(1, keepdims=True)
    rep = {}
    for name in ("tf32", "bf16"):
        a, b = res["fp32"], res[name]
        rep[name] = dict(max_abs_dlogit=float(np.abs(a["logits"] - b["logits"]).max()),
                         max_abs_dpolicy=float(np.abs(softmax(a["logits"]) - softmax(b["logits"])).max()),
                         max_abs_dvalue=float(np.abs(a["values"] - b["values"]).max()),
                         move_agreement=float((a["act"] == b["act"]).mean()),
                         visit_count_identical=float((a["vis"] == b["vis"]).all(1).mean()),
                         mean_visit_l1=float(np.abs(a["vis"] - b["vis"]).sum(1).mean() / (2 * (S - 1))))
    rep["config"] = dict(board=N, sims=S, games=G, net="GomokuNetEZ 8x128, seeded, perturbed BN statistics", reference="fp32 (allow_tf32 off)")
    os.makedirs("gpurun_out", exist_ok=True)
    json.dump(rep, open(os.path.join("gpurun_out", "bf16_vs_fp32.json"), "w"), indent=1)
    print(json.dumps(rep))
    assert rep["bf16"]["max_abs_dpolicy"] < 0.02 and rep["bf16"]["max_abs_dvalue"] < 0.05, rep
    assert rep["tf32"]["max_abs_dpolicy"] <= rep["bf16"]["max_abs_dpolicy"] + 1e-3, rep
    assert rep["bf16"]["move_agreement"] > 0.5 and rep["bf16"]["mean_visit_l1"] < 0.35, rep


def test_selfplay_with_the_network_searcher_play_equals_stepping():
    """SelfPlayEngine with a GomokuNetEZ evaluator (the production path of universal_worker, workers.py:129-241):
    play(sink=...) -- lock-step network searches cut into chunks, finished games packed on the device and handed
    to the sink -- produces exactly the games a plain loop of step() calls does, every game is a legal finished
    Gomoku game, and the trajectories land in a DeviceReplayBuffer ready to be sampled."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.game import GomokuGame
    from datou_gomoku_muzero_b200.network import NetworkSearch
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    N, S, G, moves = 6, 20, 16, 30
    net = _net(3, n=N, blocks=1, ch=16)

    def run(chunked):
        e = SearchEngine(G, board_size=N, num_simulations=S, n_in_row=4, accum_dtype="float32")
        sp = SelfPlayEngine(e, net if chunked else NetworkSearch(e, net), noise_seed=77)
        assert isinstance(sp.searcher, NetworkSearch)
        traj = TrajectoryStore(e, extra_slots=8 * G)
        got = []
        if chunked:
            sp.play(moves_per_game=moves, traj=traj, sink=got.append, chunk=7)
        else:
            for _ in range(moves):
                sp.step(traj=traj)
            got.append(traj.pack_finished(recycle=True))
        assert sp.moves_played == G * moves
        games = {}
        for pk in got:
            for i in range(len(pk)):
                games.setdefault(int(pk.table[i][1]), []).append(pk.game(i).copy())
        return games, got, e

    ga, packs, e = run(True)
    gb, _, _ = run(False)
    assert sum(len(v) for v in ga.values()) >= G // 2 and set(ga) == set(gb)
    for g in ga:
        assert len(ga[g]) == len(gb[g])
        for a, b in zip(ga[g], gb[g]):          # field by field (numpy does not copy a structured dtype's padding; slot ids depend on recycling)
            assert len(a) == len(b)
            for f in a.dtype.names:
                if f not in ("slot", "game_seq"):
                    assert np.array_equal(a[f], b[f]), (g, f)
    # every recorded game replays to a finished game on the host GomokuGame with the recorded winner
    pk = packs[0]
    for i in range(len(pk)):
        r, gm = pk.game(i), GomokuGame(N, 4)
        for t in range(len(r)):
            assert np.array_equal(r["board"][t].reshape(N, N), gm.board) and gm.get_game_ended() is None
            assert abs(float(r["policy"][t].sum()) - 1.0) < 1e-12 and r["policy"][t][int(r["action"][t])] > 0
            gm.do_move(int(r["action"][t]))
        assert gm.get_game_ended() is not None and int(gm.get_game_ended()) == int(pk.table[i][3])
    buf = DeviceReplayBuffer(4096, N)
    for p in packs:
        buf.add_packed(p)
    assert len(buf) == sum(p.n_moves for p in packs)
    batch, idx, w = buf.sample(32)
    assert batch is not None and len(idx) == 32
    with pytest.raises(ValueError):
        SelfPlayEngine(e, "e1")
