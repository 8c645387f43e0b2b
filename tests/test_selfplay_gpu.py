"""Persistent self-play kernel: whole games on the device, checked move for move against the CPU
oracle's game loop (same E0 evaluator, the kernel's own counter-based Gumbel noise regenerated on
the host side of the test), then turned into GameRecord / TrainingSlice like workers.py:183-230."""
import os

import numpy as np
import pytest

from _golden_util import GOLDEN_DIR

pytestmark = pytest.mark.gpu


def _noise_for_game(eng, g, n_moves, noise_seed):
    import torch
    out = torch.empty((n_moves, eng.A), dtype=torch.float64, device=eng.device)
    for k in range(n_moves):
        eng.fill_gumbel(out[k], noise_seed, (k * eng.G + g) * eng.A)
    return out.cpu().numpy()


@pytest.mark.parametrize("N,S,G,mode", [(6, 36, 24, "AlphaZero"), (9, 64, 40, "AlphaZero"), (6, 50, 24, "MuZero")])
def test_selfplay_games_match_oracle(N, S, G, mode):
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    from oracle import oracle
    A, seed, nseed = N * N, 5, 77
    eng = SearchEngine(G, board_size=N, num_simulations=S, mode=mode)
    sp = SelfPlayEngine(eng, "e0", seed=seed, noise_seed=nseed)
    traj = TrajectoryStore(eng, extra_slots=8)
    finished = []
    for _ in range(6):
        sp.play(moves_per_game=A // 3, traj=traj, restart=True)
        finished += traj.harvest()
    moves, nfin = eng.play_counters()
    assert nfin == len(finished) and nfin >= G          # every game ended at least once
    assert moves <= 6 * G * (A // 3) and eng.tickets_idle == 0      # games may park when the 8 spare slots run out
    cfg = oracle.make_config(board_size=N, num_simulations=S, eval_seed=seed, mode=0 if mode == "AlphaZero" else 1)
    first = {}
    for r in finished:                                  # the first game of each index starts at noise counter 0
        first.setdefault(r["game"], r)
    checked = 0
    for g, r in sorted(first.items())[:12]:
        assert r["start_move_count"] == 0 and not r["start_board"].any() and r["start_player"] == 1
        gum = _noise_for_game(eng, g, r["length"], nseed)
        o = oracle.selfplay_game(cfg, np.concatenate([gum, np.zeros((1, A))]))
        assert o["T"] == r["length"], (g, o["T"], r["length"])
        assert np.array_equal(o["actions"], r["actions"]) and o["winner"] == r["winner"], g
        assert np.array_equal(o["values"], r["values"]), g
        np.testing.assert_allclose(r["policies"], o["policies"], rtol=1e-12, atol=1e-15)
        checked += 1
    assert checked >= 8


def test_reanalysis_matches_oracle_per_position():
    """Surge re-analysis (workers.py:243-305): every stored position of finished games searched again in
    one batch; policies / values must equal a per-position oracle search with the same noise."""
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.mcts import AlphaZeroMCTS
    from datou_gomoku_muzero_b200.reanalysis import positions_of, reanalyse
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore, build_game_record
    from oracle import oracle
    N, S, G, seed = 6, 24, 16, 3
    A = N * N
    eng = SearchEngine(G, board_size=N, num_simulations=S)
    sp = SelfPlayEngine(eng, "e0", seed=seed, noise_seed=9)
    traj = TrajectoryStore(eng, extra_slots=16)
    recs = []
    while len(recs) < 3:
        sp.play(moves_per_game=6, traj=traj)
        recs += traj.harvest()
    games = [build_game_record(r) for r in recs[:3]]
    eng2 = SearchEngine(32, board_size=N, num_simulations=S)
    new_seed = seed + 1                                       # "the latest model"
    bs = AlphaZeroMCTS.for_engine(eng2, "e0", eval_seed=new_seed)
    rs = np.random.RandomState(4)
    noise = []
    def gumbel_fn(n, a):
        noise.append(rs.gumbel(0, 1, (n, a))); return noise[-1]
    saved = config.BOARD_SIZE
    config.BOARD_SIZE = N
    try:
        out = reanalyse(games, bs, board_size=N, gumbel_fn=gumbel_fn)
    finally:
        config.BOARD_SIZE = saved
    allnoise = np.concatenate(noise)
    cfg = oracle.make_config(board_size=N, num_simulations=S, eval_seed=new_seed)
    off = 0
    for gr, (pol, targets, vals) in zip(games, out):
        b, pl, lm, mc = positions_of(gr, N)
        T = len(gr.actions)
        opol, oval, oact, _ = oracle.search_batch(cfg, b, pl, lm, mc, allnoise[off:off + T])
        np.testing.assert_allclose(pol, opol, rtol=1e-12, atol=1e-15)
        assert np.array_equal(vals, oval)                       # the re-searched root values, bit for bit
        assert len(targets) == T and all(isinstance(t, float) for t in targets)
        # the new value targets: workers.py:291-292 restated (float32 rewards there, unlike self-play: float32 sums)
        rew = np.array(gr.rewards, dtype=np.float32); v32 = np.array(oval, dtype=np.float32)
        exp = np.zeros(T, np.float32)
        for t in range(T):
            acc = sum((config.DISCOUNT ** i) * rew[t + i] for i in range(config.N_STEPS) if t + i < T)
            boot = v32[t + config.N_STEPS] * (config.DISCOUNT ** config.N_STEPS) if t + config.N_STEPS < T else 0.0
            exp[t] = acc + boot
        assert np.array_equal(np.array(targets, np.float32), exp)
        off += T


def test_device_ring_batches_match_host_slices():
    """Trainer batches gathered from the device replay ring (gmz_traj_pack -> DeviceReplayBuffer.batch) vs the host
    post-processing (build_game_record + cut_training_slices) of the same kernel-played games: two engines play the
    same seeded E0 self-play, one is harvested to the host, the other packed into a ring.  The persistent kernel's
    finish order is not fixed, so games are paired by engine game index and action sequence."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore, build_game_record, cut_training_slices
    N, G = 6, 12
    sps, trajs = [], []
    for _ in range(2):
        eng = SearchEngine(G, board_size=N, num_simulations=20)
        sps.append(SelfPlayEngine(eng, "e0", seed=2, noise_seed=3))
        trajs.append(TrajectoryStore(eng, extra_slots=24))
    buf = DeviceReplayBuffer(4096, N)
    fin, at = [], {}                                   # at: (game, actions) -> ring position of the game's first move
    for _ in range(40):
        sps[0].play(moves_per_game=5, traj=trajs[0])
        fin += trajs[0].harvest()
        sps[1].play(moves_per_game=5, traj=trajs[1])
        pg = trajs[1].pack_finished()
        if pg is not None:
            for i in range(len(pg)):
                at[(int(pg.table[i][1]), tuple(pg.game(i)["action"].tolist()))] = buf.sum_tree.write_ptr + int(pg.offsets[i])
            buf.add_packed(pg)
        pairs = [(r, at[k]) for r in fin if (k := (r["game"], tuple(r["actions"].tolist()))) in at]
        if len(pairs) >= 6:
            break
    assert len(pairs) >= 6 and len(buf) < buf.capacity          # the ring has not wrapped: positions are as recorded
    for r, p0 in pairs:
        sl = cut_training_slices(build_game_record(r))
        obs, act, rew, pi, val = (x.cpu().numpy() for x in buf.batch(torch.arange(p0, p0 + len(sl), device="cuda")))
        for t, s in enumerate(sl):
            assert np.array_equal(obs[t], s.observation) and np.array_equal(act[t], s.action_history)
            assert np.array_equal(rew[t], s.reward_history) and np.array_equal(pi[t], s.policy_history)
            assert np.array_equal(val[t], s.value_history)


def test_device_batch_d4_augmentation_matches_reference_loss_path():
    """gmz_records_batch vs what the reference's calculate_loss feeds its networks (loss.py:37-51,
    captured in tests/golden/augment_kat.npz) for all 8 symmetries, and vs the numpy restatement."""
    import torch
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    from oracle import oracle
    from test_records_gpu import _load_game
    z = np.load(os.path.join(GOLDEN_DIR, "selfplay_az_6_36.npz"))
    g = np.load(os.path.join(GOLDEN_DIR, "augment_kat.npz"))
    N, nir, S, K, seed, U, n_steps, version = (int(x) for x in z["params"][:8])
    T = len(z["actions"])
    pick = [0, 3, 7, T // 2, T - 7, T - 5, T - 3, T - 1]            # as tests/golden/make_golden.py gen_augment
    saved = (config.DISCOUNT, config.N_STEPS, config.NUM_UNROLL_STEPS)
    config.DISCOUNT, config.N_STEPS, config.NUM_UNROLL_STEPS = float(z["discount"]), n_steps, U
    try:
        eng = SearchEngine(4, board_size=N, num_simulations=8)
        traj = TrajectoryStore(eng, extra_slots=8)
        slot = 5
        T = _load_game(traj, slot, z)
        traj.fin_queue[0] = torch.tensor([slot, 0, T, int(z["winner"])], dtype=torch.int32).cuda()
        traj.fin_count.fill_(1)
        buf = DeviceReplayBuffer(T, N)
        buf.add_packed(traj.pack_finished())
        samples = torch.tensor(pick, device="cuda")                    # the game fills ring positions 0 .. T-1
        base = [x.cpu().numpy() for x in buf.batch(samples)]
        assert np.array_equal(base[0], g["obs"]) and np.array_equal(base[1], g["act"]) and np.array_equal(base[3], g["pi"])
        valid = g["act"] != -1
        for k in range(4):
            for f in (0, 1):
                obs, act, rew, pi, val = (x.cpu().numpy() for x in buf.batch(samples, rot_k=k, flip=bool(f)))
                tag = f"k{k}f{f}"
                assert np.array_equal(obs, g["obs_" + tag]), tag
                assert np.array_equal(pi.astype(np.float32), g["pi_" + tag]), tag
                assert np.array_equal(act[valid], g["act_" + tag][valid]) and (act[~valid] == -1).all(), tag
                o_obs, o_act, o_pi = oracle.augment_batch(g["obs"], g["act"], g["pi"], k, bool(f))
                assert np.array_equal(obs, o_obs) and np.array_equal(pi, o_pi) and np.array_equal(act[valid], o_act[valid])
                assert np.array_equal(rew, base[2]) and np.array_equal(val, base[4])          # scalars do not move
    finally:
        config.DISCOUNT, config.N_STEPS, config.NUM_UNROLL_STEPS = saved


def test_stepwise_selfplay_with_external_evaluator_matches_persistent_kernel():
    """SelfPlayEngine.step() (stepwise kernels + an evaluator callable + gmz_selfplay_step) must play
    the same games, move for move, as the persistent kernel when the evaluator is E0 and the noise is the
    same counter-based stream."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    N, S, G, seed, nseed = 6, 30, 16, 8, 21
    A = N * N
    # reference run: persistent kernel
    e1 = SearchEngine(G, board_size=N, num_simulations=S)
    sp1 = SelfPlayEngine(e1, "e0", seed=seed, noise_seed=nseed)
    t1 = TrajectoryStore(e1, extra_slots=64)
    fin1 = []
    for _ in range(5):
        sp1.play(moves_per_game=8, traj=t1); fin1 += t1.harvest()
    # stepwise run: evaluator = the stand-alone E0 kernel, noise = same per-game counters
    e2 = SearchEngine(G, board_size=N, num_simulations=S)

    def evaluator(obs):
        return e2.e0_eval(obs, seed)
    sp2 = SelfPlayEngine(e2, evaluator, noise_seed=nseed)
    t2 = TrajectoryStore(e2, extra_slots=64)
    counters = np.zeros(G, np.int64)          # searches done per game (the play kernel's noise_ctr)
    fin2 = []
    gum = torch.empty((G, A), dtype=torch.float64, device="cuda")
    for _ in range(40):
        for g in range(G):
            e2.fill_gumbel(gum[g], nseed, int((counters[g] * G + g) * A))
        pol, val, act, _ = sp2.search(gumbel=gum)
        e2.selfplay_step(pol, val, act, t2, True)
        counters += 1
        fin2 += t2.harvest()
    first1, first2 = {}, {}
    for r in fin1: first1.setdefault(r["game"], r)
    for r in fin2: first2.setdefault(r["game"], r)
    common = sorted(set(first1) & set(first2))
    assert len(common) >= 8
    for g in common:
        a, b = first1[g], first2[g]
        assert a["length"] == b["length"] and np.array_equal(a["actions"], b["actions"]) and a["winner"] == b["winner"], g
        assert np.array_equal(a["values"], b["values"]) and np.array_equal(a["policies"], b["policies"]), g


def test_muzero_searcher_selfplay_matches_persistent_kernel():
    """MuZero mode: SelfPlayEngine with (initial_fn, recurrent_fn) = E0 as torch ops (hidden states through
    the device pool kernels) plays the same games as the persistent MuZero-mode kernel."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.muzero import MuZeroDeviceSearch, TorchE0
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    N, S, G, seed, nseed = 6, 40, 12, 9, 33
    A = N * N
    e1 = SearchEngine(G, board_size=N, num_simulations=S, mode="MuZero")
    sp1 = SelfPlayEngine(e1, "e0", seed=seed, noise_seed=nseed)
    t1 = TrajectoryStore(e1, extra_slots=64)
    fin1 = []
    for _ in range(5):
        sp1.play(moves_per_game=8, traj=t1); fin1 += t1.harvest()
    e2 = SearchEngine(G, board_size=N, num_simulations=S, mode="MuZero")
    e0 = TorchE0(N, seed=seed)
    sp2 = SelfPlayEngine(e2, (e0.initial, e0.recurrent), noise_seed=nseed)
    assert isinstance(sp2.searcher, MuZeroDeviceSearch)
    t2 = TrajectoryStore(e2, extra_slots=64)
    counters = np.zeros(G, np.int64)
    fin2 = []
    gum = torch.empty((G, A), dtype=torch.float64, device="cuda")
    for _ in range(40):
        for g in range(G):
            e2.fill_gumbel(gum[g], nseed, int((counters[g] * G + g) * A))
        pol, val, act, _ = sp2.search(gumbel=gum)
        e2.selfplay_step(pol, val, act, t2, True)
        counters += 1
        fin2 += t2.harvest()
    first1, first2 = {}, {}
    for r in fin1: first1.setdefault(r["game"], r)
    for r in fin2: first2.setdefault(r["game"], r)
    common = sorted(set(first1) & set(first2))
    assert len(common) >= 6
    for g in common:
        a, b = first1[g], first2[g]
        assert a["length"] == b["length"] and np.array_equal(a["actions"], b["actions"]) and a["winner"] == b["winner"], g
        assert np.array_equal(a["values"], b["values"]) and np.array_equal(a["policies"], b["policies"]), g
    with pytest.raises(ValueError):
        SelfPlayEngine(e2, lambda obs: None)
    # play() drives the same stepwise loop for a learned-dynamics evaluator (lock-step moves, sink per chunk)
    got, before = [], sp2.moves_played
    sp2.play(moves_per_game=5, traj=t2, sink=got.append, chunk=2)
    assert sp2.moves_played == before + 5 * G
    for pk in got:
        for i in range(len(pk)):
            r = pk.game(i)
            assert len(r) == int(pk.table[i][2]) and np.allclose(r["policy"].sum(axis=1), 1.0, atol=1e-12)
