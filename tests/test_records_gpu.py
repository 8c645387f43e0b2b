"""Device-side trajectory hand-off on the GPU: gmz_traj_pack against what the reference's universal_worker emitted
(goldens), the device replay ring (PER tree + packed records) against the reference buffer's semantics restated with the
oracle, and long self-play runs through a sink without parking."""
import os

import numpy as np
import pytest

from _golden_util import GOLDEN_DIR
from test_packed_records_cpu import NAMES

pytestmark = pytest.mark.gpu


def _load_game(traj, slot, z, game=0):
    import torch
    T = len(z["actions"])
    traj.policy[slot, :T] = torch.from_numpy(z["policies"]).cuda()
    traj.value[slot, :T] = torch.from_numpy(z["search_values"]).cuda()
    traj.action[slot, :T] = torch.from_numpy(z["actions"]).cuda()
    traj.start_board[slot].zero_()
    traj.start_info[slot] = torch.tensor([1, 0, -1, game], dtype=torch.int32).cuda()
    return T


@pytest.mark.parametrize("name", NAMES)
def test_pack_kernel_matches_reference_game_record(name):
    """Records written by gmz_traj_pack == observations / boards / policies / rewards / n-step value targets of the
    GameRecord the reference's universal_worker produced, bit for bit (incl. the float32-valued games), and the
    trainer batches gathered from them in a DeviceReplayBuffer == the TrainingSlices it cut."""
    import torch
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    N, U, n_steps = int(z["params"][0]), int(z["params"][5]), int(z["params"][6])
    saved = (config.DISCOUNT, config.N_STEPS, config.NUM_UNROLL_STEPS)
    config.DISCOUNT, config.N_STEPS, config.NUM_UNROLL_STEPS = float(z["discount"]), n_steps, U
    try:
        eng = SearchEngine(4, board_size=N, num_simulations=8)
        traj = TrajectoryStore(eng, extra_slots=8)
        T = _load_game(traj, 6, z, game=3)
        T2 = _load_game(traj, 9, z, game=1)          # the same game twice: two CTAs, two offsets
        traj.fin_queue[0] = torch.tensor([6, 3, T, int(z["winner"])], dtype=torch.int32).cuda()
        traj.fin_queue[1] = torch.tensor([9, 1, T2, int(z["winner"])], dtype=torch.int32).cuda()
        traj.fin_count.fill_(2)
        free0 = traj.free_slots_left()
        pg = traj.pack_finished(recycle=True)
        assert len(pg) == 2 and pg.n_moves == 2 * T and traj.free_slots_left() == free0 + 2 and int(traj.fin_count.item()) == 0
        for i, (slot, game) in enumerate([(6, 3), (9, 1)]):
            r = pg.game(i)
            assert np.array_equal(r["obs"], z["observations"]) and np.array_equal(r["board"], z["boards"])
            assert np.array_equal(r["policy"], z["policies"]) and np.array_equal(r["action"], z["actions"])
            assert np.array_equal(r["reward"].astype(np.float64), z["rewards"])
            assert np.array_equal(r["value_target"], z["values_targets"].astype(np.float32))
            assert np.array_equal(r["search_value"], z["search_values"])
            assert (r["t"] == np.arange(T)).all() and (r["length"] == T).all() and (r["winner"] == int(z["winner"])).all()
            assert (r["game"] == game).all() and (r["slot"] == slot).all() and (r["game_seq"] == i).all()
            assert (r["move_count"] == np.arange(T)).all() and (r["to_move"] == np.where(np.arange(T) % 2 == 0, 1, -1)).all()
            assert np.array_equal(r["last_move"], np.concatenate([[-1], z["actions"][:-1]]))
        sl = pg.training_slices(1)
        assert np.array_equal(np.stack([s.observation for s in sl]), z["slice_obs"])
        assert np.array_equal(np.stack([s.value_history for s in sl]), z["slice_val"])
        # the device ring's batches of both games == the TrainingSlices the reference cut, bit for bit, same dtypes
        buf = DeviceReplayBuffer(pg.n_moves, N)
        buf.add_packed(pg)
        batch = [x.cpu().numpy() for x in buf.batch(torch.arange(pg.n_moves, device="cuda"))]
        for part in (slice(0, T), slice(T, 2 * T)):
            for got, key in zip(batch, ("slice_obs", "slice_act", "slice_rew", "slice_pi", "slice_val")):
                assert got.dtype == z[key].dtype and np.array_equal(got[part], z[key]), key
    finally:
        config.DISCOUNT, config.N_STEPS, config.NUM_UNROLL_STEPS = saved


def test_device_replay_buffer_follows_reference_buffer_semantics():
    """DeviceReplayBuffer (ring of records + device SumTree) vs the reference's InMemoryReplayBuffer restated with the
    oracle's SumTree over the slices the records imply: same tree (bit-exact float64), same sampled indices and
    weights, same batch tensors, through ring wrap-around, priority updates and D4 augmentation."""
    import torch
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    from oracle import oracle
    N, S, G, U = 6, 16, 16, 5
    saved = (config.NUM_UNROLL_STEPS, config.ENABLE_PER)
    config.NUM_UNROLL_STEPS, config.ENABLE_PER = U, True
    try:
        eng = SearchEngine(G, board_size=N, num_simulations=S)
        sp = SelfPlayEngine(eng, "e0", seed=4, noise_seed=5)
        traj = TrajectoryStore(eng, extra_slots=32)
        cap = 300                                            # small: the ring wraps several times
        buf = DeviceReplayBuffer(cap, N)
        ref_tree, ref_data, maxp = oracle.SumTree(cap), [None] * cap, 1.0
        rs = np.random.RandomState(1)
        rounds = 0
        for it in range(8):
            sp.play(moves_per_game=12, traj=traj)
            pg = traj.pack_finished()
            if pg is None:
                continue
            buf.add_packed(pg)
            for i in range(len(pg)):                         # the reference adds slice by slice (workers.py:399-407)
                for sl in pg.training_slices(i):
                    ref_data[ref_tree.write_ptr] = sl
                    ref_tree.add(maxp)
            assert buf.sum_tree.write_ptr == ref_tree.write_ptr and len(buf) == ref_tree.count
            assert np.array_equal(buf.sum_tree.tree.cpu().numpy(), ref_tree.tree)
            if len(buf) < 32:
                continue
            B = 32
            u = rs.random_sample(B)
            k, fl = int(rs.randint(4)), bool(rs.randint(2))
            (obs, act, rew, pi, val), idx, w = buf.sample(B, u01=torch.from_numpy(u).cuda(), rot_k=k, flip=fl)
            ridx, rpr, rw = ref_tree.sample(B, u, config.PER_BETA)
            assert np.array_equal(idx.cpu().numpy(), ridx)
            np.testing.assert_allclose(w.cpu().numpy(), rw, rtol=1e-6)
            sl = [ref_data[int(i) - cap + 1] for i in ridx]
            o0 = np.stack([s.observation for s in sl]); a0 = np.stack([s.action_history for s in sl])
            p0 = np.stack([s.policy_history for s in sl])
            eo, ea, ep = oracle.augment_batch(o0, a0, p0, k, fl)
            assert np.array_equal(obs.cpu().numpy(), eo) and np.array_equal(pi.cpu().numpy(), ep)
            got_a = act.cpu().numpy()
            assert np.array_equal(got_a[a0 != -1], ea[a0 != -1]) and (got_a[a0 == -1] == -1).all()
            assert np.array_equal(rew.cpu().numpy(), np.stack([s.reward_history for s in sl]))
            assert np.array_equal(val.cpu().numpy(), np.stack([s.value_history for s in sl]))
            td = (rs.randn(B) * 2).astype(np.float32)
            buf.update_priorities(idx, torch.from_numpy(td).cuda())
            pri = np.abs(td) + np.float32(config.PER_EPSILON)
            maxp = ref_tree.update_batch(ridx, pri.astype(np.float64), maxp)
            assert np.array_equal(buf.sum_tree.tree.cpu().numpy(), ref_tree.tree)
            assert float(buf.max_priority.item()) == maxp
            rounds += 1
        assert rounds >= 3 and ref_tree.count == cap             # wrapped
        # get_leaf (replay_buffer.py:27-38): device descent == oracle descent
        for v in rs.uniform(0, ref_tree.tree[0], 20):
            assert buf.sum_tree.get_leaf(v) == ref_tree.get_leaf(v)
    finally:
        config.NUM_UNROLL_STEPS, config.ENABLE_PER = saved


def test_long_selfplay_run_through_a_sink_never_parks():
    """play(sink=...) cuts a long run into launches sized to the spare trajectory slots and recycles them on the
    device in between: no game parks, every finished game arrives, every move is accounted for."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    N, S, G = 6, 12, 64
    eng = SearchEngine(G, board_size=N, num_simulations=S)
    sp = SelfPlayEngine(eng, "e0", seed=1, noise_seed=2)
    traj = TrajectoryStore(eng, extra_slots=16)
    buf = DeviceReplayBuffer(50_000, N)
    got = []
    def sink(pg):
        got.append((len(pg), pg.n_moves)); buf.add_packed(pg)
    sp.play(moves_per_game=150, traj=traj, sink=sink)
    moves, nfin = eng.play_counters()
    assert moves == G * 150 and eng.tickets_unserved == 0 and eng.tickets_idle == 0
    assert sum(g for g, _ in got) == nfin and nfin > 3 * G and len(got) > 10
    assert len(buf) == sum(m for _, m in got) <= moves


def test_reanalysis_writeback_into_the_device_ring():
    """DeviceReplayBuffer.rewrite_targets = the re-analysis write-back (db_manager.py:189-214) for records resident on
    the device: after it, the batches built from the ring carry exactly the windows `writeback_windows` produces for the
    new policies / value targets, and nothing else of the records changes."""
    import torch
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.reanalysis import writeback_windows
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    N, S, G = 6, 12, 16
    A, U = N * N, int(config.NUM_UNROLL_STEPS)
    eng = SearchEngine(G, board_size=N, num_simulations=S)
    sp = SelfPlayEngine(eng, "e0", seed=4, noise_seed=5)
    traj = TrajectoryStore(eng, extra_slots=32)
    buf = DeviceReplayBuffer(4096, N)
    packs = []
    sp.play(moves_per_game=40, traj=traj, sink=lambda pg: (packs.append(pg), buf.add_packed(pg)))
    pg = packs[0]
    assert len(pg) >= 1
    T = int(pg.offsets[1] - pg.offsets[0])                       # first game of the first pack sits at ring positions 0 .. T-1
    before = buf.ring[:T + 3].clone()
    rs = np.random.RandomState(9)
    new_pol = rs.dirichlet(np.ones(A), size=T)
    new_val = rs.uniform(-1, 1, T).astype(np.float32)
    buf.rewrite_targets(np.arange(T), new_pol, new_val)
    obs, act, rew, pi, val = buf.batch(torch.arange(T, device="cuda"))
    pw, vw = writeback_windows(new_pol, new_val.tolist(), unroll_steps=U)
    assert np.array_equal(pi.cpu().numpy(), pw) and np.array_equal(val.cpu().numpy(), vw)
    after = buf.ring[:T + 3]
    changed = (after != before).any(dim=0).nonzero().flatten().cpu().numpy()
    assert set(changed) <= set(range(36, 40)) | set(range(64, 64 + 8 * A))      # only value_target and policy bytes
    assert torch.equal(after[T:], before[T:])                                   # the next game's records are untouched
    with pytest.raises(ValueError):
        buf.rewrite_targets([buf.capacity], new_pol[:1], new_val[:1])
