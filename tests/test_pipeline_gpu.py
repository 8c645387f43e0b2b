"""End-to-end on the device with a real (small) GomokuNetEZ: network-driven self-play -> trajectory
store -> packed move records -> device replay ring -> PER sampling -> trainer batch tuple, i.e. universal_worker +
inference_server_worker + data_loader_worker (workers.py:129-439) without a host hop in the data path."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_network_selfplay_to_training_batch():
    import torch
    from datou_gomoku_muzero_b200.config import Config, config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.network import DeviceEvaluator, GomokuNetEZ
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.tactics import missed_win_stats
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    N, S, G = 6, 16, 32
    A = N * N
    torch.manual_seed(0)
    net = GomokuNetEZ(Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=A, NUM_RES_BLOCKS=2, NUM_FILTERS=16, HEAD_HIDDEN_DIM=8))
    eng = SearchEngine(G, board_size=N, num_simulations=S)
    ev = DeviceEvaluator(net, eng.leaf_obs, dtype=torch.float32, graph=True)
    sp = SelfPlayEngine(eng, ev, noise_seed=1)
    traj = TrajectoryStore(eng, extra_slots=96)
    saved = (config.ENABLE_PER, config.N_IN_ROW)
    config.ENABLE_PER = True
    try:
        cap = 4096                                            # more than G games can record: the ring does not wrap
        buf = DeviceReplayBuffer(cap, N)
        packs = []
        for _ in range(A):
            sp.step(traj=traj)
            pg = traj.pack_finished()
            if pg is not None:
                packs.append(pg)
                buf.add_packed(pg)
            if sum(len(p) for p in packs) >= 6:
                break
        rec = np.concatenate([p.host() for p in packs])       # ring position k holds rec[k]
        assert sum(len(p) for p in packs) >= 6 and len(buf) == len(rec) < cap
        for pg in packs:                                      # a finished game is a legal Gomoku game
            for i in range(len(pg)):
                r = pg.game(i)
                assert len(set(r["action"].tolist())) == int(r["length"][0]) == len(r) and int(r["winner"][0]) in (-1, 0, 1)
                np.testing.assert_allclose(r["policy"].sum(1), 1.0, atol=1e-9)
        (obs, act, rew, pi, val), idx, w = buf.sample(16)
        U = config.NUM_UNROLL_STEPS
        assert obs.shape == (16, U + 1, 3, N, N) and act.shape == (16, U) and pi.shape == (16, U + 1, A)
        assert obs.dtype == torch.float32 and pi.dtype == torch.float64 and val.dtype == torch.float32 and w.dtype == torch.float32
        for b, p in enumerate((idx - (cap - 1)).tolist()):    # first unrolled action / policy are the record's own
            assert int(act[b, 0]) == int(rec[p]["action"])
            assert np.array_equal(pi[b, 0].cpu().numpy(), rec[p]["policy"])
        buf.update_priorities(idx, np.abs(np.random.RandomState(0).randn(16)).astype(np.float32))
        assert abs(buf.sum_tree.total_priority() - float(buf.sum_tree.tree[cap - 1:].sum())) < 1e-9
        gr = packs[0].game_record(0)
        mf, mt = missed_win_stats(gr)
        assert 0 <= mf <= mt <= len(gr.actions)
    finally:
        config.ENABLE_PER, config.N_IN_ROW = saved
