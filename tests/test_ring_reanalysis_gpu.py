"""Re-analysis of the device replay ring in place (DeviceReplayBuffer.reanalyse; gmz_set_roots_from_records,
gmz_records_writeback, gmz_records_retarget): the same policies, root values and value targets as the host driver
(records -> roots -> reanalyse_positions -> per-game n-step targets with float32 rewards), whole-game widening, batching
independence, mid-game starts, every board size, a network evaluator, and the edge cases."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _fill(N, G, S, cap, moves, roots=None, max_rounds=60, **eng_kw):
    """A DeviceReplayBuffer of `cap` records filled by persistent E0 self-play until the ring has wrapped and its oldest
    live game is cut (its first moves overwritten)."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng = SearchEngine(G, board_size=N, num_simulations=S, **eng_kw)
    sp = SelfPlayEngine(eng, "e0", seed=11, noise_seed=12)
    if roots is not None:
        eng.set_roots(*roots)
    traj = TrajectoryStore(eng, extra_slots=G)
    buf = DeviceReplayBuffer(cap, N)
    added = [0]

    def sink(pg):
        buf.add_packed(pg)
        added[0] += pg.n_moves
    for _ in range(max_rounds):
        sp.play(moves_per_game=moves, traj=traj, sink=sink)
        if added[0] > cap and _host(buf)[buf.sum_tree.write_ptr]["t"] > 0:
            return buf
    raise AssertionError("the ring never wrapped with a cut oldest game")


def _host(buf):
    from datou_gomoku_muzero_b200.trajectory import record_dtype
    return buf.ring.cpu().numpy().view(record_dtype(buf.N)).reshape(-1)


def _engines(N, Gs, S, **kw):
    from datou_gomoku_muzero_b200.engine import SearchEngine
    return [SearchEngine(G, board_size=N, num_simulations=S, **kw) for G in Gs]


def _games(r):
    """Split consecutive records of a stretch into games: [(lo, hi)] index ranges."""
    starts = [0] + [k for k in range(1, len(r)) if r["t"][k] == 0]
    return list(zip(starts, starts[1:] + [len(r)]))


def _expected(snap, start, n, engines, evaluator="e0", eval_seed=0, noise_seed=0, cls=None):
    """The host driver on the snapshot: roots from the record headers and boards -> reanalyse_positions on fresh engines
    -> per game the float32 restatement of workers.py:291-292 (tests/test_selfplay_gpu.py).  Returns (policies, values,
    value targets float32) of the n records from ring position start."""
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.reanalysis import reanalyse_positions
    cap = len(snap)
    r = snap[(start + np.arange(n)) % cap]
    A = r["policy"].shape[1]
    pol, val = reanalyse_positions(engines, r["board"].reshape(n, A), r["to_move"].astype(np.int8), r["last_move"],
                                   r["move_count"], evaluator=evaluator, eval_seed=eval_seed, noise_seed=noise_seed, cls=cls)
    vt = np.zeros(n, np.float32)
    ns, d = config.N_STEPS, config.DISCOUNT
    for lo, hi in _games(r):
        rew = r["reward"][lo:hi].astype(np.float32)
        v32 = val[lo:hi].astype(np.float32)
        T = hi - lo
        for t in range(T):
            acc = sum((d ** i) * rew[t + i] for i in range(ns) if t + i < T)
            boot = v32[t + ns] * (d ** ns) if t + ns < T else 0.0
            vt[lo + t] = acc + boot
    return pol, val, vt


def _changed_bytes_only_targets(before, after, A, touched):
    """Every byte outside the policy / search_value / value_target of the `touched` ring positions is unchanged."""
    b = before.view(np.uint8).reshape(len(before), -1).copy()
    a = after.view(np.uint8).reshape(len(after), -1).copy()
    for x in (a, b):
        x[touched, 36:48] = 0                  # value_target f32, pad, search_value f64
        x[touched, 64:64 + 8 * A] = 0          # policy f64[A]
    assert np.array_equal(a, b)


def _check_parity(buf, snap, tree0, start, n, pol, val, vt):
    from datou_gomoku_muzero_b200.reanalysis import writeback_windows
    import torch
    cap, A = buf.capacity, buf.A
    after = _host(buf)
    pos = (start + np.arange(n)) % cap
    r = after[pos]
    assert np.array_equal(r["policy"], pol)
    assert np.array_equal(r["search_value"], val)
    assert np.array_equal(r["value_target"], vt)
    _changed_bytes_only_targets(snap, after, A, pos)
    assert torch.equal(buf.sum_tree.tree, tree0)
    _, _, _, pi, v = (x.cpu().numpy() for x in buf.batch(torch.as_tensor(pos, device=buf.device)))
    for lo, hi in _games(r):
        pw, vw = writeback_windows(pol[lo:hi], vt[lo:hi], buf.unroll)
        assert np.array_equal(pi[lo:hi], pw) and np.array_equal(v[lo:hi], vw)


@pytest.mark.parametrize("N,mode,accum", [(6, "AlphaZero", "float64"), (9, "AlphaZero", "float32"), (6, "MuZero", "float64"),
                                          (9, "AlphaZero", "float64")])
def test_reanalyse_matches_host_driver(N, mode, accum):
    from datou_gomoku_muzero_b200.mcts import AlphaZeroMCTS, MuZeroMCTS
    S, G = 16, 24
    buf = _fill(N, 32, S, 700 if N == 6 else 1500, moves=N * N // 3)
    snap, tree0 = _host(buf), buf.sum_tree.tree.clone()
    kw = dict(mode=mode, accum_dtype=accum)
    start, n = buf.reanalyse(_engines(N, (G, G), S, **kw), eval_seed=5, noise_seed=7)
    assert (start, n) == (buf.sum_tree.write_ptr, buf.capacity)          # wrapped ring: every record, oldest first
    pol, val, vt = _expected(snap, start, n, _engines(N, (G, G), S, **kw), eval_seed=5, noise_seed=7,
                             cls=MuZeroMCTS if mode == "MuZero" else AlphaZeroMCTS)
    assert not np.array_equal(pol, snap["policy"][(start + np.arange(n)) % buf.capacity])   # the new evaluator moved them
    _check_parity(buf, snap, tree0, start, n, pol, val, vt)


def test_explicit_stretch_widens_to_whole_games():
    import torch
    N, S = 9, 16
    buf = _fill(N, 32, S, 1500, moves=27)
    snap, cap, wp = _host(buf), buf.capacity, buf.sum_tree.write_ptr
    rel = (np.arange(cap) - wp) % cap                 # age order: 0 = oldest live record
    mid = int(np.flatnonzero((rel > cap // 3) & (rel < 2 * cap // 3) & (snap["t"] > 0) & (snap["t"] < snap["length"] - 1))[0])
    t, T = int(snap["t"][mid]), int(snap["length"][mid])
    start, n = buf.reanalyse(_engines(N, (16,), S), first=mid, count=1, eval_seed=5, noise_seed=3)
    assert (start, n) == ((mid - t) % cap, T)
    game = (start + np.arange(n)) % cap
    after = _host(buf)
    changed = np.flatnonzero((after.view(np.uint8).reshape(cap, -1) != snap.view(np.uint8).reshape(cap, -1)).any(1))
    assert set(changed.tolist()) <= set(game.tolist()) and len(changed) > 0
    _changed_bytes_only_targets(snap, after, buf.A, game)
    pol, val, vt = _expected(snap, start, n, _engines(N, (16,), S), eval_seed=5, noise_seed=3)
    assert np.array_equal(after["policy"][game], pol) and np.array_equal(after["value_target"][game], vt)
    # a stretch starting inside the cut oldest game starts at write_ptr and covers that game's live suffix
    buf.ring.copy_(torch.from_numpy(snap.view(np.uint8).reshape(cap, -1)).to(buf.device))
    cut_t, cut_T = int(snap["t"][wp]), int(snap["length"][wp])
    inside = (wp + min(1, cut_T - cut_t - 1)) % cap
    start, n = buf.reanalyse(_engines(N, (16,), S), first=inside, count=1, eval_seed=5, noise_seed=3)
    assert (start, n) == (wp, cut_T - cut_t)


def test_batching_does_not_matter():
    import torch
    N, S = 6, 16
    buf = _fill(N, 32, S, 700, moves=12)
    snap = buf.ring.clone()
    n = len(buf)
    outs = []
    assert n % 16 and n % 29                          # every run ends with a partial batch
    for Gs in ((16,), (16, 16, 16), (29, 29)):
        buf.ring.copy_(snap)
        assert buf.reanalyse(_engines(N, Gs, S), eval_seed=8, noise_seed=9) == (buf.sum_tree.write_ptr, n)
        outs.append(buf.ring.clone())
    assert not torch.equal(outs[0], snap)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


def test_mid_game_starts_take_the_colour_from_the_header():
    from datou_gomoku_muzero_b200.engine import SearchEngine
    N, G, S = 9, 32, 16
    A = N * N
    rs = np.random.RandomState(5)
    boards = np.zeros((G, A), np.int8)
    last, mc = np.zeros(G, np.int32), np.zeros(G, np.int32)
    for g in range(G):
        k = 2 * int(rs.randint(2, 8)) + 1               # odd number of stones: white to move
        cells = rs.permutation(A)[:k]
        boards[g, cells[0::2]], boards[g, cells[1::2]] = 1, -1
        last[g], mc[g] = cells[-1], k
    buf = _fill(N, G, S, 400, moves=8, roots=(boards, -np.ones(G, np.int8), last, mc))
    snap, tree0 = _host(buf), buf.sum_tree.tree.clone()
    parity = np.where(snap["t"] % 2 == 0, 1, -1)
    assert (snap["to_move"] != parity).sum() > 0 and (snap["move_count"] != snap["t"]).sum() > 0
    start, n = buf.reanalyse(_engines(N, (16, 16), S), eval_seed=4, noise_seed=6)
    pol, val, vt = _expected(snap, start, n, _engines(N, (16, 16), S), eval_seed=4, noise_seed=6)
    _check_parity(buf, snap, tree0, start, n, pol, val, vt)


@pytest.mark.parametrize("N", [15, 19])
def test_larger_boards(N):
    S, G = 8, 32
    buf = _fill(N, 32, S, 1200 if N == 15 else 1800, moves=40)
    snap, tree0 = _host(buf), buf.sum_tree.tree.clone()
    start, n = buf.reanalyse(_engines(N, (G, G), S), eval_seed=2, noise_seed=1)
    pol, val, vt = _expected(snap, start, n, _engines(N, (G, G), S), eval_seed=2, noise_seed=1)
    _check_parity(buf, snap, tree0, start, n, pol, val, vt)


def test_network_evaluator():
    import torch
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.network import GomokuNetEZ
    N, S, G = 6, 8, 32
    torch.manual_seed(0)
    net = GomokuNetEZ(Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=N * N, NUM_RES_BLOCKS=1, NUM_FILTERS=16, HEAD_HIDDEN_DIM=8)).cuda().eval()

    @torch.no_grad()
    def ev(obs):
        lg, v, _ = net.initial_inference(obs)
        return lg.float().contiguous(), v.float().reshape(-1).contiguous()
    buf = _fill(N, 32, S, 500, moves=12)
    snap, tree0 = _host(buf), buf.sum_tree.tree.clone()
    saved = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    try:
        start, n = buf.reanalyse(_engines(N, (G, G), S, accum_dtype="float32"), evaluator=ev, noise_seed=2)
        pol, val, vt = _expected(snap, start, n, _engines(N, (G, G), S, accum_dtype="float32"), evaluator=ev, noise_seed=2)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = saved
    _check_parity(buf, snap, tree0, start, n, pol, val, vt)
    with pytest.raises(ValueError):
        buf.reanalyse(_engines(N, (G,), S, mode="MuZero"), evaluator=ev)


def test_edge_cases():
    import torch
    from torch.profiler import ProfilerActivity, profile
    from datou_gomoku_muzero_b200 import _lib
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    N, S = 6, 8
    eng = _engines(N, (8,), S)[0]
    empty = DeviceReplayBuffer(64, N)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        assert empty.reanalyse([eng]) == (0, 0)
        torch.cuda.synchronize()
    assert not [e.name for e in prof.events() if e.name.startswith("k_")]
    with pytest.raises(ValueError):
        empty.reanalyse([eng], first=0, count=1)
    buf = _fill(N, 16, S, 300, moves=12)
    cap, wp = buf.capacity, buf.sum_tree.write_ptr
    for first, count in ((wp, cap + 1), ((wp + 5) % cap, cap - 4), (cap, 1), (-1, 1), (wp, -1)):
        with pytest.raises(ValueError):
            buf.reanalyse([eng], first=first, count=count)
    with pytest.raises(ValueError):
        buf.reanalyse(_engines(9, (8,), S))
    with pytest.raises(ValueError):
        buf.reanalyse([eng], evaluator="e1")
    # the roots call with a live engine: n > G is rejected, n = 0 leaves the roots alone
    lib = _lib.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.gmz_set_roots_from_records(eng.handle, C.c_void_p(buf.ring.data_ptr()), cap, 0, eng.G + 1, st) != 0
    assert b"gmz_set_roots_from_records" in lib.gmz_last_error() and b"num_games" in lib.gmz_last_error()
    eng.reset_games()
    before = [x.clone() for x in eng.get_roots()]
    assert lib.gmz_set_roots_from_records(eng.handle, C.c_void_p(buf.ring.data_ptr()), cap, 0, 0, st) == 0
    assert all(torch.equal(a, b) for a, b in zip(before, eng.get_roots()))


def test_roots_from_records_equal_set_roots():
    """gmz_set_roots_from_records == gmz_set_roots fed with the records' boards and header fields (padding: full boards)."""
    import torch
    N, S, G = 9, 16, 32
    buf = _fill(N, 16, S, 400, moves=20)
    snap = _host(buf)
    a, b = _engines(N, (G, G), S)
    k, first = 27, (buf.sum_tree.write_ptr + 300) % buf.capacity
    r = snap[(first + np.arange(k)) % buf.capacity]
    a.set_roots_from_records(buf.ring, buf.capacity, first, k)
    bd = np.ones((G, N * N), np.int8); pl = np.ones(G, np.int8); lm = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    bd[:k], pl[:k], lm[:k], mc[:k] = r["board"].reshape(k, -1), r["to_move"], r["last_move"], r["move_count"]
    b.set_roots(bd, pl, lm, mc)
    assert all(torch.equal(x, y) for x, y in zip(a.get_roots(), b.get_roots()))
    gum = torch.from_numpy(np.random.RandomState(0).gumbel(0, 1, (G, N * N))).cuda()
    outs = []
    for e in (a, b):
        e.search_e0(gum, 3)
        outs.append([x.clone() for x in e.finalize()])
    assert all(torch.equal(x, y) for x, y in zip(*outs))
    assert (outs[0][2][k:] == -1).all()                  # padding games are inactive
