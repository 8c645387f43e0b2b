"""Checkpoint and restore of the device replay ring (DeviceReplayBuffer.state_dict / load_state_dict; gmz_records_compact,
gmz_records_expand): the round trip through torch.save / torch.load at the same capacity is bit for bit, at another
capacity it keeps the newest records, the consistency check refuses a ring it could not rebuild, and the edge cases."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _per():
    """Prioritised replay on: priorities, max_priority and PER sampling are part of the saved state."""
    from datou_gomoku_muzero_b200.config import config
    saved = config.ENABLE_PER
    config.ENABLE_PER = True
    yield
    config.ENABLE_PER = saved


def _fill(N, G, S, cap, moves, roots=None, max_rounds=60, **eng_kw):
    """A DeviceReplayBuffer of `cap` records filled by persistent E0 self-play until the ring has wrapped and its oldest
    live game is cut.  Returns (buf, more): more() plays one more round and returns its PackedGames."""
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

    def more():
        got = []
        while not got:
            sp.play(moves_per_game=moves, traj=traj, sink=got.append)
        return got
    for _ in range(max_rounds):
        sp.play(moves_per_game=moves, traj=traj, sink=sink)
        if added[0] > cap and _host(buf)[buf.sum_tree.write_ptr]["t"] > 0:
            return buf, more
    raise AssertionError("the ring never wrapped with a cut oldest game")


def _host(buf):
    from datou_gomoku_muzero_b200.trajectory import record_dtype
    return buf.ring.cpu().numpy().view(record_dtype(buf.N)).reshape(-1)


def _body(buf):
    """The meaningful bytes of every ring position: 0 .. 64 + 21A (the tail padding is not record content)."""
    return buf.ring[:, :64 + 21 * buf.A]


def _round_trip(buf, tmp_path, capacity=None):
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    path = tmp_path / "ring.pt"
    torch.save(buf.state_dict(), path)
    out = DeviceReplayBuffer(buf.capacity if capacity is None else capacity, buf.N, unroll_steps=buf.unroll)
    out.load_state_dict(torch.load(path, weights_only=True))
    return out


def _assert_same(a, b):
    assert torch.equal(_body(a), _body(b))
    assert torch.equal(a.sum_tree.tree, b.sum_tree.tree)
    assert (a.sum_tree.write_ptr, a.sum_tree.count) == (b.sum_tree.write_ptr, b.sum_tree.count)
    assert torch.equal(a.max_priority, b.max_priority)


def _same_batches(a, b, B=64, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    for rot_k, flip in ((0, False), (1, True), (3, False)):
        u = torch.rand(B, dtype=torch.float64, device="cuda", generator=g)
        (ta, ia, wa), (tb, ib, wb) = a.sample(B, u01=u, rot_k=rot_k, flip=flip), b.sample(B, u01=u, rot_k=rot_k, flip=flip)
        assert torch.equal(ia, ib) and torch.equal(wa, wb)
        assert all(torch.equal(x, y) for x, y in zip(ta, tb))


def _train_a_little(buf, seed=3):
    """Priorities from random TD errors on sampled slices, as the trainer sets them."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    for _ in range(3):
        _, idx, _ = buf.sample(128, u01=torch.rand(128, dtype=torch.float64, device="cuda", generator=g))
        buf.update_priorities(idx, torch.randn(128, device="cuda", generator=g) * 2)


def test_round_trip_same_capacity(tmp_path):
    from datou_gomoku_muzero_b200.engine import SearchEngine
    N, S = 9, 16
    buf, more = _fill(N, 32, S, 1500, moves=27)
    wp, cap = buf.sum_tree.write_ptr, buf.capacity
    buf.reanalyse([SearchEngine(32, board_size=N, num_simulations=S, accum_dtype="float32")], first=(wp + cap // 2) % cap,
                  count=200, eval_seed=5, noise_seed=7)
    _train_a_little(buf)
    assert float(buf.max_priority) > 1.0
    out = _round_trip(buf, tmp_path)
    _assert_same(buf, out)
    _same_batches(buf, out)
    pos = torch.arange(cap, device="cuda")
    assert all(torch.equal(x, y) for x, y in zip(buf.batch(pos, 2, True), out.batch(pos, 2, True)))
    for pg in more():                                 # the same later appends keep both identical
        buf.add_packed(pg)
        out.add_packed(pg)
    _assert_same(buf, out)
    _same_batches(buf, out, seed=1)


def _white_to_move_roots(N, G, seed=5):
    A = N * N
    rs = np.random.RandomState(seed)
    boards = np.zeros((G, A), np.int8)
    last, mc = np.zeros(G, np.int32), np.zeros(G, np.int32)
    for g in range(G):
        k = 2 * int(rs.randint(2, 8)) + 1               # odd number of stones: white to move
        cells = rs.permutation(A)[:k]
        boards[g, cells[0::2]], boards[g, cells[1::2]] = 1, -1
        last[g], mc[g] = cells[-1], k
    return boards, -np.ones(G, np.int8), last, mc


@pytest.mark.parametrize("N,cap,moves,kw", [
    (6, 500, 12, dict(n_in_row=4)),
    (9, 1200, 27, dict(mode="MuZero")),
    (9, 400, 8, dict(white_to_move=True)),
    (15, 1200, 40, {}),
    (19, 1800, 40, {}),
])
def test_board_sizes_and_modes(tmp_path, N, cap, moves, kw):
    kw = dict(kw)
    roots = _white_to_move_roots(N, 32) if kw.pop("white_to_move", False) else None
    buf, _ = _fill(N, 32, 8, cap, moves=moves, roots=roots, **kw)
    if roots is not None:
        h = _host(buf)
        assert (h["to_move"] != np.where(h["t"] % 2 == 0, 1, -1)).sum() > 0     # games that began with white to move
    _train_a_little(buf)
    out = _round_trip(buf, tmp_path)
    _assert_same(buf, out)
    _same_batches(buf, out)


@pytest.mark.parametrize("factor", [2.0, 0.55])
def test_round_trip_other_capacity(tmp_path, factor):
    from datou_gomoku_muzero_b200.replay_buffer import SumTree
    N = 9
    buf, _ = _fill(N, 32, 8, 1000, moves=27)
    _train_a_little(buf)
    cap, n, wp = buf.capacity, len(buf), buf.sum_tree.write_ptr
    h = _host(buf)
    new_cap = int(cap * factor)
    while new_cap < n and h["t"][(wp + n - new_cap) % cap] == 0:         # a smaller ring: cut inside a game
        new_cap += 1
    out = _round_trip(buf, tmp_path, capacity=new_cap)
    kept = min(n, new_cap)
    old_pos = (wp + np.arange(n - kept, n)) % cap                        # the newest `kept`, oldest first
    assert (out.sum_tree.write_ptr, out.sum_tree.count) == (kept % new_cap, kept)
    assert torch.equal(_body(out)[:kept], _body(buf)[torch.as_tensor(old_pos, device="cuda")])
    assert not _body(out)[kept:].any()
    assert torch.equal(out.max_priority, buf.max_priority)
    ref = SumTree(new_cap)
    ref.add_many(buf.sum_tree.tree[torch.as_tensor(old_pos + cap - 1, device="cuda")])
    assert torch.equal(out.sum_tree.tree, ref.tree)
    # every kept slice: its successors in the game are newer, so they were kept too
    new_b = out.batch(torch.arange(kept, device="cuda"), 1, False)
    old_b = buf.batch(torch.as_tensor(old_pos, device="cuda"), 1, False)
    assert all(torch.equal(x, y) for x, y in zip(new_b, old_b))


@pytest.mark.parametrize("where", ["obs", "board"])
def test_consistency_check_refuses_an_altered_record(tmp_path, where):
    N = 6
    A = N * N
    buf, _ = _fill(N, 16, 8, 400, moves=12)
    h = _host(buf)
    p = int(np.flatnonzero((h["t"] > 2) & (np.arange(buf.capacity) != buf.sum_tree.write_ptr))[7])   # not a segment start
    col = 64 + 8 * A + 4 * (A + 5) + 3 if where == "obs" else 64 + 20 * A + 11      # a byte of the opponent plane / the board
    buf.ring[p, col] ^= 0x40 if where == "obs" else 0x01
    ring0, tree0 = buf.ring.clone(), buf.sum_tree.tree.clone()
    with pytest.raises(ValueError, match=f"ring position {p}\\b"):
        buf.state_dict()
    assert torch.equal(buf.ring, ring0) and torch.equal(buf.sum_tree.tree, tree0)


def test_edge_cases(tmp_path):
    from torch.profiler import ProfilerActivity, profile
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    empty = DeviceReplayBuffer(64, 6)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sd = empty.state_dict()
        fresh = DeviceReplayBuffer(64, 6)
        fresh.load_state_dict(sd)
        torch.cuda.synchronize()
    assert not [e.name for e in prof.events() if e.name.startswith("k_")]
    assert sd["count"] == 0 and sd["headers"].shape == (0, 64) and sd["base_boards"].shape == (0, 36)
    _assert_same(empty, fresh)
    again = _round_trip(empty, tmp_path)
    _assert_same(empty, again)
    # a board-size mismatch is refused before any device work
    buf, _ = _fill(6, 16, 8, 300, moves=12)
    sd = buf.state_dict()
    other = DeviceReplayBuffer(300, 9)
    ring0 = other.ring.clone()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with pytest.raises(ValueError, match="board size"):
            other.load_state_dict(sd)
        torch.cuda.synchronize()
    assert not [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert torch.equal(other.ring, ring0) and len(other) == 0
    # a ring that is not full, restored into a used buffer: positions that hold no live record are zeroed as in a new one
    big = DeviceReplayBuffer(2 * buf.capacity, 6)
    big.load_state_dict(sd)
    used = DeviceReplayBuffer(2 * buf.capacity, 6)
    used.ring.fill_(0x5a)
    used.load_state_dict(big.state_dict())
    _assert_same(big, used)
    assert not _body(used)[len(used):].any()
