"""Re-analysis with the production evaluators (mcts.resolve_searchers): learned dynamics (MuZeroDeviceSearch with per-game
node budgets in a compact arena) and graph-captured NetworkSearch, on the ring route (DeviceReplayBuffer.reanalyse) and
the host route (reanalyse_positions), against the fused E0 kernel and against each other."""
import warnings

import numpy as np
import pytest

from test_ring_reanalysis_gpu import _check_parity, _engines, _expected, _fill, _host

pytestmark = pytest.mark.gpu

S = 32


def _e0_pair(N, seed):
    from datou_gomoku_muzero_b200.muzero import TorchE0
    e0 = TorchE0(N, seed=seed)
    return e0.initial, e0.recurrent


def _mz(engines, initial, recurrent, **kw):
    from datou_gomoku_muzero_b200.muzero import MuZeroDeviceSearch
    return [MuZeroDeviceSearch(e, initial, recurrent, graph=True, **kw) for e in engines]


def _needed_rows(snap, start, n, engines):
    """Host restatement of the arena size: per engine, the largest batch sum of (evals_per_search(S, K, min(K, empty)) + 1)
    over its batches, one row per padding game."""
    from datou_gomoku_muzero_b200.muzero import evals_per_search
    r = snap[(start + np.arange(n)) % len(snap)]
    empty = (r["board"].reshape(n, -1) == 0).sum(1)
    need, s0, b = [0] * len(engines), 0, 0
    while s0 < n:
        i = b % len(engines)
        e = engines[i]
        k = min(e.G, n - s0)
        rows = sum(evals_per_search(e.S, e.K, min(e.K, int(x))) + 1 for x in empty[s0:s0 + k]) + (e.G - k)
        need[i] = max(need[i], rows)
        s0, b = s0 + k, b + 1
    return need


def _net(N, seed=0):
    import torch
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.network import GomokuNetEZ
    torch.manual_seed(seed)
    net = GomokuNetEZ(Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=N * N, NUM_RES_BLOCKS=1, NUM_FILTERS=16, HEAD_HIDDEN_DIM=8)).cuda()
    with torch.no_grad():                      # non-trivial BatchNorm statistics, so every folded tensor matters
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.weight.uniform_(0.5, 1.5); m.running_mean.uniform_(-0.1, 0.1); m.running_var.uniform_(0.5, 1.5)
    return net.eval()


def _mz_net(N, net):
    import torch
    from datou_gomoku_muzero_b200.muzero import FoldedRecurrentInference
    from datou_gomoku_muzero_b200.network import FoldedInitialInference
    fi, fr = FoldedInitialInference(net, torch.bfloat16), FoldedRecurrentInference(net, torch.bfloat16)

    def initial(obs):
        p, v, h = fi(obs.to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
        return p.float().contiguous(), v.reshape(-1).float(), h
    return initial, fr


class _Deterministic:
    def __enter__(self):
        import torch
        self.saved = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False

    def __exit__(self, *exc):
        import torch
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = self.saved


@pytest.mark.parametrize("N,accum", [(6, "float64"), (6, "float32"), (9, "float64"), (9, "float32")])
def test_learned_dynamics_equal_fused_kernel(N, accum):
    import torch
    buf = _fill(N, 32, S, 700 if N == 6 else 1500, moves=N * N // 3)
    snap = buf.ring.clone()
    h = _host(buf)
    if N == 6:                                                     # budgets above the k = K case are exercised
        assert ((h["board"].reshape(len(h), -1) == 0).sum(1) < 16).sum() > 0
    kw = dict(mode="MuZero", accum_dtype=accum)
    start, n = buf.reanalyse(_engines(N, (24, 24), S, **kw), evaluator="e0", eval_seed=5, noise_seed=7)
    fused = buf.ring.clone()
    assert not torch.equal(fused, snap)
    buf.ring.copy_(snap)
    engines = _engines(N, (24, 24), S, **kw)
    searchers = _mz(engines, *_e0_pair(N, 5))
    assert buf.reanalyse(engines, evaluator=searchers, noise_seed=7) == (start, n)
    assert torch.equal(buf.ring, fused)
    assert all(int(s.overflow) == 0 for s in searchers)
    need = _needed_rows(_host(buf), start, n, engines)
    assert [s.pool.shape[0] for s in searchers] == need
    assert sum(need) < sum(e.G * e.S for e in engines)


@pytest.mark.parametrize("kind", ["e0_pair", "muzero_net", "alphazero_net"])
def test_host_route_equals_ring_route(kind):
    import torch
    from datou_gomoku_muzero_b200.mcts import AlphaZeroMCTS, MuZeroMCTS
    from datou_gomoku_muzero_b200.network import NetworkSearch
    N, G = 6, 24
    buf = _fill(N, 32, S, 600, moves=12)
    snap, tree0 = _host(buf), buf.sum_tree.tree.clone()
    with _Deterministic():
        if kind == "alphazero_net":
            engines = _engines(N, (G, G), S, accum_dtype="float32")
            searchers = [NetworkSearch(e, _net(N)) for e in engines]
        else:
            engines = _engines(N, (G, G), S, mode="MuZero", accum_dtype="float64" if kind == "e0_pair" else "float32")
            searchers = _mz(engines, *(_e0_pair(N, 3) if kind == "e0_pair" else _mz_net(N, _net(N))))
        torch.backends.cudnn.benchmark = False                     # NetworkSearch switches it on
        start, n = buf.reanalyse(engines, evaluator=searchers, eval_seed=3, noise_seed=4)
        pol, val, vt = _expected(snap, start, n, engines, evaluator=searchers, eval_seed=3, noise_seed=4,
                                 cls=AlphaZeroMCTS if kind == "alphazero_net" else MuZeroMCTS)
    _check_parity(buf, snap, tree0, start, n, pol, val, vt)
    assert not np.array_equal(pol, snap["policy"][(start + np.arange(n)) % buf.capacity])
    if kind != "alphazero_net":
        assert all(int(s.overflow) == 0 for s in searchers)


def test_batching_does_not_matter():
    import torch
    N = 6
    buf = _fill(N, 32, S, 700, moves=12)
    snap = buf.ring.clone()
    n = len(buf)
    assert n % 16 and n % 29                                       # every run ends with a partial batch
    outs = []
    for Gs in ((16,), (16, 16, 16), (29, 29)):
        buf.ring.copy_(snap)
        engines = _engines(N, Gs, S, mode="MuZero")
        searchers = _mz(engines, *_e0_pair(N, 8))
        assert buf.reanalyse(engines, evaluator=searchers, noise_seed=9) == (buf.sum_tree.write_ptr, n)
        assert all(int(s.overflow) == 0 for s in searchers)
        assert [s.pool.shape[0] for s in searchers] == _needed_rows(_host(buf), buf.sum_tree.write_ptr, n, engines)
        outs.append(buf.ring.clone())
    assert not torch.equal(outs[0], snap)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


def test_rejected_inputs_touch_nothing():
    import torch
    from torch.profiler import ProfilerActivity, profile
    from datou_gomoku_muzero_b200.network import NetworkSearch
    N, G = 6, 16
    buf = _fill(N, 16, S, 300, moves=12)
    snap = buf.ring.clone()
    az, mz = _engines(N, (G,), S), _engines(N, (G, G), S, mode="MuZero")
    pair, net = _e0_pair(N, 1), _net(N)

    def ev(obs):
        return torch.zeros((obs.shape[0], N * N), device=obs.device), torch.zeros(obs.shape[0], device=obs.device)
    other = _engines(N, (G,), S, mode="MuZero")[0]
    cases = [(mz, ev), (az, pair), (mz, net), (mz, _mz(mz[:1], *pair) + _mz([other], *pair)),
             (az, [NetworkSearch(_engines(N, (G,), S)[0], net)]), (mz, _mz(mz, *pair)[:1]),
             (mz, _mz(mz, *pair, nodes_per_game=2))]
    torch.cuda.synchronize()
    for engines, evaluator in cases:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            with pytest.raises(ValueError):
                buf.reanalyse(engines, evaluator=evaluator)
            torch.cuda.synchronize()
        assert not [e.name for e in prof.events() if e.name.startswith("k_")]
        assert torch.equal(buf.ring, snap)


def test_no_host_sync_inside_a_batch():
    import torch
    N = 6
    buf = _fill(N, 32, S, 700, moves=12)
    snap = buf.ring.clone()
    counts = []
    for Gs in ((48, 48), (24, 24)):                               # >= 4 and >= 8 batches over the whole ring
        engines = _engines(N, Gs, S, mode="MuZero")
        searchers = _mz(engines, *_e0_pair(N, 2))
        assert len(buf) // Gs[0] >= 4
        buf.ring.copy_(snap)
        buf.reanalyse(engines, evaluator=searchers, noise_seed=1)            # warm-up: arena sized, graphs captured
        ref = buf.ring.clone()
        buf.ring.copy_(snap)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("warn")
        try:
            with warnings.catch_warnings(record=True) as w:
                warnings.simplefilter("always")
                buf.reanalyse(engines, evaluator=searchers, noise_seed=1)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        counts.append(sum("synchroniz" in str(x.message) for x in w))
        torch.cuda.synchronize()
        assert torch.equal(buf.ring, ref)
    assert counts == [1, 1]


def test_hot_swapped_weights_take_effect():
    import torch
    from datou_gomoku_muzero_b200.network import NetworkSearch
    N, G = 6, 24
    buf = _fill(N, 32, S, 500, moves=12)
    snap = buf.ring.clone()
    net1, net2 = _net(N, 1), _net(N, 2)
    with _Deterministic():
        engines = _engines(N, (G, G), S, accum_dtype="float32")
        searchers = [NetworkSearch(e, net1) for e in engines]
        torch.backends.cudnn.benchmark = False
        buf.reanalyse(engines, evaluator=searchers, noise_seed=3)            # captures the graphs with net1's weights
        first = buf.ring.clone()
        for s in searchers:
            s.update_weights(net2.state_dict())
        buf.ring.copy_(snap)
        buf.reanalyse(engines, evaluator=searchers, noise_seed=3)
        swapped = buf.ring.clone()
        fresh_engines = _engines(N, (G, G), S, accum_dtype="float32")
        fresh = [NetworkSearch(e, net2) for e in fresh_engines]
        torch.backends.cudnn.benchmark = False
        buf.ring.copy_(snap)
        buf.reanalyse(fresh_engines, evaluator=fresh, noise_seed=3)
    assert not torch.equal(swapped, first)
    assert torch.equal(swapped, buf.ring)
