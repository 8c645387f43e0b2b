"""GPU parity: the CUDA engine (through the C ABI) against (a) the golden vectors produced by
the imported reference and (b) the CPU oracle on seeded random inputs.  Bar: visit counts,
chosen moves, per-simulation leaf traces, terminal flags and root values bit-exact; policies within
1e-12 relative + 1e-15 absolute, a few ulp of float64 (a float32 improved policy would fail)."""
import os

import numpy as np
import pytest

from _golden_util import GOLDEN_DIR, load_search_cases

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-12, 1e-15   # policies: the oracle's own tolerance against the reference goldens


def _engine(c, G=1, mode=None):
    from datou_gomoku_muzero_b200.engine import SearchEngine
    return SearchEngine(G, board_size=c["N"], n_in_row=c["n_in_row"], num_simulations=c["S"], num_top_actions=c["K"],
                        mode=mode or ("AlphaZero" if c["mode"] == "az" else "MuZero"), c_visit=c["c_visit"],
                        c_scale=c["c_scale"], minmax_delta=c["delta"], discount=c["discount"],
                        accum_dtype="float32" if c["vdtype"] else "float64")


def _check(c, pol, val, act, vis, ta, td, tag):
    tag += f" div={c['logit_div']} f32={c['vdtype']}"
    assert np.array_equal(vis, c["visits"]), f"{tag}: visit counts"
    assert int(act) == c["action"], f"{tag}: action {act} vs {c['action']}"
    if ta is not None:
        n = len(c["leaf_actions"])
        assert np.array_equal(ta[:n], c["leaf_actions"]), f"{tag}: leaf action trace"
        assert np.array_equal(td[:n], c["leaf_depths"]), f"{tag}: leaf depth trace"
    np.testing.assert_allclose(val, c["value"], rtol=RTOL, atol=ATOL, err_msg=tag)
    assert float(val) == c["value"], f"{tag}: root value bits"        # float64 / float32 accumulation is bit-exact
    np.testing.assert_allclose(pol, c["policy"], rtol=RTOL, atol=ATOL, err_msg=tag)


@pytest.mark.parametrize("N", [6, 9, 15, 19])
def test_fused_search_matches_reference_goldens(N):
    for c in [c for c in load_search_cases("az", N) if c["kind"] == 0]:
        eng = _engine(c, G=3)
        eng.set_roots(np.tile(c["board"].reshape(1, -1), (3, 1)), [c["player"]] * 3, [c["last_move"]] * 3, [c["move_count"]] * 3)
        ta, td = eng.search_e0(np.tile(c["gumbel"], (3, 1)), c["seed"], c["logit_div"], trace=True)
        pol, val, act, vis = (t.cpu().numpy() for t in eng.finalize())
        ta, td = ta.cpu().numpy(), td.cpu().numpy()
        for g in range(3):
            _check(c, pol[g], val[g], act[g], vis[g], ta[g], td[g], f"fused az N={N} case {c['idx']} game {g}")


@pytest.mark.parametrize("N", [6, 9, 15, 19])
def test_stepwise_search_matches_reference_goldens(N):
    cases = [c for c in load_search_cases("az", N) if c["kind"] == 0]
    if N >= 15:
        cases = cases[::3]
    for c in cases:
        eng = _engine(c, G=2)
        eng.set_roots(np.tile(c["board"].reshape(1, -1), (2, 1)), [c["player"]] * 2, [c["last_move"]] * 2, [c["move_count"]] * 2)
        ta, td = eng.search_stepwise_e0(np.tile(c["gumbel"], (2, 1)), c["seed"], c["logit_div"], trace=True)
        pol, val, act, vis = (t.cpu().numpy() for t in eng.finalize())
        for g in range(2):
            _check(c, pol[g], val[g], act[g], vis[g], None if ta is None else ta[g].cpu().numpy(),
                   None if td is None else td[g].cpu().numpy(), f"stepwise az N={N} case {c['idx']} game {g}")


@pytest.mark.parametrize("N", [6, 9, 15, 19])
def test_constant_evaluator_goldens(N):
    """MockModel-style evaluator (tests/test_mcts_logic.py:60-80): logits 0, value const (incl. > 1 -> clip)."""
    import torch
    for c in [c for c in load_search_cases("az", N) if c["kind"] == 1]:
        eng = _engine(c, G=1)
        eng.set_roots(c["board"].reshape(1, -1), [c["player"]], [c["last_move"]], [c["move_count"]])
        lg = torch.zeros((1, N * N), dtype=torch.float32, device="cuda")
        v = torch.full((1,), c["const_value"], dtype=torch.float32 if c["vdtype"] else torch.float64, device="cuda")
        eng.root_expand(lg, v, c["gumbel"].reshape(1, -1))
        for _ in range(c["S"] - 1):
            eng.select()
            eng.expand_backup(lg, v)
        pol, val, act, vis = (t.cpu().numpy() for t in eng.finalize())
        _check(c, pol[0], val[0], act[0], vis[0], None, None, f"const az N={N} case {c['idx']}")


@pytest.mark.parametrize("N", [6, 9, 15, 19])
def test_muzero_search_matches_reference_goldens(N):
    """MuZero mode through gmz_select_mz / gmz_expand_backup with the E0 recurrent evaluator run
    on the host (hidden state = 64-bit hash per node slot)."""
    import torch
    import e0_py
    cases = load_search_cases("mz", N)
    if N == 15:
        cases = cases[::2]
    for c in cases:
        A = N * N
        eng = _engine(c, G=1)
        eng.set_roots(c["board"].reshape(1, -1), [c["player"]], [c["last_move"]], [c["move_count"]])
        hidden = {}
        obs = eng.root_obs().cpu().numpy()[0]
        if c["kind"] == 0:
            h0 = e0_py.hash_obs(obs, c["seed"])
            lg, v = e0_py.heads(h0, A, c["logit_div"])
        else:
            h0, lg, v = 1, np.zeros(A, np.float32), c["const_value"]
        hidden[0] = h0
        vdt = np.float32 if c["vdtype"] else np.float64
        eng.root_expand(lg.reshape(1, -1), np.array([v], vdt), c["gumbel"].reshape(1, -1))
        trace_a, trace_d, n_eval = [], [], 0
        for _ in range(c["S"]):
            ps, ac, cs, dp = (int(t.cpu()[0]) for t in eng.select_mz())
            if ps < 0:
                break
            if c["kind"] == 0:
                hc = e0_py.child_hidden(hidden[ps], ac)
                lg, v = e0_py.heads(hc, A, c["logit_div"])
                r = e0_py.reward_of(hc, c["logit_div"])
            else:
                hc, lg, v, r = 2, np.zeros(A, np.float32), c["const_value"], c["const_reward"]
            hidden[cs] = hc
            trace_a.append(ac); trace_d.append(dp); n_eval += 1
            eng.expand_backup(lg.reshape(1, -1), np.array([v], vdt), np.array([r], vdt))
        assert n_eval == c["n_recurrent"], f"mz N={N} case {c['idx']}: {n_eval} evaluations vs {c['n_recurrent']}"
        pol, val, act, vis = (t.cpu().numpy() for t in eng.finalize())
        _check(c, pol[0], val[0], act[0], vis[0], np.array(trace_a), np.array(trace_d), f"mz N={N} case {c['idx']}")


def test_e0_kernel_matches_python():
    import torch
    import e0_py
    from datou_gomoku_muzero_b200.engine import SearchEngine
    rs = np.random.RandomState(5)
    for N in (6, 9, 15, 19):
        A = N * N
        eng = SearchEngine(1, board_size=N, num_simulations=2)
        B = 16
        obs = np.zeros((B, 3, N, N), np.float32)
        for b in range(B):
            cells = rs.randint(-1, 2, size=(N, N))
            obs[b, 0] = cells == 1; obs[b, 1] = cells == -1
            if b % 4:
                a = rs.randint(A); obs[b, 2, a // N, a % N] = 1
        seed, div = int(rs.randint(1 << 30)), int(rs.choice([0, 2, 3, 16]))
        lg, v = eng.e0_eval(torch.from_numpy(obs).cuda(), seed, div)
        lg, v = lg.cpu().numpy(), v.cpu().numpy()
        for b in range(B):
            h = e0_py.hash_obs(obs[b], seed)
            l2, v2 = e0_py.heads(h, A, div)
            assert np.array_equal(lg[b], l2) and v[b] == v2, (N, b)


def test_fused_kernels_reject_divisors_that_are_not_powers_of_two():
    """gmz_e0_eval_obs takes any logit_div >= 0 (checked above with 3); the fused kernels compute a logit as one exact
    multiply and say so instead of computing something else (include/gmz.h)."""
    import torch
    from datou_gomoku_muzero_b200._lib import GmzError
    from datou_gomoku_muzero_b200.engine import SearchEngine
    eng = SearchEngine(2, board_size=6, num_simulations=8)
    gum = torch.zeros((2, 36), dtype=torch.float64, device="cuda")
    for bad in (3, 12, -1):
        with pytest.raises(GmzError, match="power of two"):
            eng.search_e0(gum, 1, bad)
        with pytest.raises(GmzError, match="power of two"):
            eng.selfplay_e0(2, 1, bad)
    eng.search_e0(gum, 1, 8); eng.search_e0(gum, 1, 0)


@pytest.mark.parametrize("div,accum", [(16, "float64"), (0, "float64"), (0, "float32"), (16, "float32")])
@pytest.mark.parametrize("N,S,G", [(9, 100, 64), (15, 400, 96), (19, 64, 16), (6, 50, 64)])
def test_random_positions_match_oracle(N, S, G, div, accum):
    """Seeded random mid-game positions + random noise: fused kernel vs CPU oracle, with quantised and dense
    (unquantised, div = 0) logits, in float64 and float32 (production dtype) accumulation."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    A = N * N
    rs = np.random.RandomState(N * 1000 + S)
    boards = np.zeros((G, A), np.int8); players = np.ones(G, np.int8)
    last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    for g in range(G):
        k = int(rs.randint(0, A))
        if g == 0:
            k = A          # full board -> inactive game -> sentinel
        p = 1
        for a in rs.permutation(A)[:k]:
            boards[g, a] = p; last[g] = a; p = -p
        players[g] = p; mc[g] = k
    gumbel = rs.gumbel(0, 1, (G, A))
    seed = 77
    eng = SearchEngine(G, board_size=N, num_simulations=S, num_top_actions=16, accum_dtype=accum)
    eng.set_roots(boards, players, last, mc)
    eng.search_e0(gumbel, seed, div)
    pol, val, act, vis = (t.cpu().numpy() for t in eng.finalize())
    cfg = oracle.make_config(board_size=N, num_simulations=S, num_top_actions=16, eval_seed=seed, logit_div=div,
                             accum_dtype=int(accum == "float32"))
    opol, oval, oact, ovis = oracle.search_batch(cfg, boards, players, last, mc, gumbel)
    assert act[0] == -1 and pol[0].sum() == 0 and val[0] == 0.0      # sentinel (mcts.py:214-215)
    assert np.array_equal(vis, ovis)
    assert np.array_equal(act, oact)
    np.testing.assert_allclose(val, oval, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(pol, opol, rtol=RTOL, atol=ATOL)
    assert np.array_equal(val, oval), "value accumulation should be bit-exact"
    # the roots must come back unchanged (search() must not mutate the game)
    b2, p2, l2, m2 = (t.cpu().numpy() for t in eng.get_roots())
    assert np.array_equal(b2.reshape(G, A), boards) and np.array_equal(p2, players)
    assert np.array_equal(l2, last) and np.array_equal(m2, mc)


def test_game_step_matches_reference_kat():
    """do_move + get_game_ended (game.py:20-63) on device vs the reference KATs."""
    from datou_gomoku_muzero_b200.engine import SearchEngine
    z = np.load(os.path.join(GOLDEN_DIR, "game_kat.npz"))
    for N, nir in sorted({(int(a), int(b)) for a, b in zip(z["N"], z["nir"])}):
        sel = np.flatnonzero((z["N"] == N) & (z["nir"] == nir))
        G, A = len(sel), N * N
        boards = z["boards"][sel][:, :A].copy()
        last = z["last"][sel].astype(np.int32)
        colour = boards[np.arange(G), last].copy()
        boards[np.arange(G), last] = 0                     # take the last stone back, then replay it
        eng = SearchEngine(G, board_size=N, n_in_row=nir, num_simulations=2)
        eng.set_roots(boards, colour, np.full(G, -1, np.int32), z["move_count"][sel] - 1)
        w = eng.game_step(last).cpu().numpy()
        assert np.array_equal(w, z["ended"][sel]), (N, nir)
        b2, p2, l2, m2 = (t.cpu().numpy() for t in eng.get_roots())
        assert np.array_equal(b2.reshape(G, A), z["boards"][sel][:, :A])
        assert np.array_equal(p2, -colour) and np.array_equal(l2, last) and np.array_equal(m2, z["move_count"][sel])


@pytest.mark.parametrize("N,S,G", [(9, 100, 48), (15, 400, 32), (6, 50, 40)])
def test_muzero_device_search_matches_oracle(N, S, G):
    """MuZero mode entirely on the device (hidden-state pool + E0 as torch integer ops) vs the oracle."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.muzero import MuZeroDeviceSearch, TorchE0, evals_per_search
    from oracle import oracle
    A, seed = N * N, 31
    rs = np.random.RandomState(N + S)
    boards = np.zeros((G, A), np.int8); players = np.ones(G, np.int8)
    last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    for g in range(G):
        k = int(rs.randint(0, A - 1)) if g % 5 else A - 1 - (g % 3)      # some games with < 16 valid moves
        p = 1
        for a in rs.permutation(A)[:k]:
            boards[g, a] = p; last[g] = a; p = -p
        players[g] = p; mc[g] = k
    gumbel = rs.gumbel(0, 1, (G, A))
    eng = SearchEngine(G, board_size=N, num_simulations=S, mode="MuZero")
    eng.set_roots(boards, players, last, mc)
    e0 = TorchE0(N, seed=seed)
    mz = MuZeroDeviceSearch(eng, e0.initial, e0.recurrent)
    mz.search(torch.from_numpy(gumbel).cuda())
    pol, val, act, vis = (t.cpu().numpy() for t in eng.finalize())
    cfg = oracle.make_config(board_size=N, num_simulations=S, mode=1, eval_seed=seed)
    opol, oval, oact, ovis = oracle.search_batch(cfg, boards, players, last, mc, gumbel)
    assert np.array_equal(vis, ovis) and np.array_equal(act, oact)
    assert np.array_equal(val, oval)
    np.testing.assert_allclose(pol, opol, rtol=RTOL, atol=ATOL)
    assert evals_per_search(S, 16, 16) == {100: 33, 400: 100, 50: 22}[S]      # SURVEY App. A.6 batch schedule


def test_folded_recurrent_inference_matches_module():
    import torch
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.muzero import FoldedRecurrentInference
    from datou_gomoku_muzero_b200.network import FoldedInitialInference, GomokuNetEZ
    torch.manual_seed(1)
    cfg = Config(BOARD_SIZE=9, ACTION_SPACE_SIZE=81, NUM_RES_BLOCKS=2, NUM_FILTERS=32, HEAD_HIDDEN_DIM=16)
    net = GomokuNetEZ(cfg).cuda().eval()
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.2); m.running_var.uniform_(0.5, 1.5); m.weight.normal_(1, 0.2); m.bias.normal_(0, 0.2)
    obs = (torch.rand(16, 3, 9, 9, device="cuda") < 0.3).float()
    act = torch.randint(0, 81, (16,), device="cuda")
    p, v, h = net.initial_inference(obs)
    p2, v2, h2, r2 = net.recurrent_inference(h, act.reshape(-1, 1))
    fi, fr = FoldedInitialInference(net, torch.float32), FoldedRecurrentInference(net, torch.float32)
    fp, fv, fh = fi(obs.contiguous(memory_format=torch.channels_last))
    torch.testing.assert_close(fp, p, rtol=1e-3, atol=1e-3)
    torch.testing.assert_close(fv, v, rtol=1e-3, atol=1e-3)
    lp, lv, lr, lh = fr(fh, act)
    torch.testing.assert_close(lp, p2, rtol=1e-3, atol=2e-3)
    torch.testing.assert_close(lv, v2.reshape(-1), rtol=1e-3, atol=2e-3)
    torch.testing.assert_close(lr, r2.reshape(-1), rtol=1e-3, atol=2e-3)
    torch.testing.assert_close(lh, h2, rtol=1e-3, atol=2e-3)


@pytest.mark.parametrize("div,accum", [(16, "float64"), (0, "float32")])
@pytest.mark.parametrize("N,S,G", [(9, 100, 64), (15, 400, 64), (6, 50, 48)])
def test_muzero_fused_search_matches_oracle(N, S, G, div, accum):
    """MuZero mode inside the persistent kernel (E0's recurrent evaluator inlined) vs the oracle."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    A, seed = N * N, 17
    rs = np.random.RandomState(3 * N + S)
    boards = np.zeros((G, A), np.int8); players = np.ones(G, np.int8)
    last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    for g in range(G):
        k = int(rs.randint(0, A - 1)) if g % 4 else A - 1 - (g % 5)
        p = 1
        for a in rs.permutation(A)[:k]:
            boards[g, a] = p; last[g] = a; p = -p
        players[g] = p; mc[g] = k
    gumbel = rs.gumbel(0, 1, (G, A))
    eng = SearchEngine(G, board_size=N, num_simulations=S, mode="MuZero", accum_dtype=accum)
    eng.set_roots(boards, players, last, mc)
    ta, td = eng.search_e0(torch.from_numpy(gumbel).cuda(), seed, div, trace=True)
    pol, val, act, vis = (t.cpu().numpy() for t in eng.finalize())
    cfg = oracle.make_config(board_size=N, num_simulations=S, mode=1, eval_seed=seed, logit_div=div,
                             accum_dtype=int(accum == "float32"))
    opol, oval, oact, ovis = oracle.search_batch(cfg, boards, players, last, mc, gumbel)
    assert np.array_equal(vis, ovis) and np.array_equal(act, oact) and np.array_equal(val, oval)
    np.testing.assert_allclose(pol, opol, rtol=RTOL, atol=ATOL)
    r = oracle.search(cfg, boards[1], players[1], last[1], mc[1], gumbel[1], trace=True)
    n = r["n_evals"]
    assert np.array_equal(ta[1].cpu().numpy()[:n], r["leaf_actions"]) and np.array_equal(td[1].cpu().numpy()[:n], r["leaf_depths"])


@pytest.mark.parametrize("mode", ["AlphaZero", "MuZero"])
def test_deep_paths_match_oracle(mode):
    """Peaked logits (logit_div = 2) grow chains deeper than one warp (> 32 edges): the descent path then
    spills from registers to the global path buffer.  Fused and stepwise kernels vs the oracle, with the
    per-simulation (leaf action, depth) traces."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    N, S, G, seed, div = 9, 300, 12, 12, 2
    A = N * N
    rs = np.random.RandomState(4)
    boards = np.zeros((G, A), np.int8); players = np.ones(G, np.int8)
    last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    gumbel = rs.gumbel(0, 1, (G, A))
    m = 0 if mode == "AlphaZero" else 1
    cfg = oracle.make_config(board_size=N, num_simulations=S, eval_seed=seed, logit_div=div, mode=m)
    opol, oval, oact, ovis = oracle.search_batch(cfg, boards, players, last, mc, gumbel)
    refs = [oracle.search(cfg, boards[g], 1, -1, 0, gumbel[g], trace=True) for g in range(G)]
    if mode == "AlphaZero":          # (MuZero mode backs every leaf up k times: its trees stay shallow)
        assert max(int(r["leaf_depths"][:r["n_evals"]].max()) for r in refs) > 40
    eng = SearchEngine(G, board_size=N, num_simulations=S, mode=mode)
    runs = [("fused", lambda: eng.search_e0(torch.from_numpy(gumbel).cuda(), seed, div, trace=True))]
    if mode == "AlphaZero":
        runs.append(("stepwise", lambda: eng.search_stepwise_e0(torch.from_numpy(gumbel).cuda(), seed, div, trace=True)))
    for name, run in runs:
        eng.set_roots(boards, players, last, mc)
        ta, td = run()
        pol, val, act, vis = (t.cpu().numpy() for t in eng.finalize())
        assert np.array_equal(vis, ovis) and np.array_equal(act, oact) and np.array_equal(val, oval), name
        if ta is not None:
            for g in range(G):
                n = refs[g]["n_evals"]
                assert np.array_equal(ta[g].cpu().numpy()[:n], refs[g]["leaf_actions"]), (name, g)
                assert np.array_equal(td[g].cpu().numpy()[:n], refs[g]["leaf_depths"]), (name, g)
