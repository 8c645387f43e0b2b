"""bench.py --dump-outputs: the last step's outputs, the same for the same arguments, in the agreed format, and equal to
what the CPU oracle's game loop computes for that move; --steps sets the number of timed moves."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G, STEPS, WARMUP = 256, 4, 3


def _bench(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--games", str(G), "--steps", str(STEPS), "--warmup", str(WARMUP),
                        "--no-net", "--no-config5", "--no-cpu-baseline", "--no-selfplay-e2e", "--e2e-depth", "2",
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    names = sorted(os.listdir(out_dir))
    return json.loads(lines[0]), {n[:-4]: np.load(os.path.join(out_dir, n)) for n in names if n.endswith(".npy")}, names


def test_dump_outputs_are_reproducible_and_match_the_oracle(tmp_path):
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from oracle import oracle
    import bench
    line, a, names = _bench(tmp_path / "a")
    _, b, _ = _bench(tmp_path / "b")
    assert names == sorted(n + ".npy" for n in ("policy", "value", "action", "board", "winner", "game"))
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for name in a:
        assert a[name].dtype in (np.float32, np.float64), name
        assert np.array_equal(a[name], b[name]), name
    A = bench.A
    assert a["policy"].shape == (G, A) and a["board"].shape == (G, A) and np.array_equal(a["game"], np.arange(G))
    moved = a["action"] >= 0
    assert moved.all() and np.allclose(a["policy"].sum(1), 1.0)
    # timed moves = steps x games: the rate times the timed seconds gives back the moves
    assert line["steps"] == STEPS
    assert abs(line["moves_per_sec"] * line["ms_per_step"] * 1e-3 * STEPS - STEPS * G) < 1e-6 * STEPS * G
    # game 0 starts from the empty board: its move number warmup + steps through the oracle's game loop
    T = line["warmup"] + STEPS
    eng = SearchEngine(G, board_size=bench.N, num_simulations=bench.S, num_top_actions=bench.K_TOP)
    gum = torch.empty((T + 1, A), dtype=torch.float64, device="cuda")
    for k in range(T + 1):
        eng.fill_gumbel(gum[k], 1000, (k * G + 0) * A)
    cfg = oracle.make_config(board_size=bench.N, num_simulations=bench.S, num_top_actions=bench.K_TOP, eval_seed=bench.E0_SEED,
                             logit_div=bench.LOGIT_DIV)
    o = oracle.selfplay_game(cfg, gum.cpu().numpy())
    assert o["T"] == T + 1                                   # a game needs at least 9 plies: it is still going
    assert int(a["action"][0]) == int(o["actions"][T - 1]) and a["value"][0] == o["values"][T - 1]
    np.testing.assert_allclose(a["policy"][0], o["policies"][T - 1], rtol=1e-12, atol=1e-15)
    assert np.array_equal(a["board"][0], o["boards"][T].reshape(-1).astype(np.float32)) and a["winner"][0] == 2
