"""What self-play from an opening book costs, at the bench's size.

    python tools/opening_selfplay_probe.py [--games 4096] [--out profiles/r09_opening_selfplay.json]

Setup: 15x15, 400 simulations, K = 16, E0 seed / logit divisor of bench.py, book = random_openings(G, 4, 15).
  * persistent: E0 self-play moves/s of the persistent kernel without recording (gmz_selfplay_e0, traj NULL, restarts
    in the kernel), on one engine that never had a book and one with the book bound, timed alternately `--reps` times
    with CUDA events over `--moves` moves per game each, after a warm-up of the same length (games are mid-flight and
    restart throughout the window).
  * deals: device time of k_selfplay_step on roots where every game's move wins (every game restarts: one deal each),
    and of k_unpark restarting all G parked games, with and without the book, CUDA events around `--deal-launches`
    launches (the roots / parking are re-made between launches, outside the timed events).
  * network: moves/s of stepwise self-play with a GomokuNetEZ (8 blocks x 128 filters, bf16, one CUDA graph per
    simulation step) from the book, `--net-moves` lock-step moves after one warm-up move.
The card name and power limit are read in the same run and written beside the numbers."""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np
import torch

import bench
from stats_probe import card


def timed_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def winning_roots(G, N):
    """Every root: black four in a row on row g % N (cells 0..3), white stones on the row below, black to move; the move
    at cell 4 of that row wins."""
    A = N * N
    boards = np.zeros((G, A), np.int8)
    r = np.arange(G) % (N - 1)
    for c in range(4):
        boards[np.arange(G), r * N + c] = 1
        boards[np.arange(G), (r + 1) * N + c] = -1
    act = (r * N + 4).astype(np.int32)
    return boards, np.ones(G, np.int8), (r * N + 3).astype(np.int32), np.full(G, 8, np.int32), act


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=400)
    ap.add_argument("--moves", type=int, default=48)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--deal-launches", type=int, default=50)
    ap.add_argument("--net-moves", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_opening_selfplay.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("opening_selfplay_probe needs a CUDA device")
    from datou_gomoku_muzero_b200._lib import check
    from datou_gomoku_muzero_b200.arena import random_openings
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    G, N, S, K = args.games, 15, args.sims, 16
    A = N * N
    book = random_openings(G, 4, N, seed=1)
    out = dict(setup=dict(games=G, board=N, sims=S, K=K, evaluator="E0 seed %d, logit_div %d" % (bench.E0_SEED, bench.LOGIT_DIV),
                          book="random_openings(%d, 4, 15, seed=1)" % G, moves_per_game_timed=args.moves, reps=args.reps),
               card=card(torch.cuda.current_device()))

    # ---- persistent kernel, alternating no book / book
    runs = {}
    for name, op in (("no_book", None), ("book", book)):
        eng = SearchEngine(G, board_size=N, num_simulations=S, num_top_actions=K)
        sp = SelfPlayEngine(eng, "e0", seed=bench.E0_SEED, logit_div=bench.LOGIT_DIV, noise_seed=3, openings=op)
        runs[name] = (eng, sp)
        sp.play(moves_per_game=args.moves)                              # warm-up: games spread over their lengths
    times = {k: [] for k in runs}
    for _ in range(args.reps):
        for name, (eng, sp) in runs.items():
            times[name].append(timed_ms(lambda: sp.play(moves_per_game=args.moves)))
    out["persistent"] = {name: dict(ms=[round(t, 2) for t in ts], moves_per_s=[round(G * args.moves / (t * 1e-3)) for t in ts],
                                    games_finished=runs[name][0].play_counters()[1])
                         for name, ts in times.items()}
    print("persistent", json.dumps(out["persistent"]), flush=True)
    del runs
    torch.cuda.empty_cache()

    # ---- deals in the stepwise kernels
    boards, players, last, mc, act = (torch.from_numpy(x).cuda() for x in winning_roots(G, N))
    pol = torch.zeros((G, A), dtype=torch.float64, device="cuda")
    val = torch.zeros(G, dtype=torch.float64, device="cuda")
    deals = {}
    for name, op in (("no_book", None), ("book", book)):
        eng = SearchEngine(G, board_size=N, num_simulations=8, num_top_actions=K)
        eng.set_openings(op)
        step_ms = 0.0
        for i in range(args.deal_launches + 2):
            eng.set_roots(boards, players, last, mc)
            t = timed_ms(lambda: eng.selfplay_step(pol, val, act, None, True))
            step_ms += t if i >= 2 else 0.0
        traj = TrajectoryStore(eng, extra_slots=G, max_moves=4)
        ids = torch.arange(traj.n_slots, dtype=torch.int32, device="cuda")
        unpark_ms = 0.0
        for i in range(args.deal_launches + 2):
            eng.set_roots(boards, players, last, mc)
            traj.fin_count.zero_()
            eng.selfplay_step(pol, val, act, traj, False)              # every game finishes and parks
            traj.free_slots.copy_(ids)
            traj.free_top.fill_(traj.n_slots)
            t = timed_ms(lambda: check(eng.lib.gmz_selfplay_unpark(eng.handle, C.byref(traj.c), eng._stream()), "unpark"))
            unpark_ms += t if i >= 2 else 0.0
        b, *_ = eng.get_roots()
        dealt_ok = bool((b.reshape(G, A).cpu().numpy() == (book.boards if op is not None else 0)).all())
        deals[name] = dict(k_selfplay_step_ms=round(step_ms / args.deal_launches, 4),
                           k_unpark_ms=round(unpark_ms / args.deal_launches, 4), roots_after_unpark_as_dealt=dealt_ok)
    deals["note"] = ("CUDA events around one launch each; every game of the step finishes and is dealt a new game, "
                     "every game of the unpark is parked and restarted")
    out["deals"] = deals
    print("deals", json.dumps(deals), flush=True)
    torch.cuda.empty_cache()

    # ---- network stepwise self-play from the book
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.network import GomokuNetEZ
    torch.manual_seed(0)
    net = GomokuNetEZ(Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=A, NUM_RES_BLOCKS=8, NUM_FILTERS=128, HEAD_HIDDEN_DIM=64)).cuda().eval()
    eng = SearchEngine(G, board_size=N, num_simulations=S, num_top_actions=K, accum_dtype="float32")
    sp = SelfPlayEngine(eng, net, noise_seed=3, openings=book)
    traj = TrajectoryStore(eng)
    with torch.no_grad():
        sp.play(moves_per_game=1, traj=traj, sink=lambda pg: None)     # warm-up: graph capture
        t = timed_ms(lambda: sp.play(moves_per_game=args.net_moves, traj=traj, sink=lambda pg: None))
    out["network"] = dict(moves=G * args.net_moves, ms=round(t, 1), moves_per_s=round(G * args.net_moves / (t * 1e-3)),
                          network="GomokuNetEZ 8 blocks x 128 filters, head hidden 64, bf16, one CUDA graph per step",
                          accum="float32")
    print("network", json.dumps(out["network"]), flush=True)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
