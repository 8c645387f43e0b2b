"""Throughput of a match between two engines (arena.Arena) at the bench's size.

    python tools/arena_probe.py [--games 4096] [--openings 16384] [--plies 120] [--net-plies 4] [--out profiles/r07_arena.json]

Setup: 15x15, n_in_row 5, 400 simulations, K = 16 (bench.py's constants), G games per player (two engines), an opening
book of random_openings(O, 4 stones) so the queues stay full during the timed plies.  Legs, each after warm-up plies:
  e0     : E0 (seed 1) against E0 (seed 2), float64 engines, `plies` timed plies;
  net    : a seeded random GomokuNetEZ 8x128 (head hidden 64, bf16, one CUDA graph per simulation step) against the same
           network with another seed, float32 engines, `net_plies` timed plies;
  kernels: torch.profiler over 6 plies of the e0 leg: device time of the match kernels (k_match_noise + k_match_step)
           against the wall time of those plies;
  selfplay: the persistent E0 self-play kernel on one of the same engines, moves/s, as a reference point.
Rates: plies/s; moves/s = games in flight moved per second (2G per ply while the queues last); games/s = games finished
in the timed window per second.  The card name and power limit are read in the same run and written beside the
numbers."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch

import bench
from stats_probe import card


def timed_plies(arena, n):
    dev = arena.engines[0].device
    f0 = arena.finished()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(n):
        arena.ply()
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    fin = arena.finished() - f0
    G = arena.engines[0].G
    return {"plies": n, "seconds": dt, "plies_per_s": n / dt, "moves_per_s": 2 * G * n / dt,
            "games_finished": fin, "games_per_s": fin / dt if fin else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--openings", type=int, default=16384)
    ap.add_argument("--plies", type=int, default=120)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--net-plies", type=int, default=4)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_arena.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("arena_probe measures on a CUDA device; none found")
    from datou_gomoku_muzero_b200.arena import Arena, random_openings
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.network import GomokuNetEZ
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    N, A, S, K, G = bench.N, bench.A, bench.S, bench.K_TOP, args.games
    dev = torch.device("cuda:0")
    mk = lambda accum="float64": SearchEngine(G, board_size=N, n_in_row=bench.N_IN_ROW, num_simulations=S, num_top_actions=K,
                                              accum_dtype=accum, device=dev)
    t0 = time.perf_counter()
    book = random_openings(args.openings, 4, N, seed=7, n_in_row=bench.N_IN_ROW)
    book_s = time.perf_counter() - t0
    out = {"what": "Arena throughput: two engines of G games each play a colour-paired match from a random 4-stone "
                   "opening book (queues never run dry in the timed plies)",
           "card": card(0),
           "config": {"board": N, "n_in_row": bench.N_IN_ROW, "num_simulations": S, "num_top_actions": K,
                      "games_per_player": G, "openings": args.openings, "opening_book_host_s": book_s}}

    ea, eb = mk(), mk()
    arena = Arena(ea, eb, eval_seed_a=1, eval_seed_b=2, logit_div_a=bench.LOGIT_DIV, logit_div_b=bench.LOGIT_DIV, seed=3)
    arena.start(book)
    for _ in range(args.warmup):
        arena.ply()
    out["e0"] = timed_plies(arena, args.plies)
    print("e0", json.dumps(out["e0"]), flush=True)

    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize(dev)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        t0 = time.perf_counter()
        for _ in range(6):
            arena.ply()
        torch.cuda.synchronize(dev)
        wall = time.perf_counter() - t0
    match_us = {}
    for ev in prof.key_averages():
        if ev.key.startswith("k_match_"):
            match_us[ev.key] = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    out["kernels"] = {"plies": 6, "wall_s_profiled": wall, "match_kernel_us": match_us,
                      "share_of_ply": sum(match_us.values()) * 1e-6 / wall,
                      "note": "device time of k_match_noise + k_match_step over the wall time of the same plies, "
                              "profiler on (the wall time is then a little longer than unprofiled)"}
    print("kernels", json.dumps(out["kernels"]), flush=True)

    sp = SelfPlayEngine(ea, "e0", seed=bench.E0_SEED, logit_div=bench.LOGIT_DIV, noise_seed=5)
    sp.play(moves_per_game=2)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    sp.play(moves_per_game=20)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    out["selfplay"] = {"moves": 20 * G, "seconds": dt, "moves_per_s": 20 * G / dt,
                       "note": "persistent E0 self-play kernel on one engine of the same configuration"}
    print("selfplay", json.dumps(out["selfplay"]), flush=True)
    del arena, sp, ea, eb
    torch.cuda.empty_cache()

    cfg = Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=A, NUM_RES_BLOCKS=8, NUM_FILTERS=128, HEAD_HIDDEN_DIM=64)
    nets = []
    for s in (0, 1):
        torch.manual_seed(s)
        nets.append(GomokuNetEZ(cfg).to(dev).eval())
    na, nb = mk("float32"), mk("float32")
    arena = Arena(na, nb, nets[0], nets[1], seed=3)
    arena.start(book)
    arena.ply()                    # warm-up: graph capture of both searchers
    out["net"] = timed_plies(arena, args.net_plies)
    out["net"]["network"] = "GomokuNetEZ 8 blocks x 128 filters, head hidden 64, seeds 0 vs 1, bf16 folded, one CUDA graph per step"
    print("net", json.dumps(out["net"]), flush=True)

    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
