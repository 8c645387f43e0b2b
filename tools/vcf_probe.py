"""Cost of the VCF solver (tactics.find_vcf, gmz_vcf_solve / gmz_records_vcf) on one GPU.

    python tools/vcf_probe.py [--reps 6] [--moves 96] [--out profiles/r11_vcf.json]

1. gmz_vcf_solve alone, CUDA events over repeated launches, on the boards of the move records of 4096-game 15x15 /
   400-simulation E0 self-play (bench.py's selfplay_e2e setup), max_attacks 8 and 16: positions per second, and the mean
   and largest node count per position.
2. bench.py's selfplay_e2e loop with SelfPlayStats(vcf_attacks=8).add in the sink against without it, the two arms
   alternating in one process (as tools/stats_probe.py does for the missed-win flags): wall-clock moves/s per arm.
3. arena.opening_vcf on a 100,000-opening random_openings book: wall-clock time and how many openings it flags.
The card name and power limit are read in the same run and written beside the numbers."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import bench
from stats_probe import card


def spread(v):
    v = np.asarray(v)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()),
            "spread_pct": float((v.max() - v.min()) / np.median(v) * 100.0), "runs": [float(x) for x in v]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=6, help="timed repetitions per self-play arm (alternating)")
    ap.add_argument("--moves", type=int, default=96, help="moves per game in one timed repetition")
    ap.add_argument("--launches", type=int, default=5, help="timed solver launches per setting")
    ap.add_argument("--openings", type=int, default=100_000)
    ap.add_argument("--opening-stones", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_vcf.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("vcf_probe needs a CUDA device")
    from datou_gomoku_muzero_b200.arena import opening_vcf, random_openings
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.tactics import VCF_BUDGET, SelfPlayStats, find_vcf
    from datou_gomoku_muzero_b200.trajectory import RECORD_HEADER, TrajectoryStore

    dev = torch.device("cuda:0")
    G, N = 4096, bench.N
    A = N * N
    eng = SearchEngine(G, board_size=N, n_in_row=bench.N_IN_ROW, num_simulations=bench.S, num_top_actions=bench.K_TOP,
                       device=dev)
    sp = SelfPlayEngine(eng, "e0", seed=bench.E0_SEED, logit_div=bench.LOGIT_DIV, noise_seed=2000)
    eng.set_roots(*bench.staggered_positions(G, 0))
    traj = TrajectoryStore(eng, extra_slots=G // 2)
    buf = DeviceReplayBuffer(400_000, N, device=dev)
    stats = SelfPlayStats(n_in_row=bench.N_IN_ROW, device=dev, vcf_attacks=8)
    state = {"batches": 0, "with_stats": False}

    def sink(pg):                     # bench.selfplay_e2e_leg's sink, plus SelfPlayStats.add in the "with" arm
        if state["with_stats"]:
            stats.add(pg)
        buf.add_packed(pg)
        if len(buf) >= 360:
            batch, idx, w = buf.sample(360, rot_k=state["batches"] % 4, flip=bool(state["batches"] & 1))
            buf.update_priorities(idx, batch[4][:, 0] - 0.5)
            state["batches"] += 1

    def run(with_stats):
        state["with_stats"] = with_stats
        m0, _ = eng.play_counters()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sp.play(moves_per_game=args.moves, traj=traj, sink=sink)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        m1, _ = eng.play_counters()
        return (m1 - m0) / dt

    run(False); run(True)                                          # warm-up of both arms
    arms = {"without": [], "with": []}
    for r in range(args.reps):
        for name in (("without", "with") if r % 2 == 0 else ("with", "without")):
            arms[name].append(run(name == "with"))
    summary = stats.summary()

    # the solver alone on the ring's records: board and side to move of each
    M = len(buf)
    rec = buf.ring[:M]
    boards = rec[:, buf._field["board"]].view(torch.int8).contiguous()
    to_move = rec[:, RECORD_HEADER.fields["to_move"][1]:RECORD_HEADER.fields["to_move"][1] + 4].contiguous().view(torch.int32)
    players = to_move.reshape(M).to(torch.int8)
    solver = {}
    for L in (8, 16):
        length, first, nodes = find_vcf(boards, players, L, VCF_BUDGET, n_in_row=bench.N_IN_ROW, board_size=N)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.launches):
            find_vcf(boards, players, L, VCF_BUDGET, n_in_row=bench.N_IN_ROW, board_size=N)
        e1.record()
        torch.cuda.synchronize()
        sec = e0.elapsed_time(e1) / 1e3 / args.launches
        ln, nd = length.cpu().numpy(), nodes.cpu().numpy()
        solver[f"max_attacks_{L}"] = {
            "positions": M, "seconds_per_call": sec, "positions_per_sec": M / sec,
            "mean_nodes": float(nd.mean()), "max_nodes": int(nd.max()), "nodes_per_sec": float(nd.sum()) / sec,
            "with_vcf": int((ln > 0).sum()), "budget_cut": int((ln < 0).sum()),
            "length_histogram": {int(k): int(v) for k, v in zip(*np.unique(ln, return_counts=True))}}

    # opening book
    t0 = time.perf_counter()
    book = random_openings(args.openings, args.opening_stones, N, seed=1)
    t_book = time.perf_counter() - t0
    opening_vcf(book, 8, VCF_BUDGET)                              # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mover, opp = opening_vcf(book, 8, VCF_BUDGET)
    t_vcf = time.perf_counter() - t0
    flagged = (mover != 0) | (opp != 0)

    wo, wi = spread(arms["without"]), spread(arms["with"])
    out = {
        "what": "VCF solver: gmz_vcf_solve time on E0 self-play ring records, bench.py's selfplay_e2e loop with / without "
                "SelfPlayStats(vcf_attacks=8).add in the sink (arms alternating in one process), and opening_vcf on a "
                "random_openings book",
        "card": card(0),
        "config": {"games": G, "board": N, "n_in_row": bench.N_IN_ROW, "num_simulations": bench.S,
                   "num_top_actions": bench.K_TOP, "evaluator": "E0 seed %d, logit_div %d" % (bench.E0_SEED, bench.LOGIT_DIV),
                   "roots": "bench.staggered_positions", "node_budget": VCF_BUDGET, "moves_per_game_per_rep": args.moves,
                   "reps_per_arm": args.reps},
        "solver_on_ring_records": solver,
        "solver_timing": "CUDA events around back-to-back find_vcf calls (kernel plus the bitmask unpacking) on the current "
                         "stream; the boards (A bytes each) stay in L2 between calls",
        "selfplay_e2e_moves_per_sec": {"without_vcf_stats": wo, "with_vcf_stats": wi,
                                       "overhead_pct": (1.0 - wi["median"] / wo["median"]) * 100.0},
        "stats_summary_with_arm": summary,
        "opening_book": {"openings": args.openings, "stones": args.opening_stones, "book_seconds": t_book,
                         "opening_vcf_seconds": t_vcf, "flagged": int(flagged.sum()),
                         "mover_vcf": int((mover > 0).sum()), "opponent_vcf": int((opp > 0).sum()),
                         "budget_cut": int(((mover < 0) | (opp < 0)).sum())},
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"solver": {k: (v["positions_per_sec"], v["mean_nodes"]) for k, v in solver.items()},
                      "without": wo["median"], "with": wi["median"], "overhead_pct": out["selfplay_e2e_moves_per_sec"]["overhead_pct"],
                      "openings_flagged": int(flagged.sum()), "opening_vcf_s": t_vcf, "card": out["card"]}))


if __name__ == "__main__":
    main()
