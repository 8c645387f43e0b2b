"""Cost and yield of the VCT solver (tactics.find_vct, gmz_vct_solve) on one GPU, next to the VCF solver.

    python tools/vct_probe.py [--records 100000] [--out profiles/r12_vct.json]

1. The boards of the move records of a 4096-game 15x15 / 400-simulation E0 self-play ring (bench.py's selfplay_e2e
   setup, as tools/vcf_probe.py builds it): gmz_vct_solve at max_attacks 8 and 16 and node budgets 5,000 and 20,000 --
   positions per second (CUDA events around one call), mean and largest node count, the share the budget cuts, and how
   many records VCT decides (length > 0) where VCF at the same max_attacks and budget does not.
2. opening_vct against opening_vcf on a 100,000-opening 10-stone random_openings book: wall-clock time, the share of
   openings decided for either side and the share cut.
The card name and power limit are read in the same run and written beside the numbers."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))

import numpy as np
import torch

import bench
from stats_probe import card


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    return out, e0.elapsed_time(e1) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=100_000, help="records solved: the first ring positions of the full 400,000-record ring")
    ap.add_argument("--moves", type=int, default=96, help="moves per game per self-play call filling the ring")
    ap.add_argument("--openings", type=int, default=100_000)
    ap.add_argument("--opening-stones", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(ROOT), "profiles", "r12_vct.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("vct_probe needs a CUDA device")
    from datou_gomoku_muzero_b200.arena import opening_vcf, opening_vct, random_openings
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.tactics import VCT_ATTACKS, VCT_BUDGET, find_vcf, find_vct
    from datou_gomoku_muzero_b200.trajectory import RECORD_HEADER, TrajectoryStore, record_fields

    dev = torch.device("cuda:0")
    G, N = 4096, bench.N
    eng = SearchEngine(G, board_size=N, n_in_row=bench.N_IN_ROW, num_simulations=bench.S, num_top_actions=bench.K_TOP,
                       device=dev)
    sp = SelfPlayEngine(eng, "e0", seed=bench.E0_SEED, logit_div=bench.LOGIT_DIV, noise_seed=2000)
    eng.set_roots(*bench.staggered_positions(G, 0))
    traj = TrajectoryStore(eng, extra_slots=G // 2)
    buf = DeviceReplayBuffer(400_000, N, device=dev)
    while len(buf) < 400_000:
        sp.play(moves_per_game=args.moves, traj=traj, sink=buf.add_packed)
    M = min(args.records, len(buf))
    rec = buf.ring[:M]
    boards = rec[:, record_fields(N)["board"]].view(torch.int8).contiguous()
    off = RECORD_HEADER.fields["to_move"][1]
    players = rec[:, off:off + 4].contiguous().view(torch.int32).reshape(M).to(torch.int8)
    kw = dict(n_in_row=bench.N_IN_ROW, board_size=N)
    find_vct(boards[:4096], players[:4096], 8, 100, **kw)                       # module load
    find_vcf(boards[:4096], players[:4096], 8, 100, **kw)
    solver = {}
    for L in (8, 16):
        for budget in (5_000, 20_000):
            (tl, _, tn), sec = timed(lambda: find_vct(boards, players, L, budget, **kw))
            (vl, _, vn), vsec = timed(lambda: find_vcf(boards, players, L, budget, **kw))
            tl, tn, vl = tl.cpu().numpy(), tn.cpu().numpy(), vl.cpu().numpy()
            solver[f"max_attacks_{L}_budget_{budget}"] = {
                "positions": M, "seconds": sec, "positions_per_sec": M / sec, "mean_nodes": float(tn.mean()),
                "max_nodes": int(tn.max()), "with_vct": int((tl > 0).sum()), "cut": int((tl < 0).sum()),
                "cut_share": float((tl < 0).mean()),
                "vct_decides_vcf_does_not": int(((tl > 0) & (vl <= 0)).sum()),
                "vct_decides_vcf_cut": int(((tl > 0) & (vl < 0)).sum()),
                "vcf_decides_vct_cut": int(((vl > 0) & (tl < 0)).sum()),
                "vcf": {"seconds": vsec, "positions_per_sec": M / vsec, "mean_nodes": float(vn.cpu().numpy().mean()),
                        "with_vcf": int((vl > 0).sum()), "cut": int((vl < 0).sum())},
                "length_histogram": {int(k): int(v) for k, v in zip(*np.unique(tl, return_counts=True))}}
            print(f"L={L} budget={budget}: {M / sec:.0f} pos/s, cut {float((tl < 0).mean()) * 100:.2f} %", flush=True)

    book = random_openings(args.openings, args.opening_stones, N, seed=1)
    t0 = time.perf_counter()
    vm, vo = opening_vcf(book, 8, 20_000)
    t_vcf = time.perf_counter() - t0
    t0 = time.perf_counter()
    tm, to = opening_vct(book, VCT_ATTACKS, VCT_BUDGET)
    t_vct = time.perf_counter() - t0
    O = len(vm)
    out = {
        "what": "VCT solver (gmz_vct_solve) against the VCF solver on E0 self-play ring records and on a random_openings "
                "book",
        "card": card(0),
        "config": {"games": G, "board": N, "n_in_row": bench.N_IN_ROW, "num_simulations": bench.S,
                   "evaluator": "E0 seed %d, logit_div %d" % (bench.E0_SEED, bench.LOGIT_DIV),
                   "ring_records_solved": M, "vct_defaults": {"max_attacks": VCT_ATTACKS, "node_budget": VCT_BUDGET}},
        "solver_on_ring_records": solver,
        "solver_timing": "CUDA events around one find_vct / find_vcf call (kernel plus the bitmask unpacking) after a "
                         "warm-up call on 4096 records",
        "opening_book": {
            "openings": O, "stones": args.opening_stones,
            "opening_vcf": {"max_attacks": 8, "node_budget": 20_000, "seconds": t_vcf,
                            "decided_share": float(((vm > 0) | (vo > 0)).mean()),
                            "cut_share": float(((vm < 0) | (vo < 0)).mean())},
            "opening_vct": {"max_attacks": VCT_ATTACKS, "node_budget": VCT_BUDGET, "seconds": t_vct,
                            "decided_share": float(((tm > 0) | (to > 0)).mean()),
                            "cut_share": float(((tm < 0) | (to < 0)).mean()),
                            "mover_vct": int((tm > 0).sum()), "opponent_vct": int((to > 0).sum())},
            "vct_decides_vcf_does_not": int((((tm > 0) | (to > 0)) & ~((vm > 0) | (vo > 0))).sum()),
            "kept_by_vct_filter": int(((tm == 0) & (to == 0)).sum()),
        },
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"opening_book": out["opening_book"], "card": out["card"]}))


if __name__ == "__main__":
    main()
