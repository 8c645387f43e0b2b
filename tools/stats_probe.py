"""Cost of the missed-win statistics on device self-play (tactics.SelfPlayStats, gmz_records_tactics).

    python tools/stats_probe.py [--reps 6] [--moves 96] [--out profiles/r03_stats_probe.json]

1. gmz_records_tactics alone, CUDA events over many launches, on the move records of 4096-game 15x15 / 400-simulation
   self-play chunks (bench.py's selfplay_e2e setup): microseconds per 1000 records.
2. bench.py's selfplay_e2e loop (persistent E0 play -> pack -> DeviceReplayBuffer.add_packed -> sample(360) +
   update_priorities per chunk) with and without SelfPlayStats.add in the sink, the two arms alternating in one
   process: wall-clock moves/s of each repetition, median and spread per arm.
The card name and power limit are read in the same run and written beside the numbers."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import bench


def card(index):
    out = {"name": torch.cuda.get_device_name(index)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        out["nvidia_smi"] = q
        parts = [p.strip() for p in q.split(",")]
        if len(parts) >= 3:
            out["power_limit"], out["max_sm_clock"] = parts[1], parts[2]
    except Exception as ex:            # the numbers stay valid; the card line says why it is incomplete
        out["nvidia_smi_error"] = repr(ex)[:200]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=6, help="timed repetitions per arm (alternating)")
    ap.add_argument("--moves", type=int, default=96, help="moves per game in one timed repetition")
    ap.add_argument("--launches", type=int, default=200, help="kernel launches in the kernel timing")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_stats_probe.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stats_probe needs a CUDA device")
    from datou_gomoku_muzero_b200 import _lib
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.tactics import SelfPlayStats, record_flags
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore

    dev = torch.device("cuda:0")
    G = 4096
    eng = SearchEngine(G, board_size=bench.N, n_in_row=bench.N_IN_ROW, num_simulations=bench.S, num_top_actions=bench.K_TOP,
                       device=dev)
    sp = SelfPlayEngine(eng, "e0", seed=bench.E0_SEED, logit_div=bench.LOGIT_DIV, noise_seed=2000)
    eng.set_roots(*bench.staggered_positions(G, 0))
    traj = TrajectoryStore(eng, extra_slots=G // 2)
    buf = DeviceReplayBuffer(400_000, bench.N, device=dev)
    stats = SelfPlayStats(n_in_row=bench.N_IN_ROW, device=dev)
    state = {"batches": 0, "sizes": [], "keep": None, "with_stats": False}

    def sink(pg):                     # bench.selfplay_e2e_leg's sink, plus SelfPlayStats.add in the "with" arm
        if state["with_stats"]:
            stats.add(pg)
        buf.add_packed(pg)
        state["sizes"].append(pg.n_moves)
        if state["keep"] is not None:
            state["keep"].append(pg)
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
    state["sizes"] = []
    for r in range(args.reps):          # packed chunks are dropped after the sink: the allocator reuses their blocks
        for name in (("without", "with") if r % 2 == 0 else ("with", "without")):
            arms[name].append(run(name == "with"))
    chunk_sizes = state["sizes"]
    summary = stats.summary()

    # kernel alone: the records of one more repetition's chunks back to back in one block, and one typical chunk
    state["keep"] = []
    run(False)
    lib, stride = _lib.load(), buf.stride
    recs = torch.cat([pg.records for pg in state["keep"]])[:100_000]
    state["keep"] = None
    flags = torch.empty(recs.shape[0], dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def time_block(block, launches):
        M = int(block.shape[0])
        out = flags[:M]
        call = lambda: _lib.check(lib.gmz_records_tactics(C.c_void_p(block.data_ptr()), M, bench.N, bench.N_IN_ROW,
                                                          C.c_void_p(out.data_ptr()), C.c_void_p(stream)), "gmz_records_tactics")
        for _ in range(10):
            call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(launches):
            call()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / launches
        return {"records": M, "us_per_launch": us, "us_per_1000_records": us * 1000.0 / M}

    big = time_block(recs, args.launches)
    med_chunk = int(np.median(chunk_sizes)) if chunk_sizes else 0
    typical = time_block(recs[:max(1, med_chunk)], args.launches) if med_chunk else None
    assert torch.equal(record_flags(recs, bench.N, bench.N_IN_ROW), flags)      # repeated launches, same flags

    def spread(v):
        v = np.asarray(v)
        return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()),
                "spread_pct": float((v.max() - v.min()) / np.median(v) * 100.0), "runs": [float(x) for x in v]}

    wo, wi = spread(arms["without"]), spread(arms["with"])
    rate = wo["median"]
    out = {
        "what": "missed-win statistics on device self-play: gmz_records_tactics kernel time, and bench.py's selfplay_e2e "
                "loop with / without SelfPlayStats.add in the sink (arms alternating in one process)",
        "card": card(0),
        "config": {"games": G, "board": bench.N, "n_in_row": bench.N_IN_ROW, "num_simulations": bench.S,
                   "num_top_actions": bench.K_TOP, "evaluator": "E0 seed %d, logit_div %d" % (bench.E0_SEED, bench.LOGIT_DIV),
                   "roots": "bench.staggered_positions", "record_bytes": stride, "moves_per_game_per_rep": args.moves,
                   "reps_per_arm": args.reps},
        "kernel": {"block": big, "typical_chunk": typical, "launches": args.launches,
                   "timing": "CUDA events around back-to-back launches on the current stream; a record's kernel reads its 64 B "
                             "header and its A-byte board, about 30 MB for the block: L2-resident between launches, as "
                             "freshly packed records are",
                   "share_of_selfplay_rate": big["us_per_1000_records"] * 1e-9 * rate,
                   "chunk_records": {"median": med_chunk, "min": int(min(chunk_sizes)) if chunk_sizes else 0,
                                     "max": int(max(chunk_sizes)) if chunk_sizes else 0, "count": len(chunk_sizes)}},
        "selfplay_e2e_moves_per_sec": {"without_stats": wo, "with_stats": wi,
                                       "overhead_pct": (1.0 - wi["median"] / wo["median"]) * 100.0},
        "stats_summary_with_arm": summary,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"kernel_us_per_1000_records": big["us_per_1000_records"], "without": wo["median"], "with": wi["median"],
                      "overhead_pct": out["selfplay_e2e_moves_per_sec"]["overhead_pct"], "spread_without_pct": wo["spread_pct"],
                      "spread_with_pct": wi["spread_pct"], "card": out["card"]}))


if __name__ == "__main__":
    main()
