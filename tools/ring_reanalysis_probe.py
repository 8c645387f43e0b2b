"""Re-analysis of the device replay ring in place (DeviceReplayBuffer.reanalyse) against the host route.

    python tools/ring_reanalysis_probe.py [--capacity 1000000] [--reps 3] [--out profiles/r04_ring_reanalysis.json]

Setup: 15x15, 400 simulations (bench.py's constants), a DeviceReplayBuffer of `capacity` records filled by E0 self-play
of 4096 games through sp.play(sink=buf.add_packed), 4 re-analysis engines of 4096 games, E0 with a new seed as "the
latest model".  Both routes start from the same snapshot of the ring and use the same seeds:
  ring route : buf.reanalyse(engines)  -- roots loaded from the records, search, write-back and n-step targets on the GPU;
  host route : ring -> host, roots from the record headers and boards, reanalysis.reanalyse_positions (pinned staging,
               H2D, search, D2H), per-game compute_n_step_returns with float32 rewards, buf.rewrite_targets.
Runs alternate (one warm-up each, then `reps` each); wall-clock medians and spread.  Bytes over PCIe are computed from
the shapes each route copies.  The three new kernels are timed alone with CUDA events over back-to-back launches.  The
check: both routes leave identical policy and value_target bytes (and the host route leaves every other byte but the
header's search_value, which only the ring route rewrites, as the ring route does).
The card name and power limit are read in the same run and written beside the numbers."""
import argparse
import ctypes as C
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--capacity", type=int, default=1_000_000, help="ring records (filled completely before the runs)")
    ap.add_argument("--games", type=int, default=4096, help="games per engine (self-play and re-analysis)")
    ap.add_argument("--engines", type=int, default=4, help="re-analysis engines")
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions per route (alternating)")
    ap.add_argument("--launches", type=int, default=50, help="launches per kernel in the kernel timing")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_ring_reanalysis.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ring_reanalysis_probe needs a CUDA device")
    from datou_gomoku_muzero_b200 import _lib
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.reanalysis import reanalyse_positions
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore, compute_n_step_returns, record_dtype

    dev = torch.device("cuda:0")
    N, A, G, cap = bench.N, bench.A, args.games, args.capacity
    mk = lambda: SearchEngine(G, board_size=N, n_in_row=bench.N_IN_ROW, num_simulations=bench.S, num_top_actions=bench.K_TOP,
                              device=dev)
    eng = mk()
    sp = SelfPlayEngine(eng, "e0", seed=bench.E0_SEED, logit_div=bench.LOGIT_DIV, noise_seed=2000)
    traj = TrajectoryStore(eng, extra_slots=G // 2)
    buf = DeviceReplayBuffer(cap, N, device=dev)
    t0 = time.perf_counter()
    while len(buf) < cap:
        sp.play(moves_per_game=48, traj=traj, sink=buf.add_packed)
    torch.cuda.synchronize()
    fill_s = time.perf_counter() - t0
    del sp, traj, eng
    engs = [mk() for _ in range(args.engines)]
    snap = buf.ring.clone()
    stride, lib = buf.stride, _lib.load()
    seeds = dict(eval_seed=bench.E0_SEED + 1, logit_div=bench.LOGIT_DIV, noise_seed=78)

    def ring_route():
        return buf.reanalyse(engs, **seeds)

    def host_route():
        h = buf.ring.cpu().numpy().view(record_dtype(N)).reshape(-1)           # D2H of every record
        start = buf.sum_tree.write_ptr if len(buf) == cap else 0
        n = len(buf)
        idx = (start + np.arange(n)) % cap
        r = h[idx]
        pol, val = reanalyse_positions(engs, r["board"].reshape(n, A), r["to_move"].astype(np.int8), r["last_move"],
                                       r["move_count"], **seeds)
        vt = np.empty(n, np.float32)
        starts = np.flatnonzero(r["t"] == 0).tolist()
        bounds = ([0] if not starts or starts[0] != 0 else []) + starts + [n]
        for lo, hi in zip(bounds[:-1], bounds[1:]):                          # the per-game target loop
            vt[lo:hi] = compute_n_step_returns(r["reward"][lo:hi].astype(np.float32), [np.float64(x) for x in val[lo:hi]],
                                               config.DISCOUNT, config.N_STEPS)
        buf.rewrite_targets(idx, pol, vt)
        return start, n, len(bounds) - 1

    def timed(fn):
        buf.ring.copy_(snap)
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t, out

    timed(ring_route); timed(host_route)                                    # warm-up of both routes
    runs = {"ring": [], "host": []}
    check = None
    for rep in range(args.reps):
        for name in (("ring", "host") if rep % 2 == 0 else ("host", "ring")):
            dt, out = timed(ring_route if name == "ring" else host_route)
            runs[name].append(dt)
            if name == "ring":
                ring_start, n = out
                if rep == 0:
                    after_ring = buf.ring.clone()
            else:
                n_games = out[2]
                if rep == 0:
                    after_host = buf.ring.clone()
        if rep == 0:
            P = slice(64, 64 + 8 * A)
            check = {"policy_bytes_identical": bool(torch.equal(after_ring[:, P], after_host[:, P])),
                     "value_target_bytes_identical": bool(torch.equal(after_ring[:, 36:40], after_host[:, 36:40])),
                     "other_bytes_identical": bool(torch.equal(after_ring[:, :36], after_host[:, :36])
                                                   and torch.equal(after_ring[:, 48:64], after_host[:, 48:64])
                                                   and torch.equal(after_ring[:, 64 + 8 * A:], after_host[:, 64 + 8 * A:])),
                     "policies_changed_by_new_evaluator": bool(not torch.equal(after_ring[:, P], snap[:, P])),
                     "search_value_rewritten_by_ring_route_only": bool(not torch.equal(after_ring[:, 40:48], snap[:, 40:48])
                                                                      and torch.equal(after_host[:, 40:48], snap[:, 40:48]))}
            del after_ring, after_host
    assert check["policy_bytes_identical"] and check["value_target_bytes_identical"] and check["other_bytes_identical"], check

    # the three new kernels alone: CUDA events around back-to-back launches on the current stream
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    e = engs[0]
    dpow = torch.tensor([config.DISCOUNT ** i for i in range(config.N_STEPS + 1)], dtype=torch.float64, device=dev)
    ringp = C.c_void_p(buf.ring.data_ptr())
    calls = {
        "k_set_roots_records": (lambda: e.set_roots_from_records(buf.ring, cap, ring_start, G), G),
        "k_records_writeback": (lambda: _lib.check(lib.gmz_records_writeback(ringp, cap, N, ring_start, G, C.c_void_p(e.policy.data_ptr()),
                                                                            C.c_void_p(e.value.data_ptr()), stream)), G),
        "k_records_retarget": (lambda: _lib.check(lib.gmz_records_retarget(ringp, cap, N, ring_start, n, C.c_void_p(dpow.data_ptr()),
                                                                          int(config.N_STEPS), stream)), n),
    }
    kern = {}
    for name, (call, recs) in calls.items():
        for _ in range(5):
            call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.launches):
            call()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / args.launches
        kern[name] = {"records_per_launch": recs, "us_per_launch": us}
    batches = (n + G - 1) // G
    kern_total_s = (batches * (kern["k_set_roots_records"]["us_per_launch"] + kern["k_records_writeback"]["us_per_launch"])
                    + kern["k_records_retarget"]["us_per_launch"]) * 1e-6

    def spread(v):
        v = np.asarray(v)
        return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()),
                "spread_pct": float((v.max() - v.min()) / np.median(v) * 100.0), "runs": [float(x) for x in v]}

    rs, hs = spread(runs["ring"]), spread(runs["host"])
    nsteps = int(config.N_STEPS)
    pcie = {
        "ring": {"h2d": (nsteps + 1) * 8, "d2h": 0,
                 "what": "discount powers for the target kernel; the default stretch needs no boundary read"},
        "host": {"d2h": cap * stride + n * (8 * A + 8 + 4), "h2d": n * (A + 1 + 4 + 4) + n * (8 + 8 * A + 4),
                 "what": "ring -> host (every record); roots H2D (board, player, last move, move count); policies, values, "
                         "actions D2H; rewrite_targets H2D (positions, policies, value targets)"},
    }
    out = {
        "what": "Surge re-analysis of a full replay ring in place (DeviceReplayBuffer.reanalyse) vs the host route (records -> "
                "host roots -> reanalyse_positions -> per-game compute_n_step_returns -> rewrite_targets), same snapshot, same "
                "seeds, routes alternating",
        "card": card(0),
        "config": {"board": N, "n_in_row": bench.N_IN_ROW, "num_simulations": bench.S, "num_top_actions": bench.K_TOP,
                   "games_per_engine": G, "engines": args.engines, "ring_capacity": cap, "record_bytes": stride,
                   "records_reanalysed": n, "games_in_ring": n_games, "evaluator": "E0 seed %d, logit_div %d" % (seeds["eval_seed"],
                                                                                                               seeds["logit_div"]),
                   "noise_seed": seeds["noise_seed"], "n_steps": nsteps, "discount": config.DISCOUNT,
                   "fill": "E0 self-play of %d games (seed %d) through sp.play(sink=buf.add_packed), %.1f s" % (G, bench.E0_SEED, fill_s),
                   "reps_per_route": args.reps},
        "seconds": {"ring_route": rs, "host_route": hs, "host_over_ring": hs["median"] / rs["median"]},
        "records_per_sec": {"ring_route": n / rs["median"], "host_route": n / hs["median"]},
        "pcie_bytes": pcie,
        "kernels": dict(kern, batches=batches, launches=args.launches,
                        total_in_ring_route_s=kern_total_s, share_of_ring_route=kern_total_s / rs["median"],
                        timing="CUDA events around back-to-back launches of one kernel on the current stream; set_roots / "
                               "write-back on one batch of G records, the target kernel on the whole stretch"),
        "check": check,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"ring_s": rs["median"], "host_s": hs["median"], "ring_spread_pct": rs["spread_pct"],
                      "host_spread_pct": hs["spread_pct"], "kernel_share": out["kernels"]["share_of_ring_route"],
                      "check": check, "card": out["card"]}))


if __name__ == "__main__":
    main()
