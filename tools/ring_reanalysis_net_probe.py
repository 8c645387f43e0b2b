"""Re-analysis of the device replay ring with the production network evaluators (mcts.resolve_searchers).

    python tools/ring_reanalysis_net_probe.py [--capacity 65536] [--az-records 16384] [--reps 3]
                                              [--out profiles/r06_ring_reanalysis_net.json]

Setup: 15x15, 400 simulations, K = 16 (bench.py's constants), engines of 4096 games with float32 accumulation, a seeded
random GomokuNetEZ at the bench's 8x128 config (HEAD_HIDDEN_DIM 64), and a DeviceReplayBuffer of `capacity` records
filled (wrapped) by E0 self-play.  Legs, each after a warm-up, repetitions alternating:
  AlphaZero : graph path (one bf16 NetworkSearch per engine, built once and reused) vs the eager callable path (the same
              folded bf16 network behind f(obs) -> (logits, values), one select -> net -> expand_backup loop), both on the
              oldest `az_records` records (widened to whole games); plus one graph run over the whole ring;
  MuZero    : ring route (buf.reanalyse with one MuZeroDeviceSearch per engine, per-game budgets in the compact arena) vs
              host route (ring -> host, reanalyse_positions with the same searchers, per-game targets, rewrite_targets);
  engines   : MuZero ring route through 1 engine vs 2 alternating engines.
Rates: records/s; simulations/s = records * S; recurrent evaluations/s (MuZero) = the sum over records of
evals_per_search(S, K, min(K, empty cells)) per second.  Memory: the arenas' bytes against the fixed nodes_per_game = S
pool those engines would hold.  The check: the two MuZero routes leave identical policy and value-target bytes, 1 and 2
engines leave identical rings, no node overflowed its budget, and each arena is no larger than its largest batch's budget
sum.  The card name and power limit are read in the same run and written beside the numbers."""
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
    ap.add_argument("--capacity", type=int, default=65536, help="ring records (the whole ring is the stretch)")
    ap.add_argument("--az-records", type=int, default=16384, help="records of the AlphaZero graph-vs-eager comparison")
    ap.add_argument("--games", type=int, default=4096, help="games per engine")
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions per arm (alternating)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_ring_reanalysis_net.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ring_reanalysis_net_probe needs a CUDA device")
    from datou_gomoku_muzero_b200.config import Config, config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.muzero import FoldedRecurrentInference, MuZeroDeviceSearch, evals_per_search
    from datou_gomoku_muzero_b200.network import FoldedInitialInference, GomokuNetEZ, NetworkSearch
    from datou_gomoku_muzero_b200.reanalysis import reanalyse_positions
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore, compute_n_step_returns, record_dtype

    dev = torch.device("cuda:0")
    N, A, S, K, G, cap = bench.N, bench.A, bench.S, bench.K_TOP, args.games, args.capacity
    mk = lambda mode="AlphaZero", accum="float64": SearchEngine(G, board_size=N, n_in_row=bench.N_IN_ROW, num_simulations=S,
                                                               num_top_actions=K, mode=mode, accum_dtype=accum, device=dev)
    eng = mk()
    sp = SelfPlayEngine(eng, "e0", seed=bench.E0_SEED, logit_div=bench.LOGIT_DIV, noise_seed=2000)
    traj = TrajectoryStore(eng, extra_slots=G // 2)
    buf = DeviceReplayBuffer(cap, N, device=dev)
    t0 = time.perf_counter()
    while len(buf) < cap or buf.sum_tree.write_ptr == 0:
        sp.play(moves_per_game=48, traj=traj, sink=buf.add_packed)
    torch.cuda.synchronize()
    fill_s = time.perf_counter() - t0
    del sp, traj, eng
    snap = buf.ring.clone()
    oldest = buf.sum_tree.write_ptr
    h0 = snap.cpu().numpy().view(record_dtype(N)).reshape(-1)[(oldest + np.arange(cap)) % cap]
    empty = (h0["board"].reshape(cap, A) == 0).sum(1)
    evals = np.array([evals_per_search(S, K, k) for k in range(K + 1)])[np.minimum(empty, K)]

    torch.manual_seed(0)
    torch.backends.cudnn.benchmark = True
    net = GomokuNetEZ(Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=A, NUM_RES_BLOCKS=8, NUM_FILTERS=128, HEAD_HIDDEN_DIM=64)).to(dev).eval()
    fi, fr = FoldedInitialInference(net, torch.bfloat16), FoldedRecurrentInference(net, torch.bfloat16)

    def initial(obs):
        p, v, h = fi(obs.to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
        return p.float().contiguous(), v.reshape(-1).float(), h

    def eager(obs):                                   # the callable path: f32 NCHW observations from the select
        p, v, _ = fi(obs.to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
        return p.float().contiguous(), v.reshape(-1).float()

    seeds = dict(noise_seed=78)

    def timed(fn):
        buf.ring.copy_(snap)
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t, out

    def alternate(arms):
        for fn in arms.values():
            timed(fn)                                 # warm-up: cuDNN plans, arenas, graph captures
        runs = {k: [] for k in arms}
        for rep in range(args.reps):
            for name in (list(arms) if rep % 2 == 0 else list(arms)[::-1]):
                runs[name].append(timed(arms[name])[0])
        return {k: spread(v) for k, v in runs.items()}

    # ---- MuZero: ring route vs host route, 1 vs 2 engines
    mz_engs = [mk("MuZero", "float32") for _ in range(2)]
    mz = [MuZeroDeviceSearch(e, initial, fr, graph=True) for e in mz_engs]

    def mz_ring():
        return buf.reanalyse(mz_engs, evaluator=mz, **seeds)

    def mz_ring_one():
        return buf.reanalyse(mz_engs[:1], evaluator=mz[:1], **seeds)

    def mz_host():
        h = buf.ring.cpu().numpy().view(record_dtype(N)).reshape(-1)
        idx = (oldest + np.arange(cap)) % cap
        r = h[idx]
        pol, val = reanalyse_positions(mz_engs, r["board"].reshape(cap, A), r["to_move"].astype(np.int8), r["last_move"],
                                       r["move_count"], evaluator=mz, cls=_mz_cls(), **seeds)
        vt = np.empty(cap, np.float32)
        starts = np.flatnonzero(r["t"] == 0).tolist()
        bounds = ([0] if not starts or starts[0] != 0 else []) + starts + [cap]
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            vt[lo:hi] = compute_n_step_returns(r["reward"][lo:hi].astype(np.float32), [np.float64(x) for x in val[lo:hi]],
                                               config.DISCOUNT, config.N_STEPS)
        buf.rewrite_targets(idx, pol, vt)
        return val

    timed(mz_ring); after_ring = buf.ring.clone()
    host_val = timed(mz_host)[1]; after_host = buf.ring.clone()
    timed(mz_ring_one); after_one = buf.ring.clone()
    P = slice(64, 64 + 8 * A)
    ring_sv = after_ring[:, 40:48].contiguous().view(torch.float64).reshape(-1).cpu().numpy()[(oldest + np.arange(cap)) % cap]
    arena_bytes = [m.pool.numel() * m.pool.element_size() for m in mz]
    fixed_bytes = [G * S * m.row_bytes for m in mz]
    need = max(int(x) for x in _batch_rows(evals, G))
    check = {"muzero_policy_bytes_identical_ring_vs_host": bool(torch.equal(after_ring[:, P], after_host[:, P])),
             "muzero_value_target_bytes_identical_ring_vs_host": bool(torch.equal(after_ring[:, 36:40], after_host[:, 36:40])),
             "muzero_search_values_identical_ring_vs_host": bool(np.array_equal(ring_sv, host_val)),
             "muzero_ring_identical_1_vs_2_engines": bool(torch.equal(after_ring, after_one)),
             "muzero_policies_changed": bool(not torch.equal(after_ring[:, P], snap[:, P])),
             "muzero_no_budget_overflow": all(int(m.overflow) == 0 for m in mz),
             "muzero_arena_within_largest_batch_budget": all(m.pool.shape[0] <= need for m in mz)}
    del after_ring, after_host, after_one
    mz_route = alternate({"ring": mz_ring, "host": mz_host})
    mz_eng = alternate({"two_engines": mz_ring, "one_engine": mz_ring_one})
    check["muzero_no_budget_overflow"] = check["muzero_no_budget_overflow"] and all(int(m.overflow) == 0 for m in mz)
    del mz
    torch.cuda.empty_cache()

    # ---- AlphaZero: graph (NetworkSearch) vs eager callable
    az_engs = [mk("AlphaZero", "float32") for _ in range(2)]
    ns = [NetworkSearch(e, net) for e in az_engs]
    torch.backends.cudnn.benchmark = True
    az_n = {}

    def az(evaluator, count):
        def run():
            start, n = buf.reanalyse(az_engs, count=count, evaluator=evaluator, **seeds)
            az_n[count] = n
        return run
    az_cmp = alternate({"graph": az(ns, args.az_records), "eager": az(eager, args.az_records)})
    az_full_s, _ = timed(az(ns, None))
    n_az = az_n[args.az_records]

    rec = {k: cap / v["median"] for k, v in mz_route.items()}
    out = {
        "what": "Surge re-analysis of a wrapped device replay ring with a seeded random GomokuNetEZ 8x128: AlphaZero graph "
                "path (NetworkSearch) vs eager callable, MuZero ring route vs host route (MuZeroDeviceSearch with per-game "
                "node budgets), 1 vs 2 alternating engines; arms alternating after a warm-up",
        "card": card(0),
        "config": {"board": N, "n_in_row": bench.N_IN_ROW, "num_simulations": S, "num_top_actions": K, "games_per_engine": G,
                   "ring_capacity": cap, "records_reanalysed_muzero": cap, "records_reanalysed_alphazero_comparison": n_az,
                   "network": "GomokuNetEZ 8 blocks x 128 filters, head hidden 64, torch.manual_seed(0), bf16 folded",
                   "accum_dtype": "float32", "noise_seed": seeds["noise_seed"], "reps_per_arm": args.reps,
                   "fill": "E0 self-play of %d games (seed %d), %.1f s" % (G, bench.E0_SEED, fill_s),
                   "records_with_fewer_than_K_empty_cells": int((empty < K).sum())},
        "alphazero": {"seconds": az_cmp,
                      "records_per_sec": {k: n_az / v["median"] for k, v in az_cmp.items()},
                      "sims_per_sec": {k: n_az * S / v["median"] for k, v in az_cmp.items()},
                      "eager_over_graph": az_cmp["eager"]["median"] / az_cmp["graph"]["median"],
                      "graph_whole_ring": {"seconds": az_full_s, "records_per_sec": cap / az_full_s,
                                           "sims_per_sec": cap * S / az_full_s, "runs": 1}},
        "muzero": {"seconds": mz_route,
                   "records_per_sec": rec,
                   "sims_per_sec": {k: v * S for k, v in rec.items()},
                   "recurrent_evals_per_sec": {k: int(evals.sum()) / v["median"] for k, v in mz_route.items()},
                   "recurrent_evals_in_stretch": int(evals.sum()),
                   "host_over_ring": mz_route["host"]["median"] / mz_route["ring"]["median"],
                   "engines": {"seconds": mz_eng,
                               "records_per_sec": {k: cap / v["median"] for k, v in mz_eng.items()},
                               "one_over_two": mz_eng["one_engine"]["median"] / mz_eng["two_engines"]["median"]},
                   "memory": {"arena_bytes_per_engine": arena_bytes, "fixed_pool_bytes_per_engine": fixed_bytes,
                              "fixed_over_arena": sum(fixed_bytes) / sum(arena_bytes),
                              "row_bytes": fixed_bytes[0] // (G * S),
                              "largest_batch_rows": need}},
        "check": check,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"az_graph_s": az_cmp["graph"]["median"], "az_eager_s": az_cmp["eager"]["median"],
                      "mz_ring_s": mz_route["ring"]["median"], "mz_host_s": mz_route["host"]["median"],
                      "mz_one_engine_s": mz_eng["one_engine"]["median"], "arena_gb": sum(arena_bytes) / 1e9,
                      "fixed_gb": sum(fixed_bytes) / 1e9, "check": check, "card": out["card"]}))
    assert all(check.values()), check


def _mz_cls():
    from datou_gomoku_muzero_b200.mcts import MuZeroMCTS
    return MuZeroMCTS


def _batch_rows(evals, G):
    """Rows each batch of G consecutive records needs (padding games: one row each)."""
    rows = evals + 1
    return [rows[s:s + G].sum() + (G - len(rows[s:s + G])) for s in range(0, len(rows), G)]


if __name__ == "__main__":
    main()
