"""Checkpoint and restore of a full device replay ring (DeviceReplayBuffer.state_dict / load_state_dict).

    python tools/ring_checkpoint_probe.py [--capacity 1000000] [--reps 3] [--out profiles/r05_ring_checkpoint.json]

Setup: 15x15, 400 simulations (bench.py's constants), a DeviceReplayBuffer of `capacity` records filled by E0 self-play
of 4096 games through sp.play(sink=buf.add_packed), then (PER on) a few update_priorities calls with random TD errors.  Each rep
runs the four legs in order -- state_dict() (ends in the host copy), torch.save to a file, torch.load(weights_only=True),
load_state_dict() into a second buffer of the same capacity followed by a device synchronise -- after one warm-up rep;
wall-clock medians and spread.  The file goes to a temporary directory that is deleted at the end (torch.save / torch.load
times are through the page cache of that machine).  The two kernels are timed alone with CUDA events over back-to-back
launches.  Bytes moved each way are computed from the dict's tensors.  The check: the restored buffer equals the saved
one on every record's bytes 0 .. 64+21A, the tree, write_ptr, count and max_priority.
The card name and power limit are read in the same run and written beside the numbers."""
import argparse
import ctypes as C
import json
import os
import sys
import tempfile
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
    ap.add_argument("--games", type=int, default=4096, help="self-play games")
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions of each leg (legs alternate)")
    ap.add_argument("--launches", type=int, default=20, help="launches per kernel in the kernel timing")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_ring_checkpoint.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ring_checkpoint_probe needs a CUDA device")
    from datou_gomoku_muzero_b200 import _lib
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore

    config.ENABLE_PER = True                                   # priorities from update_priorities are part of the state
    dev = torch.device("cuda:0")
    N, A, G, cap = bench.N, bench.A, args.games, args.capacity
    eng = SearchEngine(G, board_size=N, n_in_row=bench.N_IN_ROW, num_simulations=bench.S, num_top_actions=bench.K_TOP, device=dev)
    sp = SelfPlayEngine(eng, "e0", seed=bench.E0_SEED, logit_div=bench.LOGIT_DIV, noise_seed=2000)
    traj = TrajectoryStore(eng, extra_slots=G // 2)
    buf = DeviceReplayBuffer(cap, N, device=dev)
    t0 = time.perf_counter()
    while len(buf) < cap:
        sp.play(moves_per_game=48, traj=traj, sink=buf.add_packed)
    torch.cuda.synchronize()
    fill_s = time.perf_counter() - t0
    del sp, traj, eng
    g = torch.Generator(device=dev).manual_seed(0)
    for _ in range(8):                                         # a tree that is not all max_priority
        _, idx, _ = buf.sample(4096, u01=torch.rand(4096, dtype=torch.float64, device=dev, generator=g))
        buf.update_priorities(idx, torch.randn(4096, device=dev, generator=g))
    dst = DeviceReplayBuffer(cap, N, device=dev)
    stride, n = buf.stride, len(buf)

    def sync_timed(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t, out

    legs = {"state_dict": [], "torch_save": [], "torch_load": [], "load_state_dict": []}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "ring.pt")
        for rep in range(args.reps + 1):                       # rep 0: warm-up
            dt = {}
            dt["state_dict"], sd = sync_timed(buf.state_dict)
            dt["torch_save"], _ = sync_timed(lambda: torch.save(sd, path))
            file_bytes = os.path.getsize(path)
            del sd
            dt["torch_load"], sd = sync_timed(lambda: torch.load(path, weights_only=True))
            dt["load_state_dict"], _ = sync_timed(lambda: dst.load_state_dict(sd))
            if rep > 0:
                for k, v in dt.items():
                    legs[k].append(v)
    tensors = {k: v for k, v in sd.items() if torch.is_tensor(v)}
    dict_bytes = sum(v.numel() * v.element_size() for v in tensors.values())
    n_seg = int(sd["seg_start"].numel())
    body = 64 + 21 * A
    check = {"record_bytes_identical": bool(torch.equal(buf.ring[:, :body], dst.ring[:, :body])),
             "tree_identical": bool(torch.equal(buf.sum_tree.tree, dst.sum_tree.tree)),
             "write_ptr_count_identical": (buf.sum_tree.write_ptr, len(buf)) == (dst.sum_tree.write_ptr, len(dst)),
             "max_priority_identical": bool(torch.equal(buf.max_priority, dst.max_priority))}
    assert all(check.values()), check

    # the two kernels alone: CUDA events around back-to-back launches on the current stream
    lib, stream = _lib.load(), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())
    oldest = buf.sum_tree.write_ptr if n == cap else 0
    hd = torch.empty((n, 64), dtype=torch.uint8, device=dev)
    pol = torch.empty((n, A), dtype=torch.float64, device=dev)
    fl = torch.empty(n, dtype=torch.uint8, device=dev)
    seg, base = sd["seg_start"].to(dev), sd["base_boards"].to(dev)
    calls = {
        "k_records_compact": lambda: _lib.check(lib.gmz_records_compact(p(buf.ring), cap, N, oldest, n, p(hd), p(pol), p(fl), stream)),
        "k_records_expand": lambda: _lib.check(lib.gmz_records_expand(p(hd), p(pol), n, p(seg), p(base), n_seg, 0, N, p(dst.ring), cap,
                                                                      oldest, stream)),
    }
    traffic = {   # bytes each kernel must move: compact reads the record's meaningful bytes + its predecessor's header and
                  # board, writes header + policy + flag; expand reads header + policy (+ the base boards), writes records
        "k_records_compact": n * (body + 64 + A) + n * (64 + 8 * A + 1),
        "k_records_expand": n * (64 + 8 * A) + n_seg * A + n * stride,
    }
    kern = {}
    for name, call in calls.items():
        for _ in range(3):
            call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.launches):
            call()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.launches
        kern[name] = {"ms_per_launch": ms, "records": n, "bytes_moved": traffic[name],
                      "achieved_TB_per_s": traffic[name] / (ms * 1e-3) / 1e12}
    assert torch.equal(buf.ring[:, :body], dst.ring[:, :body])

    def spread(v):
        v = np.asarray(v)
        return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()),
                "spread_pct": float((v.max() - v.min()) / np.median(v) * 100.0), "runs": [float(x) for x in v]}

    out = {
        "what": "Checkpoint and restore of a full device replay ring: DeviceReplayBuffer.state_dict() -> torch.save -> "
                "torch.load(weights_only=True) -> load_state_dict() into a second buffer of the same capacity",
        "card": card(0),
        "config": {"board": N, "num_simulations": bench.S, "ring_capacity": cap, "records": n, "record_bytes": stride,
                   "segments": n_seg, "fill": "E0 self-play of %d games (seed %d) through sp.play(sink=buf.add_packed), %.1f s"
                   % (G, bench.E0_SEED, fill_s), "reps_per_leg": args.reps, "warmup_reps": 1},
        "seconds": {k: spread(v) for k, v in legs.items()},
        "timing": "host clock; state_dict ends in its host copy, load_state_dict in a device synchronise; torch.save / "
                  "torch.load through a temporary file (page cache), deleted at the end",
        "bytes": {"raw_ring": n * stride, "state_dict_tensors": dict_bytes, "file": file_bytes,
                  "raw_over_dict": n * stride / dict_bytes,
                  "d2h_in_state_dict": dict_bytes, "h2d_in_load_state_dict": dict_bytes,
                  "per_tensor": {k: v.numel() * v.element_size() for k, v in tensors.items()}},
        "kernels": dict(kern, launches=args.launches,
                        timing="CUDA events around back-to-back launches of one kernel over the whole live ring; bytes are "
                               "the minimum the kernel must move, computed from the shapes"),
        "check": check,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"seconds": {k: v["median"] for k, v in out["seconds"].items()},
                      "spread_pct": {k: v["spread_pct"] for k, v in out["seconds"].items()},
                      "kernels_ms": {k: kern[k]["ms_per_launch"] for k in calls}, "raw_over_dict": out["bytes"]["raw_over_dict"],
                      "check": check, "card": out["card"]}))


if __name__ == "__main__":
    main()
