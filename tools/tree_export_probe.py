"""Cost of search inspection (gmz_tree_export) at the bench's size, next to the search it inspects.

    python tools/tree_export_probe.py [--games 4096] [--launches 200] [--out profiles/r08_tree_export.json]

Setup: 15x15, 400 simulations, K = 16, float32 accumulation, dense E0 logits, one fused search (gmz_search_e0) of G
random mid-game roots.  Timed with CUDA events: the search itself (`--searches` repetitions) and `--launches` exports of
the finished trees into preallocated buffers after `--warmup` untimed ones.  Bytes are computed from shapes and the
exported node counts: what the kernel reads of the workspace and writes into the caller's buffers.  The trees' combined
size (~840 MB of child rows at 4096 x 400 nodes x 256 shorts, plus the scattered logits) is far beyond the 126 MB L2,
so every export reads them from HBM.  The card name and power limit are read in the same run and written beside the
numbers."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np
import torch

from stats_probe import card


def events_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=400)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--searches", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_tree_export.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tree_export_probe needs a CUDA device")
    from datou_gomoku_muzero_b200.engine import SearchEngine
    G, N, S, K, seed = args.games, 15, args.sims, 16, 7
    A = N * N
    rs = np.random.RandomState(0)
    boards = np.zeros((G, A), np.int8)
    players = np.ones(G, np.int8); last = np.full(G, -1, np.int32); mc = np.zeros(G, np.int32)
    for g in range(G):
        p = 1
        for a in rs.permutation(A)[:rs.randint(0, 40)]:
            boards[g, a] = p; last[g] = a; p = -p; mc[g] += 1
        players[g] = p
    gumbel = torch.from_numpy(rs.gumbel(0, 1, (G, A))).cuda()
    boards, players, last, mc = (torch.from_numpy(x).cuda() for x in (boards, players, last, mc))
    eng = SearchEngine(G, board_size=N, num_simulations=S, num_top_actions=K, accum_dtype="float32")

    def search():
        eng.set_roots(boards, players, last, mc)
        eng.search_e0(gumbel, seed, 0)

    search()                                                    # warm-up (module load)
    search_ms = events_ms(search, args.searches)
    tr = eng.export_tree()
    for _ in range(args.warmup):
        eng.export_tree(out=tr)
    export_ms = events_ms(lambda: eng.export_tree(out=tr), args.launches)

    nodes = int(tr.num_nodes.sum().item())
    trees = int((tr.num_nodes > 0).sum().item())
    AP = 128 * ((A + 127) // 128)
    read = (trees * A * 4                                       # root logit rows
            + nodes * AP * 2                                    # child rows (every node's row is scanned)
            + (nodes - trees) * 32                              # one 32-byte sector of the parent's logit row per child
            + nodes * (4 + 8)                                   # visits, value_sum
            + G * 1024)                                         # GState (upper bound: the whole record)
    written = G * S * (4 * 4 + 8 * 2 + 4) + G * (4 * 2 + 4 * 3 + 8 * 2 + 4 * 3) + G * K * (4 + 8 + 4 + 4) + G * A * 4
    out = dict(
        setup=dict(games=G, board=N, sims=S, K=K, accum="float32", logits="dense E0", search="gmz_search_e0 (fused)",
                   export_launches=args.launches, warmup=args.warmup, searches_timed=args.searches),
        card=card(torch.cuda.current_device()),
        search_ms=round(search_ms, 3),
        export_ms=round(export_ms, 4),
        export_share_of_search=round(export_ms / search_ms, 5),
        nodes=nodes, trees=trees,
        bytes_read=read, bytes_written=written,
        effective_GBps=round((read + written) / (export_ms * 1e-3) / 1e9, 1),
        note="CUDA-event times; bytes from shapes and the exported node counts (reads at 32-byte sector granularity "
             "for the scattered parent-logit gathers, the GState record as a whole)")
    print(json.dumps(out), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
