#!/usr/bin/env python
"""Headline benchmark: MCTS simulations/s (and self-play moves/s) of AlphaZero-mode 15x15 Gomoku
self-play, 400 simulations per move, 4096 concurrent games per GPU (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--games G] [--dump-outputs DIR]

A "step" is one self-play move for every game on the GPU: Gumbel noise, one full 400-simulation
search per game, decision, do_move + win/draw detection, restart of finished games.  Rank 0
prints ONE JSON line; with --dump-outputs it also writes the last step's outputs to DIR (dump_last_step).
`--impl reference` times the UNMODIFIED reference (baseline/_ref, installed by baseline/install_reference.py; its own AlphaZeroMCTS.search in one process per host core, plus its production
topology universal_worker x W + inference_server_worker at N = 1) on the same config; the C port of the search
(oracle/) is timed beside it as a second figure, and stands in alone if baseline/_ref is absent.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: the benchmark writes nothing into it

N, N_IN_ROW, S, K_TOP = 15, 5, 400, 16
A = N * N
E0_SEED, LOGIT_DIV = 2024, 16


def algorithmic_bytes_per_sim(mean_depth: float) -> float:
    """SURVEY.md section 8(d): (d-1)(16A + ceil(A/8) + 16) + 32A + 26d + 220 bytes per AZ simulation."""
    d = mean_depth
    return (d - 1.0) * (16 * A + (A + 7) // 8 + 16) + 32 * A + 26 * d + 220


def staggered_positions(G, rank, rs=None):
    """Synthetic mid-game roots: game g starts with (g*37) % 160 random stones, colours alternating."""
    rs = rs or np.random.RandomState(1234 + rank)
    boards = np.zeros((G, A), np.int8)
    players = np.ones(G, np.int8)
    last = np.full(G, -1, np.int32)
    mc = np.zeros(G, np.int32)
    for g in range(G):
        k = (g * 37) % 160
        cells = rs.permutation(A)[:k]
        boards[g, cells[0::2]] = 1
        boards[g, cells[1::2]] = -1
        players[g] = 1 if k % 2 == 0 else -1
        last[g] = cells[-1] if k else -1
        mc[g] = k
    return boards, players, last, mc


WORKLOAD = ("AlphaZero-mode 15x15 Gomoku self-play, 400 sims/move, 4096 concurrent games per GPU "
            "(BASELINE configs[1]), E0 fixed deterministic evaluator")


def bench_config(games):
    """The workload object both arms (`--impl ours` / `--impl reference`) print, byte for byte; what differs
    between the arms (how a step is carried out) is reported under `notes`."""
    return {"workload": WORKLOAD, "games_per_gpu": games, "board": N, "n_in_row": N_IN_ROW, "num_simulations": S,
            "num_top_actions": K_TOP, "evaluator": "E0 seed %d, quantised logits k/%d" % (E0_SEED, LOGIT_DIV),
            "roots": "staggered synthetic mid-game positions (0..159 stones)",
            "l2": "GPU arm: node pools (4 GB per GPU) exceed the 126 MB L2, no explicit flush; CPU arm: n/a"}


PLAY_KERNEL_SOURCES = ("gmz_common.cuh", "gmz_tree.cuh", "gmz_play.cuh", "gmz_play_inst.cu", "gmz_internal.h")


def _strip_comments(text):
    import re
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"//[^\n]*", "", text)
    return "\n".join(l.rstrip() for l in text.split("\n") if l.strip())


def kernel_source_sha(read=None):
    """Hash of the sources the play kernel is compiled from, comments and blank lines removed: stamps `roofline.traffic`
    (an ncu measurement) with the kernel it was taken on.  `read(name) -> str` overrides where the sources come from."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "datou_gomoku_muzero_b200", "csrc")
    for f in PLAY_KERNEL_SOURCES:
        h.update(_strip_comments(read(f) if read else open(os.path.join(d, f)).read()).encode())
    return h.hexdigest()[:16]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def _nvml(self):
        """Fast path: NVML in-process (a sample every few ms); None if NVML cannot be used."""
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(torch.cuda.get_device_properties(self.index).uuid)).encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            return pynvml, h
        except Exception:
            return None

    def run(self):
        nv = self._nvml()
        bits = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))
        while not self.stop_flag and nv is not None:
            try:
                pynvml, h = nv
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                self.samples.append([str(sm), str(mx), str(pw)] + [("Active" if r & b else "Not Active") for b, _ in bits])
            except Exception:
                nv = None
                break
            time.sleep(0.005)
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def port_leg(budget_s, threads=None):
    """The C port of the reference search (oracle/gmz_oracle.c, OpenMP over games) on the host threads: a bounded
    sample of the workload, `budget_s` seconds of searches."""
    from oracle import oracle
    threads = threads or host_threads()
    games = threads * 8
    cfg = oracle.make_config(board_size=N, n_in_row=N_IN_ROW, num_simulations=S, num_top_actions=K_TOP,
                             eval_seed=E0_SEED, logit_div=LOGIT_DIV)
    boards, players, last, mc = staggered_positions(games, 0)
    rs = np.random.RandomState(7)
    oracle.search_batch(cfg, boards, players, last, mc, rs.gumbel(0, 1, (games, A)), n_threads=threads, want_visits=False)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s:
        oracle.search_batch(cfg, boards, players, last, mc, rs.gumbel(0, 1, (games, A)), n_threads=threads, want_visits=False)
        n += 1
    dt = time.perf_counter() - t0
    return {"value": games * S * n / dt, "unit": "sims/s", "cores": threads, "kind": "port",
            "sample": f"{n} batches x {games} searches of 15x15/400 sims (E0) on {threads} threads, {dt:.1f} s"}


def reference_leg(steps, warmup, threads=None, with_config1=True):
    """The unmodified reference (baseline/_ref): one process per host thread, each running AlphaZeroMCTS.search
    with E0 behind the reference's own queue protocol.  None if baseline/_ref is absent."""
    from baseline import ref_runner
    if not ref_runner.available():
        return None
    threads = threads or host_threads()
    r = ref_runner.tree_only(threads, steps, warmup=warmup, N=N, S=S, K=K_TOP, e0_seed=E0_SEED, logit_div=LOGIT_DIV)
    out = {"value": r["sims_per_sec"], "unit": "sims/s", "cores": threads, "kind": "reference", "cpu_model": cpu_model(),
           "moves_per_sec": r["moves_per_sec"], "ms_per_step": r["ms_per_step"],
           "per_process_sims_per_sec": r["per_process_sims_per_sec"],
           "sample": "%d steps x %d processes x 1 search of 15x15/400 sims: unmodified reference AlphaZeroMCTS.search "
                     "(baseline/_ref/mcts.py), E0 in-process, %.1f s" % (steps, threads, r["seconds"])}
    if with_config1:
        c1 = ref_runner.tree_only(1, 30, warmup=2, N=9, S=100, K=K_TOP, e0_seed=E0_SEED, logit_div=LOGIT_DIV)
        out["config1"] = {"workload": "BASELINE configs[0]: 9x9, 100 sims, ONE reference worker process (E0 in-process)",
                          "sims_per_sec": c1["sims_per_sec"], "moves_per_sec": c1["moves_per_sec"]}
    return out


def run_reference(args):
    """CPU arm (rank 0 only).  `value` = the unmodified reference on every host thread when baseline/_ref is
    present (kind "reference"), else the C port (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    ref = None
    try:
        ref = reference_leg(args.steps, max(1, min(args.warmup, 2)), threads)
    except Exception as ex:
        ref = None
        print("reference arm: baseline/_ref failed (%r); falling back to the C port" % (ex,), file=sys.stderr)
    port = port_leg(5.0 if ref is not None else max(5.0, args.cpu_seconds), threads)
    port["cpu_model"] = cpu_model()
    main = ref if ref is not None else port
    line = {
        "impl": "reference", "metric": "mcts_sims_per_sec", "value": main["value"], "unit": "sims/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": main.get("ms_per_step"), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "moves_per_sec": main["value"] / S,
        "config": bench_config(args.games),
        "notes": "each step is a bounded sample of the workload: one 400-simulation search per host process "
                 "(the reference is one Python process per core); float64 tree arithmetic (E0 hands Python floats)",
        "cpu_baseline": dict(main, port=port) if ref is not None else port,
        "e2e": {"value": main["value"], "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}
    if ref is not None and args.gpus == 1 and args.ref_topology_seconds > 0:
        try:        # the reference's production topology, with its own network on the GPU (reported, not the headline)
            from baseline import ref_runner
            line["reference_topology"] = ref_runner.topology(seconds=args.ref_topology_seconds, n_workers=max(1, threads - 2),
                                                             N=N, S=S, K=K_TOP)
        except Exception as ex:
            line["reference_topology"] = {"error": repr(ex)[:300]}
        # BASELINE.md section 4, items 1 (E1) and 3: config 1 with the reference's network answering in-process, and the
        # MuZero-mode counterparts (tree only with E0 on every host thread; the production topology for half the time)
        extras = {
            "config1_net": lambda: ref_runner.inprocess_net(seconds=8.0, N=9, S=100, K=K_TOP, mode="AlphaZero"),
            "config1_net_muzero": lambda: ref_runner.inprocess_net(seconds=8.0, N=9, S=100, K=K_TOP, mode="MuZero"),
            "muzero_tree_only": lambda: dict(ref_runner.tree_only(threads, 3, warmup=1, N=N, S=S, K=K_TOP, mode="MuZero", e0_seed=E0_SEED,
                                                                  logit_div=LOGIT_DIV),
                                             what="unmodified reference MuZeroMCTS.search, 15x15 / 400 sims, E0 behind its queue protocol "
                                                  "in-process, one process per host thread"),
            "reference_topology_muzero": lambda: ref_runner.topology(seconds=args.ref_topology_seconds / 2, n_workers=max(1, threads - 2),
                                                                     N=N, S=S, K=K_TOP, mode="MuZero"),
        }
        for name, fn in extras.items():
            try:
                line[name] = fn()
            except Exception as ex:
                line[name] = {"error": repr(ex)[:300]}
    print(json.dumps(line))


def host_threads():
    """Host threads this process may use (torchrun exports OMP_NUM_THREADS=1; the CPU arm ignores that:
    only rank 0 runs it, so it gets the whole box)."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except Exception:
        n = max(1, os.cpu_count() or 1)
    cap = int(os.environ.get("GMZ_BENCH_MAX_PROCS", "0") or 0)          # tests only
    return min(n, cap) if cap > 0 else n


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def config1_port_leg():
    """BASELINE configs[0]: 9x9, N_IN_ROW=5, 100 simulations, ONE self-play worker (single host thread of
    the CPU port), timed for context beside the reference's own figure."""
    from oracle import oracle
    n, s = 9, 100
    cfg = oracle.make_config(board_size=n, n_in_row=5, num_simulations=s, num_top_actions=K_TOP, eval_seed=E0_SEED)
    rs = np.random.RandomState(3)
    boards = np.zeros((64, n * n), np.int8)
    pl, lm, mc = np.ones(64, np.int8), np.full(64, -1, np.int32), np.zeros(64, np.int32)
    oracle.search_batch(cfg, boards, pl, lm, mc, rs.gumbel(0, 1, (64, n * n)), n_threads=1, want_visits=False)
    t0, k = time.perf_counter(), 0
    while time.perf_counter() - t0 < 2.0:
        oracle.search_batch(cfg, boards, pl, lm, mc, rs.gumbel(0, 1, (64, n * n)), n_threads=1, want_visits=False)
        k += 1
    dt = time.perf_counter() - t0
    return {"workload": "9x9, 100 sims, one worker (CPU port, 1 thread, E0)", "sims_per_sec": 64 * k * s / dt,
            "moves_per_sec": 64 * k / dt}


def cpu_baseline_leg(budget_s=10.0):
    """Reported on rank 0 at N = 1: the unmodified reference on the host cores (bounded sample), the C port as a
    second figure."""
    threads = host_threads()
    ref = None
    try:
        ref = reference_leg(max(2, int(budget_s // 1.5)), 1, threads)
    except Exception as ex:
        print("cpu_baseline: baseline/_ref failed (%r)" % (ex,), file=sys.stderr)
    port = port_leg(5.0 if ref is not None else budget_s, threads)
    port["cpu_model"] = cpu_model()
    port["config1"] = config1_port_leg()
    return dict(ref, port=port) if ref is not None else port


def own_bytes_per_sim(d, n_vis=3.2):
    """Bytes one simulation of THIS kernel has to move (DESIGN.md section 5): per interior select the node block's
    16 B summary and n_vis 32 B child slots (key, logit, N, W, q -- one round trip, no gather of the children's own
    arrays); the new node's logits + child rows and summary written; the parent's logits + child rows read once for
    its refreshed summary, one slot key + the summary written; the backup's stores of (N, W) to each path node's
    own arrays and of (N, W, q) to its slot in the parent's block (no loads: the statistics come down with the
    descent); the root's and root child's (N, W) read after the descent."""
    return (d - 1) * (16 + 32 * n_vis) + (4 * A + 2 * A + 16) + (4 * A + 2 * A + 16 + 8 + 16) + 32 * (d + 1) + 24


def net_leg(eng, dev, peaks, dtype_name="bf16"):
    """Same workload with the REAL network as evaluator (E1): GomokuNetEZ 8 blocks x 128 filters,
    random init (torch.manual_seed(0)), BatchNorm folded, cuDNN fused conv ops, CUDA graph;
    one full 400-simulation search for all G games through the stepwise kernels.  dtype_name "bf16", or
    "tf32" = fp32 tensors with TF32 convolutions -- the precision the reference's own server runs at on this
    GPU (workers.py:318, 350-352: fp32 model, PyTorch's default cudnn.allow_tf32)."""
    import torch
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.network import GomokuNetEZ, NetworkSearch
    torch.manual_seed(0)
    cfg = Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=A, NUM_RES_BLOCKS=8, NUM_FILTERS=128, HEAD_HIDDEN_DIM=64)
    torch.backends.cudnn.allow_tf32 = True
    ns = NetworkSearch(eng, GomokuNetEZ(cfg), dtype=torch.bfloat16 if dtype_name == "bf16" else torch.float32, graph=True)
    G = eng.G
    gum = torch.empty((G, A), dtype=torch.float64, device=dev)
    eng.fill_gumbel(gum, 4242, 0)
    eng.set_roots(*staggered_positions(G, 0))
    ns.search(gum, num_simulations=8)           # warm-up (partial search): cuDNN plans + graph capture
    # the tree kernels of one simulation step on their own (select -> expand/backup with the last network outputs)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(20):
        eng.select(out=ns.obs); eng.expand_backup(ns.ev.logits, ns.ev.values)
    t1.record(); torch.cuda.synchronize()
    tree_ms = t0.elapsed_time(t1) / 20
    eng.set_roots(*staggered_positions(G, 0))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clk = ClockSampler(dev.index or 0); clk.start()
    e0.record(); ns.search(gum); eng.finalize(want_visits=False); e1.record(); torch.cuda.synchronize()
    clk.stop_flag = True; clk.join(timeout=2)
    ms = e0.elapsed_time(e1)
    n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0.record()
    for _ in range(10):
        ns.ev._forward()
    n1.record(); torch.cuda.synchronize()
    net_ms = n0.elapsed_time(n1) / 10
    tf = 1.064e9 * G / (net_ms * 1e-3) / 1e12
    peak_tf = float(peaks.get("bf16_tflops", 1590.0))
    peak_sus = float(peaks.get("bf16_tflops_sustained", peak_tf))
    selfplay = None
    if dtype_name == "bf16":
        # production self-play with the network (universal_worker + inference server, workers.py:129-241, 314-373):
        # lock-step moves of all G games -- search, decision, trajectory record, do_move, end check, restart --
        # finished games packed on the device into the replay ring + PER tree
        from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
        from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
        from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
        sp = SelfPlayEngine(eng, ns, noise_seed=4244)
        traj = TrajectoryStore(eng)
        buf = DeviceReplayBuffer(1 << 16, N, device=dev)
        n_moves = 2
        eng.selfplay_e0(G * 40, E0_SEED, LOGIT_DIV, 4244, traj, True)      # untimed: ~40 E0-driven moves per game, so the timed
        torch.cuda.synchronize()                                           # moves start from mid-game boards, not 4096 empty ones
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(); sp.play(moves_per_game=n_moves, traj=traj, sink=buf.add_packed, chunk=n_moves); s1.record(); torch.cuda.synchronize()
        sp_ms = s0.elapsed_time(s1)
        selfplay = {"moves_per_sec": G * n_moves / (sp_ms * 1e-3), "sims_per_sec": G * n_moves * S / (sp_ms * 1e-3),
                    "moves": G * n_moves, "api": "SelfPlayEngine(engine, NetworkSearch).play(traj=, sink=DeviceReplayBuffer.add_packed)",
                    "what": "%d lock-step moves of %d games (each ~40 moves into its game): search (%d graph replays), decision, "
                            "trajectory record, do_move, end check, pack of finished games into the replay ring" % (n_moves, G, S - 1)}
        del traj, buf
    return {"evaluator": "GomokuNetEZ 8x128 %s (random init, BN folded, cuDNN fused conv+bias+relu); one CUDA graph per simulation "
                         "step {select -> network -> expand/backup}" % dtype_name,
            "accum_dtype": eng.accum_dtype,
            "sims_per_sec": G * S / (ms * 1e-3), "moves_per_sec": G / (ms * 1e-3), "ms_per_search": ms,
            "clocks": clk.summary(),      # tensor-bound legs run into the board's power cap: the SM clock during the search says how far
            "net_forward_ms": net_ms, "tree_kernels_ms_per_sim_step": tree_ms,
            "step_minus_standalone_forward_ms": ms / S - net_ms,
            **({"selfplay": selfplay} if selfplay else {}),
            "tensor": {"bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf,
                       "peak_sustained": peak_sus, "frac_sustained": tf / peak_sus,
                       "flop_per_eval": 1.064e9, "note": "algorithmic conv FLOPs (SURVEY 8d) / measured cuBLAS bf16 peak: `peak` = burst (a "
                                                         "kernel timed alone), `peak_sustained` = back-to-back GEMMs for 4 s -- the search is "
                                                         "400 forwards back to back, so the sustained figure is the one it runs against "
                                                         "(also for the tf32 leg: there is no measured tf32 peak)"}}


def muzero_leg(dev, peaks, G):
    """BASELINE configs[2]: MuZero mode, 15x15, 400 simulations (= 100 distinct recurrent evaluations per
    search, SURVEY App. A.6), G games, GomokuNetEZ 8x128 bf16 dynamics network in the tree.  Hidden states
    live in a device pool (one NHWC row per tree node); a simulation step is select -> hidden gather (+ action
    plane) -> recurrent inference -> hidden scatter -> expand/backup, replayed as one CUDA graph."""
    import torch
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.muzero import FoldedRecurrentInference, MuZeroDeviceSearch, evals_per_search
    from datou_gomoku_muzero_b200.network import FoldedInitialInference, GomokuNetEZ
    torch.manual_seed(0)
    torch.backends.cudnn.benchmark = os.environ.get("GMZ_CUDNN_BENCHMARK", "1") != "0"
    cfg = Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=A, NUM_RES_BLOCKS=8, NUM_FILTERS=128, HEAD_HIDDEN_DIM=64)
    net = GomokuNetEZ(cfg).to(dev).eval()
    fi, fr = FoldedInitialInference(net, torch.bfloat16), FoldedRecurrentInference(net, torch.bfloat16)

    def initial(obs):
        p, v, h = fi(obs.to(torch.bfloat16).contiguous(memory_format=torch.channels_last))
        return p.float().contiguous(), v.reshape(-1).float(), h

    eng = SearchEngine(G, board_size=N, n_in_row=N_IN_ROW, num_simulations=S, num_top_actions=K_TOP, mode="MuZero", device=dev)
    eng.set_roots(*staggered_positions(G, 0))
    evals = evals_per_search(S, K_TOP, K_TOP)
    mz = MuZeroDeviceSearch(eng, initial, fr, nodes_per_game=evals + 2, graph=True)
    gum = torch.empty((G, A), dtype=torch.float64, device=dev)
    eng.fill_gumbel(gum, 4243, 0)
    mz.search(gum, max_steps=evals); eng.finalize(want_visits=False)          # warm-up: cuDNN plans + graph capture
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clk = ClockSampler(dev.index or 0); clk.start()
    e0.record(); steps = mz.search(gum, max_steps=evals); eng.finalize(want_visits=False); e1.record()
    torch.cuda.synchronize()
    clk.stop_flag = True; clk.join(timeout=2)
    ms = e0.elapsed_time(e1)
    # the pool kernels on their own: bytes moved per launch / time, against the measured HBM peak
    parent, action, child, _ = eng._mz_out[:4]
    parent.copy_(mz._root_slot); action.fill_(7); child.copy_(mz._root_slot + 1)
    hrows = mz.pool[:G].clone()
    g0, g1, s1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    for _ in range(3):
        mz._gather(parent, action); mz._scatter(child, hrows)
    g0.record()
    for _ in range(20):
        mz._gather(parent, action)
    g1.record()
    for _ in range(20):
        mz._scatter(child, hrows)
    s1.record(); torch.cuda.synchronize()
    gather_ms, scatter_ms = g0.elapsed_time(g1) / 20, g1.elapsed_time(s1) / 20
    gather_bytes = G * (2 * mz.row_bytes + mz.positions * mz.embed_bytes)
    scatter_bytes = G * 2 * mz.row_bytes
    peak = float(peaks.get("hbm_gbs", 6650.0))
    tf = (1.141e9 * steps + 1.064e9) * G / (ms * 1e-3) / 1e12
    peak_tf = float(peaks.get("bf16_tflops", 1590.0))
    peak_sus = float(peaks.get("bf16_tflops_sustained", peak_tf))
    # the same MuZero-mode search with the fixed evaluator, fused in the persistent kernel (E0's recurrent half on the
    # parent's hidden hash): the counterpart of the reference's MuZero tree-only run (`--impl reference`: muzero_tree_only)
    eng.set_roots(*staggered_positions(G, 0))
    eng.search_e0(gum, E0_SEED, LOGIT_DIV)
    z0, z1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    z0.record()
    for _ in range(3):
        eng.search_e0(gum, E0_SEED, LOGIT_DIV)
    z1.record(); torch.cuda.synchronize()
    e0_ms = z0.elapsed_time(z1) / 3
    return {"workload": "MuZero-mode 15x15, 400 sims/move, %d games, GomokuNetEZ 8x128 bf16 dynamics in the tree "
                        "(BASELINE configs[2])" % G,
            "sims_per_sec": G * S / (ms * 1e-3), "moves_per_sec": G / (ms * 1e-3), "ms_per_search": ms,
            "recurrent_evals_per_search": steps, "distinct_evals_per_sec": G * (steps + 1) / (ms * 1e-3),
            "clocks": clk.summary(),      # (this leg has measured 435 ms at 1965 MHz and 615-630 ms under sw_power_cap at ~1350 MHz)
            "hidden_pool_gb": mz.pool.numel() * mz.pool.element_size() / 1e9,
            "e0_fused": {"sims_per_sec": G * S / (e0_ms * 1e-3), "ms_per_search": e0_ms,
                         "what": "same searches with the fixed evaluator E0 inside the persistent kernel (k_play_e0<NC, MZ>)"},
            "tensor": {"bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf,
                       "peak_sustained": peak_sus, "frac_sustained": tf / peak_sus},
            "hidden_gather": {"bound": "hbm", "ms": gather_ms, "achieved": gather_bytes / gather_ms / 1e6, "peak": peak,
                              "unit": "GB/s", "frac": gather_bytes / gather_ms / 1e6 / peak, "bytes": gather_bytes},
            "hidden_scatter": {"bound": "hbm", "ms": scatter_ms, "achieved": scatter_bytes / scatter_ms / 1e6, "peak": peak,
                               "unit": "GB/s", "frac": scatter_bytes / scatter_ms / 1e6 / peak, "bytes": scatter_bytes}}


def per_leg(dev, peaks, rounds=400):
    """BASELINE configs[4], first half: PER `sample(360)` + `update_priorities(360)` on a full capacity-1M sum tree
    resident on the device (replay_buffer.py:57-103), CUDA-event timed; the reference's own InMemoryReplayBuffer on
    one host core beside it.  Algorithmic bytes (SURVEY 8d): 168 B per sample, 320 B per update."""
    import ctypes as C
    import torch
    from datou_gomoku_muzero_b200 import replay_buffer as rb
    cap, B = 1_000_000, 360
    rs = np.random.RandomState(0)
    tree = rb.SumTree(cap, device=dev)
    torch.cuda.synchronize()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record(); tree.add_many(np.abs(rs.randn(cap)) + 1e-6); f1.record(); torch.cuda.synchronize()
    u = torch.from_numpy(rs.random_sample((rounds, B))).to(dev)
    newp = torch.from_numpy(np.abs(rs.randn(rounds, B)) + 1e-6).to(dev)
    idx = torch.empty(B, dtype=torch.int64, device=dev); pr = torch.empty(B, dtype=torch.float64, device=dev)
    w = torch.empty(B, dtype=torch.float32, device=dev)
    lib, st, P = tree.lib, tree._stream(), (lambda t: C.c_void_p(t.data_ptr()))

    def step(i):
        lib.gmz_per_sample(P(tree.tree), cap, cap, P(u[i]), B, 0.4, P(idx), P(pr), P(w), st)
        lib.gmz_per_update(P(tree.tree), cap, P(idx), P(newp[i]), B, st)
    for i in range(10):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(10, rounds):
        step(i)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (rounds - 10)
    peak = float(peaks.get("hbm_gbs", 6650.0))
    nbytes = B * (168 + 320)
    out = {"workload": "PER sample(360) + update_priorities(360), capacity 1M, full tree (BASELINE configs[4])",
           "us_per_batch": ms * 1e3, "samples_per_sec": B / (ms * 1e-3), "fill_1M_adds_ms": f0.elapsed_time(f1),
           "roofline": {"bound": "hbm", "kernel": "k_per_sample + k_per_update", "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": peak,
                        "unit": "GB/s", "frac": nbytes / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_batch": nbytes,
                        "note": "360 dependent 20-level descents per launch: latency bound by construction, not bandwidth bound"}}
    try:
        from baseline import ref_runner
        if ref_runner.available():
            r = ref_runner.per(cap, B, rounds=60)
            out["cpu_reference"] = {"kind": "reference", "cores": 1, "us_per_batch": r["us_per_batch"], "samples_per_sec": r["samples_per_sec"],
                                    "sample": "60 x (sample(360) + update_priorities) of the reference InMemoryReplayBuffer, capacity 1M"}
    except Exception as ex:
        out["cpu_reference"] = {"error": repr(ex)[:200]}
    return out


def reanalysis_leg(dev, positions=1_000_000, depth=4):
    """BASELINE configs[4], second half: Surge re-analysis (workers.py:243-305) of `positions` stored positions with
    the latest evaluator, through the public re-analysis driver: host boards -> pinned staging -> H2D -> search ->
    D2H policies / values, `depth` batches of G in flight."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.reanalysis import reanalyse_positions
    G = 4096
    engs = [SearchEngine(G, board_size=N, n_in_row=N_IN_ROW, num_simulations=S, num_top_actions=K_TOP, device=dev) for _ in range(depth)]
    base = staggered_positions(16 * G, 3)          # 65 536 distinct stored positions, cycled to `positions`
    reps = (positions + 16 * G - 1) // (16 * G)
    boards = np.tile(base[0], (reps, 1))[:positions]; players = np.tile(base[1], reps)[:positions]
    last = np.tile(base[2], reps)[:positions]; mc = np.tile(base[3], reps)[:positions]
    reanalyse_positions(engs, boards[:depth * G], players[:depth * G], last[:depth * G], mc[:depth * G], eval_seed=E0_SEED + 1,
                        logit_div=LOGIT_DIV, noise_seed=77)          # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pol, val = reanalyse_positions(engs, boards, players, last, mc, eval_seed=E0_SEED + 1, logit_div=LOGIT_DIV, noise_seed=78,
                                   want_policies="checksum")
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    del engs
    return {"workload": "Surge re-analysis of %d stored positions, 15x15 / 400 sims, E0 (BASELINE configs[4])" % positions,
            "positions": positions, "seconds": dt, "positions_per_sec": positions / dt, "sims_per_sec": positions * S / dt,
            "h2d_bytes": int(boards.nbytes + players.nbytes + last.nbytes + mc.nbytes), "d2h_bytes": int(positions * (A * 8 + 8)),
            "pipeline_depth": depth, "api": "reanalysis.reanalyse_positions(engines, host boards/players/last_moves/move_counts)",
            "value_mean": float(np.mean(val)), "policy_checksum": float(pol)}


def selfplay_e2e_leg(dev, rank, world, G, steps):
    """Self-play END TO END on the device: play -> finished games packed into move records (observations, policies,
    boards, rewards, n-step targets) -> appended to the device replay ring + PER tree -> one training batch of 360
    slices sampled per chunk (workers.py:162-230 + 399-433 with no host object in between).  Wall-clock moves/s
    including every kernel and the one small D2H read (the finished-game table) per chunk.  At N > 1 it is followed by
    the trajectory gather: every rank's last packed chunk -> rank 0 with NCCL (replaces data_queue)."""
    import torch
    import torch.distributed as dist
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.parallel import gather_packed_games
    from datou_gomoku_muzero_b200.replay_buffer import DeviceReplayBuffer
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng = SearchEngine(G, board_size=N, n_in_row=N_IN_ROW, num_simulations=S, num_top_actions=K_TOP, device=dev)
    sp = SelfPlayEngine(eng, "e0", seed=E0_SEED, logit_div=LOGIT_DIV, noise_seed=2000 + rank)
    eng.set_roots(*staggered_positions(G, rank))
    traj = TrajectoryStore(eng, extra_slots=G // 2)
    buf = DeviceReplayBuffer(400_000, N, device=dev)             # 1.9 GB of records
    state = {"packed": None, "batches": 0, "d2h": 0, "records": 0}

    def sink(pg):
        buf.add_packed(pg)
        state["packed"], state["records"] = pg, state["records"] + pg.n_moves
        state["d2h"] += pg.table.nbytes + 4
        if len(buf) >= 360:
            batch, idx, w = buf.sample(360, rot_k=state["batches"] % 4, flip=bool(state["batches"] & 1))
            buf.update_priorities(idx, batch[4][:, 0] - 0.5)     # stand-in TD errors (device)
            state["batches"] += 1
    sp.play(moves_per_game=steps, traj=traj, sink=sink)          # warm-up of the timed length: the caching allocator then holds
                                                                 # blocks of the sizes the timed chunk packs into (steady state)
    m0, f0 = eng.play_counters()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sp.play(moves_per_game=steps, traj=traj, sink=sink)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    m1, f1 = eng.play_counters()
    out = {"what": "play (persistent kernel) -> gmz_traj_pack -> DeviceReplayBuffer.add_packed -> sample(360) + update_priorities "
                   "per chunk, all on the device", "moves": m1 - m0, "seconds": dt, "moves_per_sec": (m1 - m0) / dt,
           "sims_per_sec": (m1 - m0) * S / dt, "games_finished": f1 - f0, "records_packed": state["records"],
           "record_bytes": int(buf.stride), "batches_sampled": state["batches"], "d2h_bytes_total": int(state["d2h"]),
           "h2d_bytes_total": 0, "replay_len": len(buf)}
    pg = state["packed"]
    if pg is not None:                                           # the host-facing form of the same bytes
        t0 = time.perf_counter()
        items = pg.data_queue_items(0)
        dt2 = time.perf_counter() - t0
        out["host_objects"] = {"what": "last chunk: D2H of the records + GameRecord / TrainingSlice views (workers.py:230 tuples)",
                               "games": len(items), "moves": pg.n_moves, "seconds": dt2, "moves_per_sec": pg.n_moves / dt2,
                               "d2h_bytes": int(pg.n_moves * buf.stride)}
    if world > 1:
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gather_packed_games(pg, N, dst=0, device=dev)            # warm-up (NCCL channels)
        torch.cuda.synchronize(); dist.barrier()
        e0.record(); got = gather_packed_games(pg, N, dst=0, device=dev); e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            nbytes = got.n_moves * buf.stride if got is not None else 0
            out["trajectory_gather"] = {"what": "every rank's last packed chunk -> rank 0: all_gather(counts) + gather(records) + "
                                                "gather(game tables), NCCL", "games": 0 if got is None else len(got),
                                        "moves": 0 if got is None else got.n_moves, "bytes": int(nbytes), "ms": float(t.item()),
                                        "gb_per_s": nbytes / (float(t.item()) * 1e-3) / 1e9 if nbytes else 0.0}
    return out


def weight_broadcast_leg(dev, rank, world):
    """BASELINE configs[3]: the trainer rank publishes GomokuNetEZ's weights to every self-play rank
    (`model_update_queue` in the reference, workers.py:587-593) as one NCCL broadcast of a flat buffer."""
    import torch
    import torch.distributed as dist
    from datou_gomoku_muzero_b200.config import Config
    from datou_gomoku_muzero_b200.network import GomokuNetEZ
    from datou_gomoku_muzero_b200.parallel import FlatWeights
    torch.manual_seed(100 + rank)                       # every rank starts from DIFFERENT weights
    cfg = Config(BOARD_SIZE=N, ACTION_SPACE_SIZE=A, NUM_RES_BLOCKS=8, NUM_FILTERS=128, HEAD_HIDDEN_DIM=64)
    net = GomokuNetEZ(cfg).to(dev)
    fw = FlatWeights(net)                               # parameters become views into one flat buffer per dtype
    nbytes = fw.nbytes
    for _ in range(2):
        fw.broadcast(src=0)
    torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        fw.broadcast(src=0)
    e1.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 5], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    chk = torch.stack([p.detach().double().sum() for p in net.parameters()]).sum().reshape(1)
    lo, hi = chk.clone(), chk.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    return {"what": "GomokuNetEZ 8x128 parameters + buffers living in one flat buffer per dtype (parallel.FlatWeights), "
                    "in-place NCCL broadcast from rank 0",
            "bytes": int(nbytes), "ms": float(t.item()), "gb_per_s": nbytes / (float(t.item()) * 1e-3) / 1e9,
            "ranks_identical_after": bool(lo.item() == hi.item())}


DUMP_MAX_GAMES = 4096          # 4096 games x (policy f64 + board f32) = 11 MB: a dump stays small at any --games


def dump_last_step(out_dir, G, dev, n_steps):
    """--dump-outputs: what the timed path computes for rank 0's games in step `n_steps` (= warmup + timed steps), the
    arrays its caller reads from the TrajectoryStore and the engine: policy f64 [g, A], root value f64 [g], action [g],
    board after the move f32 [g, A], winner [g] (+-1, 0 draw, 2 game goes on), game index [g] -- all G games, or a
    fixed seeded sample of DUMP_MAX_GAMES.  The persistent kernel hands the timed moves to the games by a ticket
    counter, so how many of them each game gets, and so which of its moves falls in the last step, depends on timing.
    To give the same outputs for the same arguments, the dump replays the games on a fresh engine (same roots, seeds
    and kernel) in one-move launches, in which every game makes exactly one move, and records the last one."""
    import torch
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine
    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    eng = SearchEngine(G, board_size=N, n_in_row=N_IN_ROW, num_simulations=S, num_top_actions=K_TOP, device=dev)
    sp = SelfPlayEngine(eng, "e0", seed=E0_SEED, logit_div=LOGIT_DIV, noise_seed=1000)
    eng.set_roots(*staggered_positions(G, 0))
    for _ in range(n_steps - 1):
        sp.play(moves_per_game=1)
    # a fresh store puts game g's next move in slot g; with no spare slot a game that ends there stays on its final board
    last = TrajectoryStore(eng, extra_slots=0, max_moves=1)
    sp.play(moves_per_game=1, traj=last)
    fin = last.fin_queue[:int(last.fin_count.item())].long()
    winner = torch.full((G,), 2, dtype=torch.int32, device=dev)
    winner[fin[:, 1]] = fin[:, 3].int()
    games = np.arange(G) if G <= DUMP_MAX_GAMES else np.sort(np.random.RandomState(0).choice(G, DUMP_MAX_GAMES, replace=False))
    sel = torch.as_tensor(games, device=dev)
    out = {"policy": last.policy[sel, 0], "value": last.value[sel, 0], "action": last.action[sel, 0].double(),
           "board": eng.get_roots()[0].reshape(G, A)[sel].float(), "winner": winner[sel].double(),
           "game": torch.as_tensor(games, dtype=torch.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.selfplay import SelfPlayEngine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator is created: send it to stderr,
        # stdout carries the one JSON line only
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    G = args.games

    eng = SearchEngine(G, board_size=N, n_in_row=N_IN_ROW, num_simulations=S, num_top_actions=K_TOP, device=dev)
    sp = SelfPlayEngine(eng, "e0", seed=E0_SEED, logit_div=LOGIT_DIV, noise_seed=1000 + rank)
    eng.set_roots(*staggered_positions(G, rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- mean leaf depth of this workload (one untimed traced search) for the algorithmic bytes
    sp.e.fill_gumbel(sp.gumbel, 999, 0)
    _, td = eng.search_e0(sp.gumbel, E0_SEED, LOGIT_DIV, trace=True)
    mean_depth = float(td[:, : S - 1].float().mean().item())
    del td

    from datou_gomoku_muzero_b200.trajectory import TrajectoryStore
    traj = TrajectoryStore(eng, extra_slots=max(64, G // 2))
    for _ in range(args.warmup):
        sp.play(moves_per_game=1, traj=traj)          # warm-up steps: G moves each
    traj.harvest(copy_policies=False)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    # ---- timed region: K steps = K*G self-play moves (noise, 400-sim search, decision, trajectory
    # record, do_move, win/draw check, restart), ONE persistent launch, games advance independently
    launches0 = eng.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m0, f0 = eng.play_counters()
    barrier()
    ev0.record()
    # trajectory slots are recycled by the host between launches and a game ends about every 85 moves, so a
    # long run is cut into launches of <= 48 steps with a (policy-free) harvest in between -- inside the timing
    remaining = args.steps
    while remaining > 0:
        n = min(48, remaining)
        sp.play(moves_per_game=n, traj=traj)
        remaining -= n
        if remaining > 0:
            traj.harvest(copy_policies=False)
    ev1.record()
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    launches = eng.launches - launches0
    m1, f1 = eng.play_counters()
    moves_done, finished = m1 - m0, f1 - f0
    kernel_ms = elapsed_ms / args.steps               # the play kernel IS the timed region
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    per_rank_ms = [elapsed_ms / args.steps]
    if world > 1:
        allms = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allms, t)
        per_rank_ms = [float(x.item()) / args.steps for x in allms]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    md = torch.tensor([moves_done], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(md, op=dist.ReduceOp.SUM)
    moves_total = float(md.item())
    harvested = len(traj.harvest(copy_policies=False))

    # ---- e2e: the public batch API with HOST buffers (pinned staging, H2D of roots + noise, search,
    # decision, D2H of policy/value/action every step), double-buffered over two engines so the heavy
    # tail of one batch overlaps the next batch (PipelinedBatchSearch)
    from datou_gomoku_muzero_b200.mcts import PipelinedBatchSearch
    engs = [eng] + [SearchEngine(G, board_size=N, n_in_row=N_IN_ROW, num_simulations=S, num_top_actions=K_TOP, device=dev)
                    for _ in range(args.e2e_depth - 1)]
    pipe = PipelinedBatchSearch(engs, evaluator="e0", eval_seed=E0_SEED, logit_div=LOGIT_DIV)
    hb, hp, hl, hm = staggered_positions(G, rank)
    hgums = [np.random.RandomState(5 + rank + 17 * i).gumbel(0, 1, (G, A)) for i in range(3)]
    for i in range(args.e2e_depth):
        pipe.result(pipe.submit(hb, hp, hl, hm, hgums[i % 3]))
    barrier()
    e2e_steps = max(2 * args.e2e_depth, args.steps)      # as many host batches as timed kernel steps: the pipeline drain amortises
    t0 = time.perf_counter()
    inflight = []
    for i in range(e2e_steps):
        inflight.append(pipe.submit(hb, hp, hl, hm, hgums[i % 3]))
        if len(inflight) >= args.e2e_depth:
            pol, val, act = pipe.result(inflight.pop(0))
    while inflight:
        pol, val, act = pipe.result(inflight.pop(0))
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    sampler.stop_flag = True
    sampler.join(timeout=2)

    bcast = weight_broadcast_leg(dev, rank, world) if world > 1 else None
    sp_e2e = None
    if not args.no_selfplay_e2e:
        del pipe, engs
        import gc
        gc.collect(); torch.cuda.empty_cache()
        try:
            sp_e2e = selfplay_e2e_leg(dev, rank, world, G, max(args.steps, 24))
        except Exception as ex:
            sp_e2e = {"error": repr(ex)[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    sims_per_step = G * S * world
    value = moves_total * S / (elapsed_ms * 1e-3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    bytes_per_launch = algorithmic_bytes_per_sim(mean_depth) * (moves_done / args.steps) * (S - 1)   # per step
    achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
    traffic, traffic_note = None, "no ncu measurement on record"
    try:        # ncu dram__bytes_read.sum + dram__bytes_write.sum per bench step, valid only for the kernel it was taken on
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tj.get("kernel_source_sha") == kernel_source_sha():
            traffic, traffic_note = tj.get("k_play_e0_bytes_per_step"), "ncu, " + str(tj.get("source", ""))
        else:
            traffic_note = "stale: measured on kernel sources %s, current %s" % (tj.get("kernel_source_sha"), kernel_source_sha())
    except Exception:
        pass
    out = {
        "metric": "mcts_sims_per_sec", "value": value, "unit": "sims/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "moves_per_sec": moves_total / (elapsed_ms * 1e-3),
        "config": bench_config(G),
        "notes": "a step = G self-play moves (noise, 400-sim search, decision, trajectory record, do_move, win/draw check, in-kernel "
                 "restart of finished games); the K timed steps run as one persistent ticketed launch of K*G moves (one launch "
                 "per 48 steps on longer runs); float64 tree arithmetic (E0 hands Python floats)",
        "ms_per_step_per_rank": per_rank_ms,
        "e2e": {"value": sims_per_step * e2e_steps / e2e_s, "unit": "sims/s",
                "h2d_bytes_per_step": int(hb.nbytes + hp.nbytes + hl.nbytes + hm.nbytes + hgums[0].nbytes),
                "d2h_bytes_per_step": int(pol.nbytes + val.nbytes + act.nbytes), "steps": e2e_steps,
                "api": "PipelinedBatchSearch.submit/result(host boards, players, last_moves, move_counts, gumbel)",
                "pipeline_depth": args.e2e_depth},
        "gpu_launches": launches,
        "games_finished_in_timed_region": int(finished), "games_harvested": harvested,
        "roofline": {"bound": "hbm", "kernel": "k_play_e0<2>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note, "kernel_ms_per_step": kernel_ms,
                     "mean_leaf_depth": mean_depth,
                     "algorithmic_bytes_per_sim": algorithmic_bytes_per_sim(mean_depth),
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                     "own_bytes_per_sim": own_bytes_per_sim(mean_depth),
                     "own_frac": own_bytes_per_sim(mean_depth) * (moves_done / args.steps) * (S - 1) / (kernel_ms * 1e-3) / 1e9 / peak,
                     "note": "achieved/frac use SURVEY 8d's bytes per simulation, i.e. the reference algorithm's dense row reads; the "
                             "certified select does not make those reads (own_bytes_per_sim = what this kernel must move, own_frac = "
                             "its share of the HBM peak; measured DRAM traffic in `traffic`): the kernel is latency/issue bound"},
        "clocks": sampler.summary(),
    }
    if bcast is not None:
        out["weight_broadcast"] = bcast
    if sp_e2e is not None:
        out["selfplay_e2e"] = sp_e2e
    if not args.no_net and world == 1:          # single-GPU context measurement
        try:
            torch.cuda.empty_cache()
            neng = SearchEngine(G, board_size=N, n_in_row=N_IN_ROW, num_simulations=S, num_top_actions=K_TOP, device=dev,
                                accum_dtype="float32")       # float32 accumulation: what the reference does with network values
            out["net"] = net_leg(neng, dev, peaks, "bf16")
            out["net_tf32"] = net_leg(neng, dev, peaks, "tf32")
            del neng
        except Exception as ex:      # the headline (fixed evaluator) stands on its own
            out["net"] = {"error": repr(ex)[:200]}
    if not args.no_net and world == 1:
        try:
            import gc
            gc.collect()
            torch.cuda.empty_cache()      # cuDNN autotuning sizes its workspace by what the caching allocator has released
            out["muzero"] = muzero_leg(dev, peaks, G)
        except Exception as ex:
            out["muzero"] = {"error": repr(ex)[:200]}
    if not args.no_config5 and world == 1:
        try:
            import gc
            gc.collect(); torch.cuda.empty_cache()
            out["per"] = per_leg(dev, peaks)
        except Exception as ex:
            out["per"] = {"error": repr(ex)[:200]}
        try:
            out["reanalysis"] = reanalysis_leg(dev, args.reanalysis_positions)
        except Exception as ex:
            out["reanalysis"] = {"error": repr(ex)[:200]}
    if not args.no_cpu_baseline and world == 1:  # reported on rank 0 at N=1 only
        out["cpu_baseline"] = cpu_baseline_leg(args.cpu_seconds)
    if args.dump_outputs:
        dump_last_step(args.dump_outputs, G, dev, args.warmup + args.steps)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--games", type=int, default=4096, help="concurrent games per GPU")
    ap.add_argument("--cpu-games", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-net", action="store_true", help="skip the real-network (E1) leg")
    ap.add_argument("--e2e-depth", type=int, default=6, help="host batches in flight in the end-to-end leg")
    ap.add_argument("--no-selfplay-e2e", action="store_true", help="skip the device-side self-play -> replay -> batch leg")
    ap.add_argument("--no-config5", action="store_true", help="skip the PER and re-analysis legs (BASELINE configs[4])")
    ap.add_argument("--reanalysis-positions", type=int, default=1_000_000)
    ap.add_argument("--ref-topology-seconds", type=float, default=60.0,
                    help="--impl reference at N = 1: seconds of the reference's universal_worker + inference_server topology (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="--impl ours: write the last step's outputs to DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU arm computes (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
