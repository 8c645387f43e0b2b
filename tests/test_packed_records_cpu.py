"""Host side of the packed-move-record hand-off (no GPU): numpy views of the record bytes reproduce the
GameRecord / TrainingSlices the reference's own universal_worker produced, and two ranks gather their records with
tensor collectives (gloo here, NCCL on the GPUs)."""
import os
import socket
import sys

import numpy as np
import pytest

from _golden_util import GOLDEN_DIR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["selfplay_az_9_100", "selfplay_az_6_36", "selfplay_mz_6_50", "selfplay_az_9_64_dense_f32", "selfplay_mz_6_50_dense_f32"]


def packed_from_golden(z, game_seq=0, game=0, slot=0):
    """What gmz_traj_pack writes for one finished game, built from the golden arrays (the GPU test compares the
    kernel's bytes with the same arrays)."""
    from datou_gomoku_muzero_b200.trajectory import record_dtype
    N = int(z["params"][0])
    T = len(z["actions"])
    r = np.zeros(T, record_dtype(N))
    r["game_seq"], r["t"], r["length"], r["winner"] = game_seq, np.arange(T), T, int(z["winner"])
    r["action"] = z["actions"]
    r["to_move"] = np.where(np.arange(T) % 2 == 0, 1, -1)
    r["last_move"] = np.concatenate([[-1], z["actions"][:-1]])
    r["move_count"] = np.arange(T)
    r["reward"] = z["rewards"].astype(np.float32)
    r["value_target"] = z["values_targets"].astype(np.float32)
    r["search_value"] = z["search_values"]
    r["game"], r["slot"] = game, slot
    r["policy"], r["obs"], r["board"] = z["policies"], z["observations"], z["boards"]
    return r


@pytest.mark.parametrize("name", NAMES)
def test_record_views_match_reference_game_record_and_slices(name):
    from datou_gomoku_muzero_b200.config import config
    from datou_gomoku_muzero_b200.trajectory import PackedGames
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    N, U, n_steps = int(z["params"][0]), int(z["params"][5]), int(z["params"][6])
    r = packed_from_golden(z)
    T = len(r)
    pg = PackedGames(r.view(np.uint8).reshape(T, -1), np.array([[0, 0, T, int(z["winner"])]], np.int32), [0, T], N)
    saved = config.NUM_UNROLL_STEPS
    config.NUM_UNROLL_STEPS = U
    try:
        gr = pg.game_record(0)
        assert np.array_equal(np.stack(gr.observations), z["observations"]) and np.array_equal(np.stack(gr.board_states), z["boards"])
        assert gr.actions == [int(a) for a in z["actions"]] and all(isinstance(a, int) for a in gr.actions)
        assert np.array_equal(np.array(gr.rewards), z["rewards"]) and all(isinstance(x, float) for x in gr.rewards)
        assert np.array_equal(np.array(gr.values, np.float64), z["values_targets"])
        assert np.array_equal(np.stack(gr.policies), z["policies"]) and gr.policies[0].dtype == np.float64
        sl = pg.training_slices(0)
        assert len(sl) == int(z["n_slices"])
        for field, key in (("observation", "slice_obs"), ("action_history", "slice_act"), ("reward_history", "slice_rew"),
                           ("policy_history", "slice_pi"), ("value_history", "slice_val")):
            got = np.stack([getattr(s, field) for s in sl])
            assert got.dtype == z[key].dtype and np.array_equal(got, z[key]), field
        items = pg.data_queue_items(model_version=7)
        assert len(items) == 1 and items[0][2] == 7 and len(items[0][1]) == T
    finally:
        config.NUM_UNROLL_STEPS = saved


def test_record_layout_matches_the_header():
    """record_dtype mirrors include/gmz.h gmz_move_record + payload; the stride is what the library reports."""
    from datou_gomoku_muzero_b200 import _lib
    from datou_gomoku_muzero_b200.trajectory import record_dtype
    lib = _lib.load()
    for N in (6, 9, 15, 19):
        dt = record_dtype(N)
        assert dt.itemsize == lib.gmz_move_record_bytes(N) and dt.itemsize % 16 == 0
        assert dt.fields["policy"][1] == 64 and dt.fields["search_value"][1] == 40 and dt.fields["board"][1] == 64 + 20 * N * N
    assert lib.gmz_move_record_bytes(0) == 0 and lib.gmz_move_record_bytes(20) == 0


def test_header_dtype_matches_the_c_struct(tmp_path):
    """trajectory.RECORD_HEADER has every gmz_move_record field at the C compiler's offset and size, and nothing else."""
    import subprocess
    from datou_gomoku_muzero_b200.trajectory import RECORD_HEADER
    src = tmp_path / "header_layout.c"
    src.write_text("#include <stddef.h>\n#include <stdio.h>\n#include \"gmz.h\"\nint main(void)\n{\n"
                   "    printf(\"sizeof %zu\\n\", sizeof(gmz_move_record));\n"
                   + "".join(f"    printf(\"{f} %zu %zu\\n\", offsetof(gmz_move_record, {f}), sizeof(((gmz_move_record *)0)->{f}));\n"
                             for f in RECORD_HEADER.names)
                   + "    return 0;\n}\n")
    exe = tmp_path / "header_layout"
    subprocess.check_call(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    lines = [ln.split() for ln in subprocess.check_output([str(exe)], text=True).splitlines()]
    assert lines[0] == ["sizeof", str(RECORD_HEADER.itemsize)]
    got = {f: (int(off), int(size)) for f, off, size in lines[1:]}
    want = {f: (off, dt.itemsize) for f, (dt, off) in RECORD_HEADER.fields.items()}
    assert got == want
    assert sum(size for _, size in got.values()) == RECORD_HEADER.itemsize      # no C field left out of the dtype


def _gather_worker(rank, world, port, out_q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    from datou_gomoku_muzero_b200.parallel import gather_packed_games
    from datou_gomoku_muzero_b200.trajectory import PackedGames
    from test_packed_records_cpu import packed_from_golden
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        names = ["selfplay_az_6_36", "selfplay_mz_6_50"] if rank == 0 else ["selfplay_mz_6_50_dense_f32"]
        if rank == 1 and world == 3:
            names = []
        recs, table, offs = [], [], [0]
        for i, nm in enumerate(names):
            z = np.load(os.path.join(GOLDEN_DIR, nm + ".npz"))
            r = packed_from_golden(z, game_seq=i, game=10 * rank + i, slot=i)
            recs.append(r); table.append([i, 10 * rank + i, len(r), int(z["winner"])]); offs.append(offs[-1] + len(r))
        import torch
        pg = None
        if recs:
            allr = np.zeros(offs[-1], recs[0].dtype)            # (np.concatenate would re-pack the padded record dtype)
            for r, o in zip(recs, offs):
                allr[o:o + len(r)] = r
            raw = allr.view(np.uint8).reshape(offs[-1], -1)
            pg = PackedGames(torch.from_numpy(raw.copy()), np.array(table, np.int32), offs, 6)
        got = gather_packed_games(pg, 6, dst=0)
        if rank == 0:
            h = got.host()
            out_q.put((len(got), got.n_moves, got.table.tolist(), [int(x) for x in got.offsets],
                       h["action"].tolist(), float(h["policy"].sum()), h["game"].tolist()))
        else:
            assert got is None
    finally:
        dist.destroy_process_group()


def test_gather_packed_games_two_ranks_gloo():
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    n_games, n_moves, table, offs, actions, polsum, games = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    zs = [np.load(os.path.join(GOLDEN_DIR, nm + ".npz")) for nm in ("selfplay_az_6_36", "selfplay_mz_6_50", "selfplay_mz_6_50_dense_f32")]
    lens = [len(z["actions"]) for z in zs]
    assert n_games == 3 and n_moves == sum(lens) and offs == [0, lens[0], lens[0] + lens[1], sum(lens)]
    assert [t[4] for t in table] == [0, 0, 1] and [t[2] for t in table] == lens          # source rank column, lengths
    assert actions == [int(a) for z in zs for a in z["actions"]]
    assert games == [0] * lens[0] + [1] * lens[1] + [10] * lens[2]
    assert abs(polsum - sum(float(z["policies"].sum()) for z in zs)) < 1e-9
