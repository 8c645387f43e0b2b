"""CPU-side checks of the boundary: the C-ABI library loads without a GPU and exports every
symbol include/gmz.h declares; host-side contract types and the game API behave like the
reference's; the product never imports the oracle."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "gmz.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gmz_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from datou_gomoku_muzero_b200 import _build, _lib
    _build.build()
    names = _declared()
    assert len(names) >= 20
    lib = ctypes.CDLL(_lib.SO)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/gmz.h but not exported by libgmz.so"
    assert set(_lib.SIGNATURES) == set(names), "ctypes SIGNATURES out of sync with include/gmz.h"
    loaded = _lib.load()
    assert loaded.gmz_version() == 200


def test_config_validation_without_gpu():
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    ok = _lib.GmzConfig(15, 5, 400, 16, 0, 4096, 0, 0, 30.0, 1.0, 1e-3, 0.997)
    nbytes = lib.gmz_workspace_bytes(ctypes.byref(ok))
    assert 4.1e9 < nbytes < 4.5e9          # 4096 games x 400 nodes x (1 KiB logits + 512 B children + 1 KiB node block + own stats)
    for bad in (_lib.GmzConfig(20, 5, 400, 16, 0, 1, 0, 0, 30.0, 1.0, 1e-3, 0.997),      # board too large
                _lib.GmzConfig(15, 5, 0, 16, 0, 1, 0, 0, 30.0, 1.0, 1e-3, 0.997),        # no simulations
                _lib.GmzConfig(15, 5, 400, 33, 0, 1, 0, 0, 30.0, 1.0, 1e-3, 0.997),      # too many top actions
                _lib.GmzConfig(15, 5, 400, 16, 7, 1, 0, 0, 30.0, 1.0, 1e-3, 0.997),      # unknown mode
                _lib.GmzConfig(15, 5, 400, 16, 0, 1, 0, 5, 30.0, 1.0, 1e-3, 0.997)):     # unknown accumulation dtype
        assert lib.gmz_workspace_bytes(ctypes.byref(bad)) == 0
        assert lib.gmz_last_error()
    assert lib.gmz_set_roots(None, None, None, None, None, None) != 0     # null engine is an error, not a crash
    f32 = _lib.GmzConfig(15, 5, 400, 16, 0, 4096, 0, _lib.GMZ_ACCUM_F32, 30.0, 1.0, 1e-3, 0.997)
    assert lib.gmz_workspace_bytes(ctypes.byref(f32)) == nbytes           # float32 accumulation: same layout
    # handles that are not live are rejected, and destroying one (again) is a harmless no-op
    bogus = ctypes.c_void_p(0x1000)
    assert lib.gmz_finalize(bogus, None, None, None, None, None) != 0 and b"destroyed" in lib.gmz_last_error()
    assert lib.gmz_destroy(bogus) == 0 and lib.gmz_destroy(None) == 0


def test_engine_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from datou_gomoku_muzero_b200 import _lib
    from datou_gomoku_muzero_b200.engine import SearchEngine
    from datou_gomoku_muzero_b200.replay_buffer import InMemoryReplayBuffer
    with pytest.raises(_lib.GmzError):
        SearchEngine(1)
    with pytest.raises(_lib.GmzError):
        InMemoryReplayBuffer(8)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "datou_gomoku_muzero_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower(), f"{f} mentions the oracle"


def test_game_api_matches_reference_kat():
    """GomokuGame host class vs the reference KATs (game.py:20-63)."""
    from datou_gomoku_muzero_b200.game import GomokuGame
    z = np.load(os.path.join(ROOT, "tests", "golden", "game_kat.npz"))
    for i in range(0, int(z["n"]), 3):
        N, nir = int(z["N"][i]), int(z["nir"][i])
        g = GomokuGame(board_size=N, n_in_row=nir)
        g.board = z["boards"][i][:N * N].reshape(N, N).copy()
        last = int(z["last"][i])
        g.last_move, g.move_count = (last // N, last % N), int(z["move_count"][i])
        w = g.get_game_ended()
        assert (2 if w is None else int(w)) == int(z["ended"][i])
        assert bool(g.check_win()) == bool(z["win"][i])
    g = GomokuGame(board_size=6)
    assert g.get_board_state(1, None).shape == (3, 6, 6) and g.get_board_state(1, None).dtype == np.float32
    g.do_move(7); g.do_move(7)                       # overwrite is allowed (game.py:22)
    assert g.board[1, 1] == -1 and g.move_count == 2 and g.current_player == 1 and g.last_move == (1, 1)
    assert len(g.get_valid_moves()) == 35


def test_contract_types():
    from datou_gomoku_muzero_b200 import GameRecord, TrainingSlice
    assert GameRecord._fields == ("observations", "actions", "rewards", "policies", "values", "board_states")
    assert TrainingSlice._fields == ("observation", "action_history", "reward_history", "policy_history", "value_history")


def test_entry_points_reject_bad_arguments_without_crashing():
    """Error behaviour of the boundary: every entry point validates its arguments before touching the
    device, returns non-zero and leaves a message in gmz_last_error() (no GPU needed for these paths)."""
    import ctypes as C
    from datou_gomoku_muzero_b200 import _lib
    lib = _lib.load()
    N = None
    calls = [
        ("gmz_set_roots", (N, N, N, N, N, N)), ("gmz_games_reset", (N, N, N)), ("gmz_root_obs", (N, N, 0, N)),
        ("gmz_get_roots", (N, N, N, N, N, N)), ("gmz_root_expand", (N, N, N, 0, N, N)),
        ("gmz_select", (N, N, 0, N, N, N)), ("gmz_select_mz", (N, N, N, N, N, N, N)),
        ("gmz_expand_backup", (N, N, N, N, 0, N)), ("gmz_finalize", (N, N, N, N, N, N)),
        ("gmz_e0_eval_obs", (N, 4, 9, 0, 16, N, N, N)), ("gmz_search_e0", (N, N, 0, 16, N, N, N)),
        ("gmz_fill_gumbel", (N, 8, 0, 0, N)), ("gmz_game_step", (N, N, N, N)),
        ("gmz_traj_init", (N, N, N)), ("gmz_selfplay_e0", (N, N, 0, 16, 0, 8, 1, N)),
        ("gmz_selfplay_unpark", (N, N, N)), ("gmz_selfplay_step", (N, N, N, N, N, 1, N, N)),
        ("gmz_play_counters", (N, N, N)), ("gmz_select_counters", (N, N, N)),
        ("gmz_hidden_gather", (N, N, N, 4, 20, 4, 36, 256, N, 0, N, N)), ("gmz_hidden_scatter", (N, N, 4, 20, 4, 9216, N, N)),
        ("gmz_tactics_classify", (N, N, 4, 9, 5, N, N)), ("gmz_per_update", (N, 8, N, N, 4, N)),
        ("gmz_per_add", (N, 8, 0, N, 4, N, N)), ("gmz_per_sample", (N, 8, 8, N, 4, 0.4, N, N, N, N)),
        ("gmz_traj_pack", (N, 9, N, 1, N, N, 5, N, N)), ("gmz_records_batch", (N, 8, 9, N, 4, 5, 0, 0, N, N, N, N, N, N)),
        ("gmz_records_tactics", (N, 4, 9, 5, N, N)), ("gmz_set_roots_from_records", (N, N, 8, 0, 4, N)),
        ("gmz_records_writeback", (N, 8, 9, 0, 4, N, N, N)), ("gmz_records_retarget", (N, 8, 9, 0, 4, N, 5, N)),
        ("gmz_records_compact", (N, 8, 9, 0, 4, N, N, N, N)), ("gmz_records_expand", (N, N, 4, N, N, 1, 0, 9, N, 8, 0, N)),
    ]
    for name, args in calls:
        rc = getattr(lib, name)(*args)
        assert rc != 0, f"{name} accepted null arguments"
        assert lib.gmz_last_error(), f"{name} left no error message"
        assert name.encode() in lib.gmz_last_error(), f"{name} error message does not name it: {lib.gmz_last_error()}"
    one = (C.c_double * 1)(1.0)
    assert lib.gmz_per_add(one, 8, 9, one, 1, (C.c_int64 * 1)(0), None) != 0          # write_ptr outside the ring
    assert lib.gmz_tactics_classify((C.c_int8 * 4)(), (C.c_int8 * 1)(1), 1, 40, 5, (C.c_int8 * 4)(), None) != 0   # board too large
    assert lib.gmz_e0_eval_obs(None, 0, 9, 0, 16, None, None, None) != 0 or True      # empty batch of nothing is a no-op or an error, never a crash
    # without a CUDA device gmz_create must fail cleanly as well
    import torch
    if not torch.cuda.is_available():
        cfg = _lib.GmzConfig(9, 5, 16, 4, 0, 2, 0, 0, 30.0, 1.0, 1e-3, 0.997)
        nbytes = lib.gmz_workspace_bytes(C.byref(cfg))
        buf = (C.c_char * (nbytes + 512))()
        addr = (C.addressof(buf) + 255) // 256 * 256
        h = C.c_void_p()
        assert lib.gmz_create(C.byref(cfg), C.c_void_p(addr), nbytes, None, C.byref(h)) != 0
        assert b"cuda" in lib.gmz_last_error().lower() or lib.gmz_last_error()
