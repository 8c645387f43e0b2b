"""ctypes wrapper over tests/csrc/tree_oracle.c -- TEST INFRASTRUCTURE: the CPU oracle's search with its whole tree.

The C file includes oracle/gmz_oracle.c unchanged, so this is the oracle's search; it is compiled on first use with the
oracle's flags into a private temporary directory (the repository tree may be read-only)."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "tree_oracle.c")
_FLAGS = ["-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-shared"]
_lib = None


class TroTree(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in (
        "parent", "action", "depth", "visits", "value_sum", "reward", "prior_logit", "counts", "minmax",
        "topk_action", "topk_round", "topk_gumbel", "topk_logit")]


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="gmz_tree_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libtree_oracle.so")
        subprocess.check_call(["gcc", *_FLAGS, "-o", so, _SRC, "-lm"])
        _lib = C.CDLL(so)
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def search_tree(cfg, board, player, last_move, move_count, gumbel):
    """One oracle search (cfg: oracle.OrcConfig) and the whole tree it built.  Returns a dict: the search's rc / policy /
    value / action / visits / leaf_actions / leaf_depths (as oracle.search(trace=True)); per node k < num_nodes (node 0
    the root, node k the k-th created) parent, node_action, depth, node_visits, value_sum, reward, prior_logit (the
    parent's logit at the node's action, NaN for the root); num_nodes, sim_count, phase, n_surv, n_init, minmax
    (minimum, maximum); the initial top-k in halving order (topk_action, topk_gumbel, topk_logit, topk_round = the
    halving round that eliminated each entry, `phase` for the survivors)."""
    A, S, K = cfg.board_size ** 2, cfg.num_simulations, cfg.num_top_actions
    board = np.ascontiguousarray(board, dtype=np.int8).reshape(A)
    gumbel = np.ascontiguousarray(gumbel, dtype=np.float64).reshape(A)
    policy = np.zeros(A, np.float64)
    value = C.c_double(0.0)
    action = C.c_int32(-1)
    visits = np.zeros(A, np.int32)
    la = np.full(S + 1, -1, np.int32)
    ld = np.full(S + 1, -1, np.int32)
    arr = dict(parent=np.zeros(S, np.int32), action=np.zeros(S, np.int32), depth=np.zeros(S, np.int32),
               visits=np.zeros(S, np.int32), value_sum=np.zeros(S, np.float64), reward=np.zeros(S, np.float64),
               prior_logit=np.zeros(S, np.float32), counts=np.zeros(5, np.int32), minmax=np.zeros(2, np.float64),
               topk_action=np.zeros(K, np.int32), topk_round=np.zeros(K, np.int32), topk_gumbel=np.zeros(K, np.float64),
               topk_logit=np.zeros(K, np.float32))
    tree = TroTree(*[arr[f].ctypes.data for f, _ in TroTree._fields_])
    rc = lib().tro_search_tree(C.byref(cfg), _p(board, C.c_int8), int(player), int(last_move), int(move_count),
                               _p(gumbel, C.c_double), _p(policy, C.c_double), C.byref(value), C.byref(action),
                               _p(visits, C.c_int32), _p(la, C.c_int32), _p(ld, C.c_int32), C.byref(tree))
    n, sim, phase, n_surv, n_init = (int(x) for x in arr["counts"])
    n_evals = int((la >= 0).sum()) if rc == 0 else 0
    out = dict(rc=rc, policy=policy, value=value.value, action=action.value, visits=visits, num_nodes=n, sim_count=sim,
               phase=phase, n_surv=n_surv, n_init=n_init, minmax=arr["minmax"],
               leaf_actions=la[:n_evals].copy(), leaf_depths=ld[:n_evals].copy())
    for f in ("parent", "action", "depth", "visits", "value_sum", "reward", "prior_logit"):
        out["node_" + f if f in ("action", "visits") else f] = arr[f][:n].copy()
    for f in ("topk_action", "topk_round", "topk_gumbel", "topk_logit"):
        out[f] = arr[f][:n_init].copy()
    return out
