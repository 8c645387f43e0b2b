"""ctypes wrapper over tests/csrc/vct_ref.c -- TEST INFRASTRUCTURE: the CPU restatement of the VCT solver
(include/gmz.h gmz_vct_solve) in its brute-force and filtered modes, compiled on first use into a private temporary
directory (the repository tree may be read-only)."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from _vcf_ref import first_bits

_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="gmz_vct_ref_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libvct_ref.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-fopenmp", "-shared", "-I", _DIR, "-o", so,
                               os.path.join(_DIR, "vct_ref.c")])
        _lib = C.CDLL(so)
        _lib.vct_ref_solve.restype = C.c_int
    return _lib


def solve(boards, players, board_size, n_in_row=5, max_attacks=8, node_budget=1 << 20, filtered=True):
    """(length int32 [B], first bool [B, A], nodes int32 [B]) as gmz_vct_solve defines them; filtered=False finds
    every set by brute force."""
    N = int(board_size)
    A = N * N
    b = np.ascontiguousarray(np.asarray(boards).reshape(-1, A), np.int8)
    B = b.shape[0]
    p = np.ascontiguousarray(np.asarray(players).reshape(B), np.int8)
    length, nodes = np.zeros(B, np.int32), np.zeros(B, np.int32)
    first = np.zeros((B, 6), np.uint64)
    ptr = lambda a, t: a.ctypes.data_as(C.POINTER(t))
    rc = lib().vct_ref_solve(ptr(b, C.c_int8), ptr(p, C.c_int8), B, N, int(n_in_row), int(max_attacks), int(node_budget),
                             int(bool(filtered)), ptr(length, C.c_int32), ptr(first, C.c_uint64), ptr(nodes, C.c_int32))
    if rc:
        raise ValueError("vct_ref_solve refused its arguments")
    return length, first_bits(first, A), nodes


def sets(board, n_in_row=5, filtered=True):
    """(X's threat moves, Y's replies R = D | K) of one position, board int8 [N, N] with X = +1: sets of (row, col)."""
    b = np.ascontiguousarray(board, np.int8)
    N = b.shape[0]
    t, r = np.zeros(6, np.uint64), np.zeros(6, np.uint64)
    lib().vct_ref_sets(b.ctypes.data_as(C.POINTER(C.c_int8)), N, int(n_in_row), int(bool(filtered)),
                       t.ctypes.data_as(C.POINTER(C.c_uint64)), r.ctypes.data_as(C.POINTER(C.c_uint64)))
    cells = lambda m: {divmod(int(a), N) for a in np.flatnonzero(first_bits(m[None], N * N)[0])}
    return cells(t), cells(r)
