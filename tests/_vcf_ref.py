"""ctypes wrapper over tests/csrc/vcf_ref.c -- TEST INFRASTRUCTURE: the CPU restatement of the VCF solver
(include/gmz.h gmz_vcf_solve), compiled on first use into a private temporary directory (the repository tree may be
read-only)."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "vcf_ref.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="gmz_vcf_ref_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libvcf_ref.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-fopenmp", "-shared", "-o", so, _SRC])
        _lib = C.CDLL(so)
        _lib.vcf_ref_solve.restype = C.c_int
    return _lib


def first_bits(first, A):
    """uint64 [B, 6] bitmasks -> bool [B, A]."""
    first = np.ascontiguousarray(first, np.uint64)
    bits = np.unpackbits(first.view(np.uint8).reshape(len(first), -1), axis=1, bitorder="little")
    return bits[:, :A].astype(bool)


def solve(boards, players, board_size, n_in_row=5, max_attacks=8, node_budget=1 << 20):
    """(length int32 [B], first bool [B, A], nodes int32 [B]) as gmz_vcf_solve defines them."""
    N = int(board_size)
    A = N * N
    b = np.ascontiguousarray(np.asarray(boards).reshape(-1, A), np.int8)
    B = b.shape[0]
    p = np.ascontiguousarray(np.asarray(players).reshape(B), np.int8)
    length, nodes = np.zeros(B, np.int32), np.zeros(B, np.int32)
    first = np.zeros((B, 6), np.uint64)
    ptr = lambda a, t: a.ctypes.data_as(C.POINTER(t))
    rc = lib().vcf_ref_solve(ptr(b, C.c_int8), ptr(p, C.c_int8), B, N, int(n_in_row), int(max_attacks), int(node_budget),
                             ptr(length, C.c_int32), ptr(first, C.c_uint64), ptr(nodes, C.c_int32))
    if rc:
        raise ValueError("vcf_ref_solve refused its arguments")
    return length, first_bits(first, A), nodes
