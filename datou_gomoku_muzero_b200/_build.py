"""In-tree nvcc build of libgmz.so (sm_100a only).  Used by __graft_entry__.build()."""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libgmz.so")
SOURCES = ["gmz_engine.cu", "gmz_per.cu", "gmz_tactics.cu", "gmz_hidden.cu", "gmz_records.cu"]
# the persistent play kernel: one object per (MuZero mode, float32 accumulation), built in parallel
PLAY_SOURCE = "gmz_play_inst.cu"
PLAY_VARIANTS = [(0, 0), (0, 1), (1, 0), (1, 1)]
HEADERS = ["gmz_common.cuh", "gmz_tree.cuh", "gmz_play.cuh", "gmz_tactics.cuh", "gmz_records.cuh", "gmz_internal.h", os.path.join("..", "..", "include", "gmz.h")]
# -fmad=false: the search's float64 / float32 arithmetic must round once per operation, like the
# reference's Python floats / NumPy scalars (SURVEY.md App. A.7); an FMA would change visit counts.
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false",
              "-std=c++17", "-Xcompiler", "-fPIC"]


# The same library with every certified select decision re-derived by the exact float64 path and the
# disagreements counted (gmz_select_counters): loaded only by tests/test_certified_select_gpu.py and
# tools/soak_parity.py through GMZ_LIB, never by the package itself.
SO_VERIFY = os.path.join(HERE, "libgmz_verify.so")


def _stale(so=SO) -> bool:
    if not os.path.exists(so):
        return True
    t = os.path.getmtime(so)
    deps = [os.path.join(CSRC, s) for s in SOURCES + [PLAY_SOURCE] + HEADERS]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, verify: bool = False, variant: str = "", defines=()) -> str:
    """variant / defines: development builds with extra -D flags into build_variants/libgmz_<variant>.so
    (loaded through the GMZ_LIB override by tools/kbench.py; never by the package itself)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    so = SO_VERIFY if verify else SO
    if variant:
        os.makedirs(os.path.join(os.path.dirname(HERE), "build_variants"), exist_ok=True)
        so = os.path.join(os.path.dirname(HERE), "build_variants", f"libgmz_{variant}.so")
    if not force and not _stale(so):
        return so
    objdir = os.path.join(HERE, "build", variant or ("verify" if verify else "release"))
    os.makedirs(objdir, exist_ok=True)
    common = [nvcc, *NVCC_FLAGS, *(["-DGMZ_VERIFY_FAST"] if verify else []), *(["-Xptxas", "-v"] if verbose else []),
              *[f"-D{d}" for d in defines]]
    jobs = []
    for s in SOURCES:
        jobs.append((common + ["-c", os.path.join(CSRC, s), "-o", os.path.join(objdir, s[:-3] + ".o")]))
    for mz, f32 in PLAY_VARIANTS:
        jobs.append(common + [f"-DGMZ_PLAY_MZ={mz}", f"-DGMZ_PLAY_F32={f32}", "-c", os.path.join(CSRC, PLAY_SOURCE),
                              "-o", os.path.join(objdir, f"gmz_play_mz{mz}_f{f32}.o")])
    with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
        list(ex.map(subprocess.check_call, jobs))
    objs = [j[-1] for j in jobs]
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", so, *objs])
    return so
