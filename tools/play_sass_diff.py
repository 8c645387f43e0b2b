"""Check that the default persistent play kernel compiles to the same machine code as at another commit.

    python tools/play_sass_diff.py [REV]        (default REV: HEAD~1)

Builds gmz_play_inst.cu of REV (from `git archive`) and of the working tree into a temporary directory, with
_build.NVCC_FLAGS and -Xptxas -v, for every (MZ, F32) pair; the working tree also for GMZ_PLAY_BOOK=1.  Every
k_play_e0 instantiation of REV is matched with the working tree's one of the same NC / MZ / F32 and BOOK = false (a
REV kernel without the BOOK parameter matches that one too); their `cuobjdump -sass` bodies are compared without the
mangled names, and ptxas's registers, stack and spill bytes of both are printed and compared.  The book variants'
ptxas figures are printed too.  Exit status 1 on any difference.  Needs nvcc and cuobjdump, no GPU."""
from __future__ import annotations

import os
import re
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from datou_gomoku_muzero_b200._build import NVCC_FLAGS  # noqa: E402

CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
KERNEL = re.compile(r"_Z9k_play_e0ILi(\d)ELb([01])ELb([01])E(?:Lb([01])E)?Ev6Params8PlayArgs")


def sass_functions(obj):
    """mangled name -> instruction lines of `cuobjdump -sass` (addresses and encodings kept)."""
    out = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", obj], check=True, capture_output=True,
                         text=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
        elif cur is not None and line.strip():
            cur.append(line.strip())
    return funcs


def ptxas_props(text):
    """mangled entry name -> (registers, stack frame, spill stores, spill loads) from -Xptxas -v output."""
    props, name, spill = {}, None, None
    for line in text.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            name, spill = m.group(1), None
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            spill = tuple(int(x) for x in m.groups())
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and name and spill is not None:
            props[name] = (int(m.group(1)),) + spill
            name = spill = None
    return props


def kernels(obj, log):
    """(NC, MZ, F32, BOOK) -> (sass body, ptxas figures) of the k_play_e0 instantiations in one object."""
    props = ptxas_props(log)
    out = {}
    for name, body in sass_functions(obj).items():
        m = KERNEL.fullmatch(name)
        if m:
            out[(int(m.group(1)), int(m.group(2)), int(m.group(3)), int(m.group(4) or 0))] = (body, props.get(name))
    return out


def compile_obj(src_root, mz, f32, book, out):
    cmd = [os.path.join(CUDA, "bin", "nvcc"), *NVCC_FLAGS, "-Xptxas", "-v", f"-DGMZ_PLAY_MZ={mz}", f"-DGMZ_PLAY_F32={f32}",
           f"-DGMZ_PLAY_BOOK={book}", "-c", os.path.join(src_root, "datou_gomoku_muzero_b200", "csrc", "gmz_play_inst.cu"),
           "-o", out]
    r = subprocess.run(cmd, check=True, capture_output=True, text=True)
    return out, r.stdout + r.stderr


def main(rev):
    with tempfile.TemporaryDirectory() as tmp:
        old_root = os.path.join(tmp, "old")
        os.makedirs(old_root)
        tar = subprocess.run(["git", "-C", ROOT, "archive", rev, "datou_gomoku_muzero_b200/csrc", "include"], check=True,
                             capture_output=True).stdout
        subprocess.run(["tar", "x", "-C", old_root], input=tar, check=True)
        jobs = []
        for mz in (0, 1):
            for f in (0, 1):
                jobs.append(("old", mz, f, 0, old_root))
                jobs.append(("new", mz, f, 0, ROOT))
                jobs.append(("new", mz, f, 1, ROOT))
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            res = list(ex.map(lambda j: compile_obj(j[4], j[1], j[2], j[3], os.path.join(tmp, f"{j[0]}_mz{j[1]}_f{j[2]}_b{j[3]}.o")),
                              jobs))
        found = {}
        for (side, *_), (obj, log) in zip(jobs, res):
            for k, v in kernels(obj, log).items():
                found[(side,) + k] = v
    bad = 0
    for (side, nc, mz, f, book), (body, props) in sorted(found.items()):
        if side != "old":
            continue
        new = found.get(("new", nc, mz, f, 0))
        if new is None:
            print(f"NC={nc} MZ={mz} F32={f}: no default kernel in the working tree")
            bad = 1
            continue
        same = body == new[0] and props == new[1]
        print(f"NC={nc} MZ={mz} F32={f} BOOK=0: {len(body)} SASS lines {'identical' if body == new[0] else 'DIFFERENT'}; "
              f"ptxas (registers, stack, spill stores, spill loads) {props} -> {new[1]}")
        bad |= not same
    for (side, nc, mz, f, book), (body, props) in sorted(found.items()):
        if side == "new" and book:
            print(f"NC={nc} MZ={mz} F32={f} BOOK=1: {len(body)} SASS lines; ptxas {props}")
    return bad


if __name__ == "__main__":
    if len(sys.argv) > 2:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1] if len(sys.argv) == 2 else "HEAD~1"))
