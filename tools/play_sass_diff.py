"""Check that the persistent play kernel compiles to the same machine code as at another commit.

    python tools/play_sass_diff.py [REV]        (default REV: HEAD~1)

Builds gmz_play_inst.cu of REV (from `git archive`) and of the working tree into a temporary directory, with
_build.NVCC_FLAGS and -Xptxas -v, for every (MZ, F32) pair.  Every k_play_e0<NC, MZ, F32> of the working tree is matched
with REV's one of the same NC / MZ / F32 (a REV that still has the opening-book parameter is built with
-DGMZ_PLAY_BOOK=1 and its BOOK = true kernel is the match); their `cuobjdump -sass` bodies are compared without the
mangled names, and ptxas's registers, stack and spill bytes of both are printed and compared.  Exit status 1 on any
difference.  Needs nvcc and cuobjdump, no GPU."""
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
    """(NC, MZ, F32) -> (sass body, ptxas figures) of the k_play_e0 instantiations in one object (BOOK = true only, where
    the kernel still has that parameter)."""
    props = ptxas_props(log)
    out = {}
    for name, body in sass_functions(obj).items():
        m = KERNEL.fullmatch(name)
        if m and m.group(4) != "0":
            out[(int(m.group(1)), int(m.group(2)), int(m.group(3)))] = (body, props.get(name))
    return out


def compile_obj(src_root, mz, f32, out):
    cmd = [os.path.join(CUDA, "bin", "nvcc"), *NVCC_FLAGS, "-Xptxas", "-v", f"-DGMZ_PLAY_MZ={mz}", f"-DGMZ_PLAY_F32={f32}",
           "-DGMZ_PLAY_BOOK=1", "-c", os.path.join(src_root, "datou_gomoku_muzero_b200", "csrc", "gmz_play_inst.cu"),
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
        jobs = [(side, mz, f, src) for mz in (0, 1) for f in (0, 1) for side, src in (("old", old_root), ("new", ROOT))]
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            res = list(ex.map(lambda j: compile_obj(j[3], j[1], j[2], os.path.join(tmp, f"{j[0]}_mz{j[1]}_f{j[2]}.o")), jobs))
        found = {}
        for (side, *_), (obj, log) in zip(jobs, res):
            for k, v in kernels(obj, log).items():
                found[(side,) + k] = v
    bad = 0
    for (side, nc, mz, f), (body, props) in sorted(found.items()):
        if side != "new":
            continue
        old = found.get(("old", nc, mz, f))
        if old is None:
            print(f"NC={nc} MZ={mz} F32={f}: no kernel at {rev}")
            bad = 1
            continue
        print(f"NC={nc} MZ={mz} F32={f}: {len(body)} SASS lines {'identical' if body == old[0] else 'DIFFERENT'}; "
              f"ptxas (registers, stack, spill stores, spill loads) {old[1]} -> {props}")
        bad |= body != old[0] or props != old[1]
    return bad

if __name__ == "__main__":
    if len(sys.argv) > 2:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1] if len(sys.argv) == 2 else "HEAD~1"))
