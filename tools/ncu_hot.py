"""Where the play kernel's instructions go: joins an .ncu-rep's per-SASS-instruction counters with the
line table of the cubin inside libgmz.so (nvdisasm -g) and prints, per source component, the static size,
the hot footprint and the dynamic instructions per simulation.
    python tools/ncu_hot.py gpurun_out/prof.ncu-rep <sims in the launch> [mangled kernel name] [libgmz.so]"""
import collections, csv, io, os, re, subprocess, sys, tempfile

rep, sims = sys.argv[1], float(sys.argv[2])
kern = sys.argv[3] if len(sys.argv) > 3 else "_Z9k_play_e0ILi2ELb0ELb0EEv6Params8PlayArgs"
# the four play-kernel cubins inside libgmz.so share one file name, so read the object of the instantiation instead
so = sys.argv[4] if len(sys.argv) > 4 else os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "datou_gomoku_muzero_b200",
                                                       "build", "release", "gmz_play_mz0_f0.o")
tmp = tempfile.mkdtemp()
subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(so)], cwd=tmp, capture_output=True)
dis, start = [], None
for cub in sorted(f for f in os.listdir(tmp) if f.endswith(".cubin")):      # the cubin that holds the kernel
    dis = subprocess.run(["nvdisasm", "-g", "-c", os.path.join(tmp, cub)], capture_output=True, text=True).stdout.split("\n")
    start = next((i for i, l in enumerate(dis) if l.startswith(".text." + kern + ":")), None)
    if start is not None:
        break
assert start is not None, f"{kern} not found in {so}"
end = next((i for i in range(start + 1, len(dis)) if dis[i].startswith("//--------------------- .text.")), len(dis))
cur, insts = ("?", 0), {}
for l in dis[start:end]:
    m = re.search(r'//## File "([^"]+)", line (\d+)', l)
    if m:
        cur = (m.group(1).split("/")[-1], int(m.group(2))); continue
    m = re.match(r"\s*/\*([0-9a-f]{4,6})\*/\s+(.*?);", l)
    if m:
        insts[int(m.group(1), 16)] = (cur, m.group(2))
raw = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv", "--print-source", "sass"], capture_output=True, text=True).stdout
rows = list(csv.reader(io.StringIO(raw)))
hdr, data = rows[1], rows[2:]
ia, isamp = hdr.index("Instructions Executed"), hdr.index("# Samples")
base = int(data[0][0], 16)
src_lines = {}
def text_of(f, l):
    if f not in src_lines:
        path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "datou_gomoku_muzero_b200", "csrc", f)
        src_lines[f] = open(path).read().split("\n") if os.path.exists(path) else []
    return src_lines[f][l - 1].strip()[:90] if 0 < l <= len(src_lines[f]) else ""
# component = enclosing function of the source line (nearest preceding line that looks like a function header)
def component(f, l):
    text_of(f, 1)
    L = src_lines.get(f, [])
    for k in range(min(l, len(L)) - 1, -1, -1):
        m = re.match(r"^(?:template.*>\s*)?(?:static\s+)?(?:__host__\s+)?(?:__device__|__global__)[^;(]*?\b(\w+)\s*\(", L[k])
        if m:
            return f"{f.split('.')[0].replace('gmz_', '')}:{m.group(1)}"
        m = re.match(r"^k_(\w+)\(", L[k])
        if m:
            return f"{f.split('.')[0].replace('gmz_', '')}:k_{m.group(1)}"
    return f
comp = collections.defaultdict(lambda: [0, 0, 0, 0]); line = collections.defaultdict(lambda: [0, 0])
ops = collections.Counter()
for r in data:
    off, e, s_ = int(r[0], 16) - base, int(r[ia]), int(r[isamp])
    (f, l), txt = insts.get(off, (("?", 0), r[1]))
    c = comp[component(f, l)]
    c[0] += 1; c[1] += 1 if e / sims >= 0.2 else 0; c[2] += e; c[3] += s_
    line[(f, l)][0] += e; line[(f, l)][1] += s_
    t = r[1].strip().split()
    ops[(t[1] if t[0].startswith("@") else t[0]).split(".")[0]] += e
tot, ts = sum(c[2] for c in comp.values()), sum(c[3] for c in comp.values())
print(f"{tot / sims:.0f} warp-instructions per simulation; hot footprint (>= 0.2 executions/sim): "
      f"{sum(c[1] for c in comp.values()) * 16 / 1024:.1f} KB\n")
print(f"{'component':34s} static   hot  dyn/sim   dyn%  stall-samples%")
for k, c in sorted(comp.items(), key=lambda x: -x[1][2])[:24]:
    print(f"{k:34s} {c[0]:6d} {c[1]:5d} {c[2] / sims:8.1f} {100 * c[2] / tot:6.1f} {100 * c[3] / max(ts, 1):8.1f}")
print("\nopcodes per simulation: " + ", ".join(f"{k} {v / sims:.0f}" for k, v in ops.most_common(22)))
print("\nhottest lines (dyn/sim, stall%):")
for (f, l), (e, s_) in sorted(line.items(), key=lambda x: -x[1][0])[:28]:
    print(f"{e / sims:7.1f} {100 * s_ / max(ts, 1):5.1f}  {f}:{l}  {text_of(f, l)}")
