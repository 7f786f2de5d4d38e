#!/usr/bin/env python3
"""Static SASS size of k_rao_fused2 per kernel PHASE (same source-line phases as tools/ncu_phases.py), without a GPU.

Counts the instructions ptxas emitted for each phase (not how often they execute) and their FP64 share; the pass loop's
instruction-cache footprint is the sum of the part-1 .. flags rows.

usage: tools/sass_phases.py [path/to/libraftk.so] [kernel symbol substring, default k_rao_fused2; the lean instantiation
       is k_rao_fused2ILb0E, the full one k_rao_fused2ILb1E]"""
import collections, os, re, subprocess, sys, tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
so = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "raft_b200", "csrc", "libraftk.so")
KERN = sys.argv[2] if len(sys.argv) > 2 else "k_rao_fused2"
FUSED = "raftk_fused2.cuh"
tmp = tempfile.mkdtemp()
subprocess.check_call(["cuobjdump", "-xelf", "all", so], cwd=tmp, stdout=subprocess.DEVNULL)
cubin = [f for f in os.listdir(tmp) if f.endswith(".cubin")][0]
sass = subprocess.check_output(["nvdisasm", "-gi", "-c", os.path.join(tmp, cubin)], text=True).split("\n")
# the phase markers are read from the source the library was built from (same directory as the library, else the tree's)
srcdir = os.path.dirname(os.path.abspath(so))
if not os.path.exists(os.path.join(srcdir, FUSED)):
    srcdir = os.path.join(ROOT, "raft_b200", "csrc")
fsrc = open(os.path.join(srcdir, FUSED)).read().split("\n")


def find(s):
    for i, l in enumerate(fsrc):
        if s in l:
            return i + 1
    return None


marks = [("stage (TMA blob)", 1), ("prologue", find("---- prologue (a)")), ("part1 walk", find("= pass part 1")),
         ("part1 warp reduce", find("warp sum of the 30 accumulators")), ("cross-warp/cluster reduce", find("for (int t = tid; t < nchunk * 32; t += T) {")),
         ("coefficients+B_drag", find("= linearised coefficients per node")), ("part2 walk", find("= pass part 2")),
         ("park+assembly", find("bin B's drag excitation waits")), ("solve6 call+conv", find("const bool ok = solve6")),
         ("flags/cluster sync", find("passes++;")), ("epilogue", find("if (P.status && rank == 0 && tid == 0)"))]
marks = [(n, l) for n, l in marks if l]
kstart = find("k_rao_fused2(DesignsDev D")
order = [n for n, _ in marks] + ["solve6 (LU)"]
agg = collections.defaultdict(collections.Counter)
infn, cur, lu, cur_idx, seen_later, in_chain = False, None, False, 0, False, False
for l in sass:
    if l.startswith("//--------------------- .text."):
        infn = KERN in l and "plan" not in l
        cur, lu, cur_idx, seen_later = None, False, 0, False
    if not infn:
        continue
    if l.lstrip().startswith("//## File"):
        # consecutive lines form one inlining chain, innermost first; an inlined helper is attributed to its outermost
        # call site in the kernel's source
        if not in_chain:
            chain, in_chain = [], True
        chain += [(f, int(n)) for f, n in re.findall(r'"[^"]*?/csrc/([\w.]+)", line (\d+)', l)]
        own = [fl for fl in chain if fl[0] == FUSED]
        cur = own[-1] if own else None
        lu = any(f == "raftk_common.cuh" and n > 84 for f, n in chain)
        continue
    in_chain = False
    m = re.search(r"/\*([0-9a-f]{4,})\*/\s+(?:@!?U?P\w+\s+)?([A-Z][\w.]*)", l)
    if not m:
        continue
    op = m.group(2)
    if cur is not None and cur[0] == FUSED and cur[1] >= kstart:
        cand = [k for k, (n, ln) in enumerate(marks) if ln <= cur[1]][-1]
        if cand > 0 or not seen_later:
            cur_idx = cand
        if cand > 0:
            seen_later = True
    ph = marks[cur_idx][0]
    if lu:
        ph = "solve6 (LU)"
    agg[ph]["instr"] += 1
    if op.startswith(("DFMA", "DMUL", "DADD", "DSETP", "MUFU")):
        agg[ph]["fp64"] += 1
    if op.startswith(("LDS", "STS")):
        agg[ph]["smem"] += 1
tot = sum(c["instr"] for c in agg.values())
print("k_rao_fused2 in %s: %d SASS instructions (%.1f KB)" % (so, tot, tot * 16 / 1024))
print("%-28s %7s %8s %6s %6s" % ("phase", "instr", "KB", "fp64", "smem"))
for ph in order:
    c = agg.get(ph)
    if c:
        print("%-28s %7d %8.1f %6.2f %6d" % (ph, c["instr"], c["instr"] * 16 / 1024, c["fp64"] / c["instr"], c["smem"]))
loop = sum(agg[p]["instr"] for p in order[order.index("part1 walk"):order.index("epilogue")] + ["solve6 (LU)"])
print("pass loop (part1 walk .. flags, LU included): %d instructions = %.1f KB" % (loop, loop * 16 / 1024))
