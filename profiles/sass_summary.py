#!/usr/bin/env python
"""SASS opcode counts and register / spill table of the sweep kernels (no GPU needed):

    python profiles/sass_summary.py [RP ...]  > profiles/r02_sass_summary.txt

Reads the objects the in-tree build leaves in ccfindr_b200/csrc/_obj (cuobjdump -sass,
cuobjdump --dump-resource-usage).  The mnemonics that show the Blackwell path: UBLKCP (bulk
asynchronous copy global -> shared, the TMA engine), UBLKPF (bulk L2 prefetch), SYNCS (mbarrier),
LDS.128 (the gathers), DFMA (fp64 FMA), LDG.E.128 (the packed entries).  For each kernel also the
size of its chunk loop and the local-memory instructions (LDL/STL) inside it."""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
OBJ = os.path.join(ROOT, "ccfindr_b200", "csrc", "_obj")
WATCH = ["UBLKCP", "UBLKPF", "SYNCS", "LDS.128", "LDS.64", "LDG.E.128", "DFMA", "DMUL", "DADD",
         "FFMA", "MUFU", "SHFL", "STG", "STL", "LDL", "BAR", "UTMALDG", "UTCMMA"]


def demangle(name):
    return subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()


def chunk_loop(code):
    """(instructions, LDS.128, LDL/STL) of the chunk loop: the innermost backward branch whose
    body holds the gathers of at least one whole chunk (4 steps)"""
    best = None
    for a, ins in code:
        m = re.search(r"BRA\S*\s+(?:\S+,\s*)?(0x[0-9a-f]+)\s*$", ins)
        if m and int(m.group(1), 16) < a:
            body = [i for x, i in code if int(m.group(1), 16) <= x <= a]
            lds = sum("LDS.128" in i for i in body)
            if lds >= 16 and (best is None or len(body) < best[0]):
                best = (len(body), lds, sum(bool(re.search(r"\b(LDL|STL)", i)) for i in body))
    return best


def main():
    rps = [int(a) for a in sys.argv[1:]] or [10, 16, 20]
    for rp in rps:
        obj = os.path.join(OBJ, "rp_inst_%d.o" % rp)
        sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
        res = subprocess.run(["cuobjdump", "--dump-resource-usage", obj], capture_output=True,
                             text=True).stdout
        usage = {}
        cur = None
        for ln in res.splitlines():
            m = re.search(r"Function (\S+):", ln)
            if m:
                cur = m.group(1)
            m = re.search(r"REG:(\d+).*?SHARED:(\d+).*?LOCAL:(\d+)", ln)
            if m and cur:
                usage[cur] = (int(m.group(1)), int(m.group(2)), int(m.group(3)))
        print("== rp_inst_%d.o  (arch %s)" % (rp, re.search(r"arch = (\S+)", sass).group(1)))
        fn = None
        counts = collections.Counter()

        def flush():
            if fn and "sweep_" in fn:
                d = demangle(fn)
                d = d[d.index("sweep_"):d.index("(vb::Sweep")] if "(vb::Sweep" in d else d
                u = usage.get(fn, (0, 0, 0))
                tot = sum(counts.values())
                print("  %-62s regs %3d  static smem %4d B  local (spill) %4d B  SASS %5d" % (
                    d, u[0], u[1], u[2], tot))
                print("     " + "  ".join("%s %d" % (k, counts[k]) for k in WATCH if counts[k]))
                loop = chunk_loop(code)
                if loop:
                    print("     chunk loop: %d instructions, %d LDS.128, %d LDL/STL" % loop)

        for ln in sass.splitlines():
            m = re.search(r"Function : (\S+)", ln)
            if m:
                flush()
                fn = m.group(1)
                counts = collections.Counter()
                code = []
                continue
            m = re.search(r"/\*([0-9a-f]{4,5})\*/\s+(.*?);", ln)
            if m:
                code.append((int(m.group(1), 16), m.group(2)))
            m = re.search(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", ln)
            if m:
                op = m.group(1)
                counts["__all__" if False else op.split(".")[0]] += 0
                for w in WATCH:
                    if op == w or op.startswith(w + ".") or (w.count(".") and op.startswith(w)):
                        counts[w] += 1
                counts["_"] += 1
        flush()


if __name__ == "__main__":
    main()
