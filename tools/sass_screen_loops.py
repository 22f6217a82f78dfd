#!/usr/bin/env python
"""Spill traffic inside the histogram screen's band loops (qo_ts.cuh::qo_mc_ts_screen_kernel), from the machine code of the object
files next to the library: per instantiation, the innermost backward-branch loop around each __any_sync of the screen (VOTE.ANY
on a predicate; the out-of-line WARPSYNC.COLLECTIVE stubs are skipped) -- the twelve-point Horner of S, the exact path of a batch
and the in-place update -- with its LDL / STL / LDS counts, and the LDL count of the whole kernel.

  python tools/sass_screen_loops.py [objects...]      (default: qo-100-tools_b200/lib/qo_ts2s?.o)"""
import glob
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def screen_loops(obj):
    sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    out = []
    for blk in re.split(r"\n\s*Function : ", sass)[1:]:
        name = blk.split("\n", 1)[0].strip()
        ins = []
        for ln in blk.split("\n"):
            m = re.search(r"/\*([0-9a-f]{4,6})\*/\s+(.*?);", ln)
            if m:
                ins.append((int(m.group(1), 16), m.group(2).strip()))
        votes = [a for i, (a, t) in enumerate(ins) if re.search(r"VOTE\.ANY P", t) and not (i and "WARPSYNC.COLLECTIVE" in ins[i - 1][1])]
        back = []
        for a, t in ins:
            m = re.search(r"\bBRA(?:\.U)?\s+(?:!?U?P\w+,\s*)?0x([0-9a-f]+)", t)
            if m and int(m.group(1), 16) < a:
                back.append((a, int(m.group(1), 16)))
        loops = []
        for v in votes:
            enc = [(b - t, t, b) for b, t in back if t <= v <= b]
            if enc:
                _, t, b = min(enc)
                body = [x for a, x in ins if t <= a <= b]
                loops.append(dict(instructions=len(body), ldl=sum("LDL" in x for x in body), stl=sum("STL" in x for x in body),
                                  lds=sum(bool(re.match(r"(@!?P\d+ )?LDS\b", x)) for x in body)))
        out.append((name, sum("LDL" in x for _a, x in ins), loops))
    return out


def main():
    objs = sys.argv[1:] or sorted(glob.glob(os.path.join(ROOT, "qo-100-tools_b200", "lib", "qo_ts2s?.o")))
    for o in objs:
        for name, ldl, loops in screen_loops(o):
            print("%s: %d LDL in the kernel; %d screen loops, %d-%d instructions, LDL %d, STL %d, LDS %d-%d" % (
                name, ldl, len(loops), min(l["instructions"] for l in loops), max(l["instructions"] for l in loops),
                sum(l["ldl"] for l in loops), sum(l["stl"] for l in loops), min(l["lds"] for l in loops), max(l["lds"] for l in loops)))


if __name__ == "__main__":
    main()
