#!/usr/bin/env python3
"""cuobjdump -sass of the built library -> opcode counts per kernel (the evidence file under profiles/).
usage: python tools/sass_evidence.py > profiles/rNN_sass_evidence.txt"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "kinectdepthmapenhancement_b200", "libkdme_b200.so")
WANT = ("UTMALDG", "SYNCS", "VABSDIFF4", "IDP.4A", "MUFU.EX2", "MUFU.RCP", "FFMA2", "FADD2", "LDS.128", "DFMA", "DADD",
        "ACQBULK", "UTMAPF", "ATOMG", "RED")
KERNELS = re.compile(r"jbf_fast_kernelILi(2|7|9|15)ELi64ELi(16|8)E|jbf_refine_kernelILi8E|jbf_upsample_gather|presmooth5|guided_fill_kernelILi7E")


def main():
    out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
    counts = collections.OrderedDict()
    cur = None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1) if KERNELS.search(m.group(1)) else None
            continue
        if cur is None:
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
        if m:
            op = m.group(1)
            for w in WANT:
                if op.startswith(w):
                    key = w if w in ("UTMALDG", "SYNCS", "ATOMG", "RED") else op
                    counts.setdefault(cur, collections.Counter())[key] += 1
                    break
    print("# cuobjdump -sass libkdme_b200.so: instruction counts per kernel (count, mangled kernel, SASS opcode)")
    print("# UTMALDG = cp.async.bulk.tensor (TMA tile+halo staging); SYNCS = mbarrier; VABSDIFF4 / IDP.4A / MUFU.EX2 = one each")
    print("# per tap per pass; FFMA2/FADD2 = packed fp32x2 math (taps and the 2Sum row combinations); DFMA/DADD only in the fp64")
    print("# refinement kernel; template arguments of jbf_fast_kernel: <radius, tile width, tile height, min CTAs/SM>")
    for k, c in counts.items():
        for op, n in sorted(c.items()):
            print(n, k, op)


if __name__ == "__main__":
    main()
