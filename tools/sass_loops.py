#!/usr/bin/env python
"""cuobjdump -sass output (file) -> for each kernel matching a pattern, every loop (backward branch) of at least N
instructions with its static instruction mix: FFMA / FFMA2 / FADD / FMUL / MUFU, the FP64 pipe and fp64 conversions
(DADD DMUL DFMA DSETP, *.F64), LDS / SHFL / integer / constant loads / special registers.  tools/sass_loop.py keeps to
the step loop; this one also shows the loops inside it (the remote candidate round and its 8-slot pool chunk).
    python tools/sass_loops.py fast.sass 'mh_steps_kernelILi3ELi2ELi0ELi1E' [N=40]"""
import collections
import re
import sys

pat = re.compile(sys.argv[2]) if len(sys.argv) > 2 else re.compile(".")
minn = int(sys.argv[3]) if len(sys.argv) > 3 else 40
funcs = collections.OrderedDict(); cur = None
for line in open(sys.argv[1]):
    m = re.search(r"Function : (\S+)", line)
    if m: cur = m.group(1); funcs[cur] = []; continue
    m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
    if m and cur: funcs[cur].append((int(m.group(1), 16), m.group(2).strip()))
op = lambda t: re.sub(r"^@!?U?P\w+\s+", "", t).split()[0]
KEYS = ["FFMA", "FFMA2", "FADD", "FMUL", "MUFU", "LDS", "SHFL", "IMAD", "LOP3", "LDC", "LDCU", "S2R", "S2UR", "POPC", "BRA"]
for name, ins in funcs.items():
    if not pat.search(name): continue
    print(name)
    for addr, text in ins:
        m = re.search(r"BRA\S*\s+(?:!?U?P\d,\s*)?0x([0-9a-f]+)", text)
        if not m or int(m.group(1), 16) >= addr: continue
        tgt = int(m.group(1), 16)
        body = [t for a, t in ins if tgt <= a <= addr]
        if len(body) < minn: continue
        c = collections.Counter(op(t).split(".")[0] for t in body)
        f64 = sum(1 for t in body if re.match(r"(DADD|DMUL|DFMA|DSETP)", op(t)) or "F64" in op(t))
        print("  0x%05x-0x%05x %4d instr  fp64 %d  " % (tgt, addr, len(body), f64) + " ".join("%s %d" % (k, c[k]) for k in KEYS if c[k]))
