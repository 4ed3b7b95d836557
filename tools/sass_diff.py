#!/usr/bin/env python
"""Compare two cuobjdump -sass dumps kernel by kernel (instructions and encodings, whitespace ignored): prints how
many kernels are identical and names the ones that differ.    python tools/sass_diff.py old.sass new.sass"""
import collections
import re
import sys


def kernels(path):
    d = collections.OrderedDict(); cur = None
    for line in open(path):
        m = re.search(r"Function : (\S+)", line)
        if m: cur = m.group(1); d[cur] = []; continue
        t = " ".join(line.split())
        if cur and t: d[cur].append(t)
    return d


old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
differ = [k for k in old if old[k] != new.get(k)]
print("identical: %d  differ: %d  only old: %d  only new: %d" % (len(old) - len(differ), len(differ),
      len([k for k in old if k not in new]), len([k for k in new if k not in old])))
for k in differ: print("  differs", k)
