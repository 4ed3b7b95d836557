#!/usr/bin/env python
"""Hit rates of the d = 2 table of acceptance-ratio bounds, from a counting build (the product build has no counters):
    python tools/build_variant.py cnt64 -DMCGPU_CELL_COUNT -DMCGPU_CELL_G=64
    python tools/cell_hits.py mcpar_b200/variants/libmcgpu_cnt64.so [bench.py arguments]
runs bench.py in this process on that library, then prints one JSON line: remote candidates the table decided,
candidate rounds of a warp in which at least one lane missed the table (and so ran the pool loop), and all rounds,
summed over the whole run (warm-up and timed windows)."""
import ctypes
import json
import os
import runpy
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib = os.path.abspath(sys.argv[1])
os.environ["MCGPU_LIB"] = lib
sys.path.insert(0, ROOT)
sys.argv = [os.path.join(ROOT, "bench.py")] + sys.argv[2:]
try:
    runpy.run_path(sys.argv[0], run_name="__main__")
except SystemExit:
    pass
c = (ctypes.c_ulonglong * 4)()
assert ctypes.CDLL(lib).mcgpu_cell_counts(c) == 0
decided, miss_rounds, rounds = c[0], c[1], c[2]
print(json.dumps({"lib": os.path.basename(lib), "table_decided_share": decided / max(1, 32 * rounds),
                  "miss_free_round_share": 1.0 - miss_rounds / max(1, rounds), "rounds": rounds,
                  "table_decided": decided, "rounds_with_miss": miss_rounds}))
