#!/usr/bin/env python
"""Collect the outputs of tools/gpu_r06.sh OUTDIR into one JSON document (profiles/r06_ab_timing.json):
    python tools/r06_summary.py OUTDIR > profiles/r06_ab_timing.json"""
import json
import os
import statistics
import sys

out = sys.argv[1]


def last_json(path):
    try:
        lines = [l for l in open(path) if l.strip().startswith("{")]
        return json.loads(lines[-1]) if lines else None
    except OSError:
        return None


smi = open(os.path.join(out, "r06_smi.txt")).read().splitlines()
doc = {"_command": "bash tools/gpu_r06.sh OUTDIR (one run on one GPU; old = libmcgpu.so of the parent commit via MCGPU_LIB, "
                   "new = this tree's build; each configuration: python bench.py --no-cpu --no-e2e --no-modes --steps 300 "
                   "[args], old and new alternately, three runs each)",
       "_card": smi[-1] if smi else "unknown"}
for tag, args in [("default", ""), ("rosen2d", "--workload rosen2d"), ("summix", "--remote-mode summix"),
                  ("pool64", "--pool 64"), ("pool256", "--pool 256")]:
    e = {"args": args}
    for side in ("old", "new"):
        runs = [last_json(os.path.join(out, "r06_%s_%s_%d.json" % (tag, side, i))) for i in (1, 2, 3)]
        runs = [r for r in runs if r]
        e[side] = {"ms_per_window": [r["ms_per_step"] for r in runs], "value": [r["value"] for r in runs],
                   "remote_iterations_mean": sorted({r.get("remote_iterations_mean") for r in runs}, key=str),
                   "exact_fallback_rate": sorted({r.get("exact_fallback_rate") for r in runs}, key=str)}
    if e["old"]["ms_per_window"] and e["new"]["ms_per_window"]:
        e["new_over_old_ms"] = round(statistics.median(e["new"]["ms_per_window"]) / statistics.median(e["old"]["ms_per_window"]), 4)
    doc[tag] = e
doc["hit_rates_default_line"] = {}
for g in (32, 64, 128):
    doc["hit_rates_default_line"]["G%d" % g] = last_json(os.path.join(out, "r06_hits_g%d.json" % g))
doc["dump_outputs_default_line"] = open(os.path.join(out, "r06_dump_cmp.txt")).read().strip().splitlines()[-1]
print(json.dumps(doc, indent=1))
