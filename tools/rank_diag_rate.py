#!/usr/bin/env python
"""Time mcgpu_history_rank_diag at 2^20 chains and n = 100 kept steps: the median of 10 calls after one warm-up call
(host clock around calls that end in a device synchronise), for DualGaussian d = 2 and Rosenbrock1 d = 16 (the wide
kernel).  Beside them: a torch.profiler split of one d = 2 call into the sorts, the rank transform, the partials
reduction and the tail-threshold select, and once at d = 2 the host path (history() to the host plus the numpy port
of tests/rank_ref.py).  Writes one JSON file with the card's name and power limit read in the same run.

    python tools/rank_diag_rate.py [--out profiles/r08_rank_diag_rate.json] [--chains 1048576]
"""
import argparse
import collections
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from mcpar_b200 import engine  # noqa: E402
import rank_ref  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(fn, reps=10):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return statistics.median(ts) * 1e3, min(ts) * 1e3


def workload(name, C, n):
    if name == "dgauss":
        d, lik, par, kw = 2, "dualgaussian", [5.0], dict(pool_m=16)
        box = ([-3.0] * 2, [3.0] * 2)
    else:
        d, lik, par, kw = 16, "rosenbrock1", None, dict(pool_m=16, coin_group=0)
        box = ([-2.0] * 16, [2.0] * 16)
    e = engine.Engine(d, C, history_steps=n, **kw)
    e.set_likelihood(lik, par); e.set_covariance(None); e.set_state_sobol(*box)
    e.burnin(100); e.sample_begin(n); e.sample(n); e.synchronize()
    return e, d


def part_of(kernel):
    if "DeviceRadixSort" in kernel:
        return "sort"
    if "DeviceScan" in kernel or "rank_" in kernel:
        return "transform"
    if "diag_radix" in kernel:
        return "tail_threshold_select"
    if "diag_" in kernel:
        return "reduction"
    return "other"


def profile_split(e, L):
    """Device time per part of one call (torch.profiler, CUDA activities), in ms."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        e.rank_diagnostics(L)
        torch.cuda.synchronize()
    parts, launches = collections.Counter(), collections.Counter()
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ev.device_time_total > 0:
            p = part_of(ev.name)
            parts[p] += ev.device_time_total / 1e3
            launches[p] += 1
    return {p: {"device_ms": round(parts[p], 3), "kernels": launches[p]} for p in sorted(parts)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_rank_diag_rate.json"))
    ap.add_argument("--chains", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=100)
    a = ap.parse_args()
    if engine.device_count() < 1:
        sys.exit("rank_diag_rate: no CUDA device (nothing is timed without one)")
    C, n = a.chains, a.steps
    N = n // 2; L = max(1, N - 2)
    out = {"card": card(), "chains": C, "kept_steps": n, "max_lag": L, "repetitions": 10,
           "timing": "median (and min) of 10 calls after one warm-up call; host clock around calls that synchronise",
           "workloads": {}}
    for name in ("dgauss", "rosen16"):
        e, d = workload(name, C, n)
        ncol = d + 1
        w = {"d": d, "split_draws_per_column": 2 * C * N, "history_bytes": C * n * ncol * 8}
        l0 = e.stats()["kernel_launches"]
        rep = e.rank_diagnostics(L)
        w["launches_per_call"] = e.stats()["kernel_launches"] - l0
        w["rank_diag_ms"], w["rank_diag_min_ms"] = timed(lambda: e.rank_diagnostics(L))
        w["rank_diag_ms_per_column"] = w["rank_diag_ms"] / ncol
        w["report"] = {k: rep[k].tolist() for k in rank_ref.FIELDS}
        if name == "dgauss":
            w["profile_one_call"] = profile_split(e, L)
            t0 = time.perf_counter(); rows = e.history(); w["history_to_host_ms"] = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter(); ref = rank_ref.report(rows); w["numpy_port_ms"] = (time.perf_counter() - t0) * 1e3
            w["host_path_ms"] = w["history_to_host_ms"] + w["numpy_port_ms"]
            w["device_equals_port_rtol_1e-10"] = bool(all(
                np.allclose(rep[k], ref[k], rtol=1e-10, atol=0, equal_nan=True) for k in rank_ref.FIELDS))
            del rows
        e.close()
        out["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", a.out, "on", out["card"])


if __name__ == "__main__":
    main()
