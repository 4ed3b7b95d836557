#!/usr/bin/env python
"""Time the history diagnostics at 2^20 chains and n = 100 kept steps: mcgpu_history_diag_partials, mcgpu_diag_finalize
and mcgpu_history_quantiles (3 probabilities), each as the median of 10 calls after one warm-up call (host clock around
calls that end in a device synchronise), for DualGaussian d = 2 and Rosenbrock1 d = 16 (the wide kernel).  Beside them,
once: history() to the host, and for d = 2 the numpy reference (tests/diag_ref.py partials + finalize, np.quantile)
on those rows.  Writes one JSON file with the card's name and power limit read in the same run.

    python tools/diag_rate.py [--out profiles/r07_diag_rate.json] [--chains 1048576]
"""
import argparse
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
import diag_ref  # noqa: E402

PROBS = (0.05, 0.5, 0.95)


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_diag_rate.json"))
    ap.add_argument("--chains", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=100)
    a = ap.parse_args()
    if engine.device_count() < 1:
        sys.exit("diag_rate: no CUDA device (nothing is timed without one)")
    C, n = a.chains, a.steps
    N = n // 2; L = max(1, N - 2)
    out = {"card": card(), "chains": C, "kept_steps": n, "max_lag": L, "probs": PROBS, "repetitions": 10,
           "timing": "median (and min) of 10 calls after one warm-up call; host clock around calls that synchronise",
           "workloads": {}}
    for name in ("dgauss", "rosen16"):
        e, d = workload(name, C, n)
        ncol = d + 1
        blk = e.diag_partials(1, L)
        w = {"d": d, "history_bytes": C * n * ncol * 8,
             "lag_dfma": ncol * 2 * C * N * (L + 1)}                 # ncol M' N (L + 1): a bound on the lag products
        w["partials_ms"], w["partials_min_ms"] = timed(lambda: e.diag_partials(1, L))
        w["finalize_ms"], w["finalize_min_ms"] = timed(lambda: engine.diag_finalize([blk]))
        w["quantiles3_ms"], w["quantiles3_min_ms"] = timed(lambda: e.quantiles(PROBS))
        w["partials_history_GBps"] = w["history_bytes"] / w["partials_ms"] * 1e-6
        w["quantile_history_GBps_per_pass"] = 8 * w["history_bytes"] / w["quantiles3_ms"] * 1e-6   # 8 radix passes
        t0 = time.perf_counter(); rows = e.history(); w["history_to_host_ms"] = (time.perf_counter() - t0) * 1e3
        if name == "dgauss":
            t0 = time.perf_counter()
            ref = engine.diag_finalize([diag_ref.partials(rows, 1, L)])
            qref = [np.quantile(rows[:, :, j].ravel(), PROBS, method="linear") for j in range(ncol)]
            w["numpy_reference_ms"] = (time.perf_counter() - t0) * 1e3
            rep = engine.diag_finalize([blk])
            w["device_equals_reference"] = bool(all(np.allclose(rep[k], ref[k], rtol=1e-10, equal_nan=True) for k in ref)
                                                and np.array_equal(e.quantiles(PROBS), np.array(qref)))
            w["host_path_ms"] = w["history_to_host_ms"] + w["numpy_reference_ms"]
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
