#!/usr/bin/env python
"""Wide device likelihood plugins on the GPU, measured in one call:
 (a) built-in wide Rosenbrock1 against the restated wide-Rosenbrock plugin (the same wide kernel template), d = 16
     and 64, 2^20 chains, PLOCAL 0.9, sum-mixture remote mode, pool M = 16: ms per exchange window (sync = 10 steps),
     the two engines' windows alternated after a warm-up, state resident on the device;
 (b) the wide logistic-regression plugin (examples/likelihoods/logistic_wide.cuh, d = 32, 64 data rows) against the
     same model on the host-callback path (mcgpu_step_propose / numpy / mcgpu_step_accept): chain-steps per second.
The card's name and power limit are read in the same call.

  python tools/plugin_wide_rate.py --out profiles/r04_plugin_wide_rate.json
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from mcpar_b200 import engine, plugin   # noqa: E402
from conftest import tiled_pinit        # noqa: E402
from plugin_rate import card, timed     # noqa: E402
from test_gpu_plugin_wide import logistic_wide_data, logistic_wide_np   # noqa: E402


def compare_rosenbrock(d, N, windows, reps):
    sync = 10
    kw = dict(pool_m=16, pl=0.9, coin_group=0, sync=sync, remote_mode=1, history_steps=0)
    pin = tiled_pinit(N, d)
    arms = {"builtin": engine.Engine(d, N, **kw), "plugin": engine.Engine(d, N, **kw)}
    arms["builtin"].set_likelihood("rosenbrock1")
    arms["plugin"].set_likelihood("plugin", plugin=plugin.shipped("rosen1_wide_d%d.cubin" % d))
    total = (reps + 1) * windows * sync
    for e in arms.values():
        e.set_covariance(None); e.set_state(pin); e.burnin(100); e.sample_begin(total)
        e.sample(windows * sync); e.synchronize()                     # warm-up: every phase and shape of the timed windows
    ms = {k: [] for k in arms}
    for _ in range(reps):
        for k, e in arms.items():                                     # A/B alternated
            ms[k].append(1e3 * timed(lambda: (e.sample(windows * sync), e.synchronize())) / windows)
    same = np.array_equal(arms["builtin"].state()["p"], arms["plugin"].state()["p"])
    for e in arms.values():
        e.close()
    med = {k: statistics.median(v) for k, v in ms.items()}
    return {"chains": N, "d": d, "pl": 0.9, "remote_mode": "summix", "pool_m": 16, "sync": sync,
            "windows_per_sample": windows, "reps": reps, "final_states_equal": bool(same),
            "plugin_over_builtin_median": med["plugin"] / med["builtin"],
            **{k: {"ms_per_window_median": med[k], "min": min(v), "max": max(v), "all": v} for k, v in ms.items()}}


def compare_logistic(N, steps_dev, steps_host):
    par, X, y, prec = logistic_wide_data()
    d = 32
    kw = dict(pool_m=16, pl=0.9, coin_group=0, remote_mode=1, history_steps=0)
    pin = tiled_pinit(N, d) * 0.25
    f = lambda x: logistic_wide_np(x, X, y, prec)                     # noqa: E731
    g = engine.Engine(d, N, **kw)
    g.set_likelihood("plugin", par, plugin=plugin.shipped("logistic_wide.cubin"))
    g.set_covariance(None); g.set_state(pin); g.burnin(20); g.sample_begin(2 * steps_dev)
    g.sample(steps_dev); g.synchronize()                              # warm-up
    t_dev = timed(lambda: (g.sample(steps_dev), g.synchronize()))
    g.close()
    h = engine.Engine(d, N, **kw)
    h.set_likelihood("host"); h.set_covariance(None); h.set_state_host(pin, f(pin))
    pt = np.empty((N, d))
    h.sample_begin(steps_host + 2)
    for _ in range(2):                                                # warm-up
        h.step_propose(pt); h.step_accept(f(pt))

    def host_steps():
        for _ in range(steps_host):
            h.step_propose(pt); h.step_accept(f(pt))
        h.synchronize()
    t_host = timed(host_steps)
    h.close()
    return {"chains": N, "d": d, "data_rows": int(par[0]), "pl": 0.9, "remote_mode": "summix", "pool_m": 16,
            "plugin": {"steps": steps_dev, "s": t_dev, "chain_steps_per_s": N * steps_dev / t_dev},
            "host_callback": {"steps": steps_host, "s": t_host, "chain_steps_per_s": N * steps_host / t_host,
                              "host_eval": "numpy on the calling thread"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--chains", type=int, default=1 << 20)
    ap.add_argument("--windows", type=int, default=10)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    res = {"card": card(),
           "rosenbrock_builtin_vs_plugin": [compare_rosenbrock(d, a.chains, a.windows, a.reps) for d in (16, 64)],
           "logistic_wide_plugin_vs_host": compare_logistic(a.chains, 100, 5)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
