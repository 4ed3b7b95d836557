#!/usr/bin/env python
"""bench.py -- MH chain-steps/s of the B200 engine (and of the reference on the host cores).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload dgauss|rosen2d|rosen16|gmix64]
                  [--remote-mode reference|summix] [--pool M] [--lag 0|1] [--dump-outputs DIR]
  python bench.py --impl reference ...        # the reference's own CPU loop (oracle/_ref)

A "step" is one exchange window of the hot path: `sync` (=10) Metropolis-Hastings steps of every chain
(proposal, likelihood, accept, update, running moments), the thinned sample-history store, the publication
of the exchange pool and the exchange itself (in-kernel peer-to-peer stores over NVLink, or an NCCL
all-gather).  Workload at N=1 is BASELINE.json configs[1] (mcpar-dgauss: DualGaussian(5), 2^20 chains, one
B200); SURVEY.md 8(d) fixes the rest (identity incov, PLOCAL 0.9, SYNCSTEP 10, thin 10).  Weak scaling:
2^20 chains per GPU.

What the line holds (contract: the task's bench section):
  value / ms_per_step   K timed windows, state resident, CUDA events on the launching stream, max over ranks.
                        Before the timed region the sampler is advanced `--advance` untimed windows so that
                        the rejection loop of the reference's remote proposal sits at its plateau (its
                        iteration count rises for ~2000 windows), and the region is placed (at most 200 windows
                        later) where its share of remote steps is closest to 1 - PLOCAL -- the job-wide coins are
                        counter-based and evaluated on the host (place_timed_region): the value does not depend
                        on K (20 / 50 / 1000 windows agree to 0.3 %, profiles/r02_steps_independence.md).
  remote mode           `reference` (default): the reference's max-mixture rejection loop over a pool of M
                        components; `summix`: the normalised sum-mixture proposal (no rejection loop).  The
                        headline is the default mode; "modes" holds short measurements of the other
                        configurations (sum-mixture at M = 16 and at the blueprint's M = 256).
  e2e                   a whole MCPar::run-shaped job through the C ABI with HOST buffers: host pinit in,
                        burn-in 500, 1000 steps, rows (thin 10) drained to a pinned host sink of the
                        reference MCout's element type (float) while the next window computes, final logL out.
  roofline              FP64 pipe: flops per chain-step counted by ncu (profiles/fp64_work.json) x chain-steps/s
                        over the DFMA peak measured in this run.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # a benchmark run leaves the tree as it found it (it may be read-only)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "mh_chain_steps_per_sec"
UNIT = "chain-steps/s"
SEED = 8675309                      # reference seed, src/mcpar.cc:271

# SURVEY.md 8(d) a-priori estimates of the hardware-equivalent fp64 flops per chain-step (used only until
# profiles/fp64_work.json holds the figure ncu counted for the workload) and textbook flops
WORKLOADS = {
    "dgauss":  dict(lik="dualgaussian", par=[5.0], d=2, F_hw=280.0, F_alg=46.0, name="mcpar-dgauss", advance=3000),
    "rosen2d": dict(lik="rosenbrock1", par=None, d=2, F_hw=167.0, F_alg=38.0, name="mcpar-rosen1 shape, 2-D Rosenbrock", advance=3000),
    "rosen16": dict(lik="rosenbrock1", par=None, d=16, F_hw=1350.0, F_alg=516.0, name="mcpar-rosen2 (d=16)", advance=300),
    # SURVEY.md 8(d) C4: GaussMix d=64, K=64, exchange every sweep (SYNCSTEP 1), diagonal incov
    "gmix64":  dict(lik="gaussmix", par="gmix64", d=64, F_hw=22600.0, F_alg=17500.0, name="sum-of-Gaussians mixture d=64 K=64",
                    sync=1, thin=100, advance=200),
}
RMODE = {"reference": 0, "summix": 1}


def gmix64_params(seed=SEED):
    """mu_ki = 10 (u - 0.5), sig2_ki = 0.5 + 1.5 u', w_k = 1 (SURVEY.md 8d C4; numpy Philox stream of the seed)."""
    import numpy as np
    rng = np.random.Generator(np.random.Philox(seed))
    K, d = 64, 64
    mu = 10.0 * (rng.random((K, d)) - 0.5)
    s2 = 0.5 + 1.5 * rng.random((K, d))
    return K, d, mu, s2, np.ones(K)


def incov_for(wl):
    import numpy as np
    if wl == "gmix64":              # C4: diagonal (2.38^2/64) I
        return np.eye(64) * (2.38 ** 2 / 64)
    if wl == "rosen16":             # SURVEY.md 8(d) C3: analytic target covariance, Roberts-Rosenthal scale
        blk = (2.38 ** 2 / 16) * np.array([[0.5, 1.0], [1.0, 2.505]])
        return np.kron(np.eye(8), blk)
    return None


def remote_plan(seed, d, nburn, nsteps, pl, first_remote_t):
    """The job-wide local/remote coin of main steps 0..nsteps-1, evaluated on the host exactly as the engine does
    (mcgpu_api.cu host_coin: word 2*NP+1 of chain 0's local Philox4x32-10 stream at step nburn + t; remote iff
    t >= first_remote_t and not coin <= pl, mcpar.cc:142-152).  Returns a list of 0/1."""
    M0, M1, W0, W1, MASK = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85, 0xFFFFFFFF
    idx = 2 * ((d + 1) // 2) + 1
    out = []
    for t in range(nsteps):
        c = [0, 0, (nburn + t) & MASK, idx // 4]
        k0, k1 = seed & MASK, (seed >> 32) & MASK
        for _ in range(10):
            p0, p1 = M0 * c[0], M1 * c[2]
            c = [((p1 >> 32) ^ c[1] ^ k0) & MASK, p1 & MASK, ((p0 >> 32) ^ c[3] ^ k1) & MASK, p0 & MASK]
            k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
        coin = c[idx % 4] / 4294967296.0
        out.append(1 if (t >= first_remote_t and not coin <= pl) else 0)
    return out


def place_timed_region(seed, d, nburn, sync, lag, pl, advance, warmup, K, slack=200):
    """Where to start the K timed windows.  With one coin per step for the whole job the share of remote steps inside a
    short timed region is a draw (K = 20 windows hold 200 coins: 20 +- 4 remote steps), and a remote step costs many
    local ones, so `value` would depend on K.  The coins are counter-based and known in advance: the region is moved
    forward by at most `slack` windows to where its remote share is closest to the long-run 1 - pl.  Returns
    (advance, remote share of the timed region)."""
    if pl >= 1.0 or K * sync > 200000:
        return advance, 0.0 if pl >= 1.0 else None
    plan = remote_plan(seed, d, nburn, (advance + slack + warmup + K) * sync, pl, sync * (1 + lag))
    cum = [0]
    for b in plan:
        cum.append(cum[-1] + b)
    best, best_err = advance, None
    for a in range(advance, advance + slack + 1):
        lo = (a + warmup) * sync
        share = (cum[lo + K * sync] - cum[lo]) / float(K * sync)
        err = abs(share - (1.0 - pl))
        if best_err is None or err < best_err - 1e-12:
            best, best_err, best_share = a, err, share
    return best, best_share


class ClockSampler:
    """SM clock and throttle reasons of ONE GPU sampled during the run by an NVML polling thread (every rank
    runs its own, started before the warm-up, so no rank enters the timed loop late)."""

    def __init__(self, index, period=0.01):
        self.samples, self.reasons, self.stop_flag, self.mx = [], set(), False, None
        self.t_mark = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:                                   # the CUDA ordinal need not be the NVML index: go by PCI address
                import torch
                pr = torch.cuda.get_device_properties(index)
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(("%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return
        self.period = period
        self.th = threading.Thread(target=self._loop, daemon=True)
        self.th.start()

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = int(get_reasons(self.h))
                self.samples.append((time.perf_counter(), mhz))
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def mark(self):
        """samples from here on were taken under load (pre-advance + timed region)"""
        self.t_mark = time.perf_counter()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": [], "samples": 0}
        if self.nv is None:
            return out
        self.stop_flag = True
        self.th.join(timeout=2)
        sm = [m for t, m in self.samples if self.t_mark is None or t >= self.t_mark]
        if sm:
            out.update(sm_mhz=statistics.median(sm), reasons=sorted(self.reasons), samples=len(sm),
                       how="NVML polled every %g ms by every rank from before the warm-up; median over the advance + timed region" % (1e3 * self.period))
        return out


def pin_to_gpu_numa(local):
    """Run this rank's host threads (and first-touch its pinned buffers) on the NUMA node of its GPU."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        dev = torch.cuda.get_device_properties(local).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/" % (dom, bus, dev)
        node = int(open(path + "numa_node").read().strip())
        cpus = open(path + "local_cpulist").read().strip()
        ids = []
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids += list(range(int(a), int(b or a) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
        return {"numa_node": node, "cpus": len(ids)}
    except Exception as ex:          # noqa: BLE001  (not fatal: the buffers are then wherever the kernel puts them)
        return {"numa_node": None, "error": str(ex)[:80]}


def cpu_reference_run(wl, nranks, nchain, nburn, nsamp, pl=0.9, bits=64):
    """Time the reference's own MCPar::run (oracle/_ref: its unmodified sources on shim
    MPI/MKL, thread ranks) on the host cores.  Returns chain-steps/s."""
    from oracle.ref import Ref, available
    from conftest import tiled_pinit
    if not available(bits):
        return None
    W = WORKLOADS[wl]
    ref = Ref(bits)
    pin = tiled_pinit(nchain, W["d"])
    o = ref.run(W["lik"], W["d"], nchain, nranks, nsamp, nburn, pin, incov=incov_for(wl), par=W["par"],
                seed=SEED, pl=pl, want_rows=False, want_maxl=False)
    return nranks * nchain * (nburn + nsamp) / o["seconds"]


def cpu_baseline_port(wl):
    """Workloads the reference cannot run (GaussMix is not one of its likelihoods): the
    oracle's plain-C restatement of the same normal-mode algorithm, one thread."""
    import numpy as np
    from oracle import mh
    K, d, gmu, gs2, gw = gmix64_params()
    N, nburn, nsamp = 128, 100, 100
    par = np.concatenate([[float(K)], gmu.ravel(), gs2.ravel(), gw])
    t0 = time.time()
    mh.run_counter("gaussmix", d, N, nsamp, nburn, gmu[np.arange(N) % K], incov=incov_for(wl), par=par,
                   seed=SEED, coin_group=0, pool_m=16, sync=1, thin=100, want_rows=False)
    sec = time.time() - t0
    return {"value": N * (nburn + nsamp) / sec, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "oracle/mh_oracle.c (orc_run_counter), %d chains x %d steps, pool M=16, one thread" % (N, nburn + nsamp),
            "seconds": round(sec, 1)}


def cpu_baseline(wl):
    """Bounded sample of the same workload on all host cores: the reference's own launch
    shape (one rank per core, 4 chains per rank as in mcpar-dgauss.cc:31)."""
    if WORKLOADS[wl]["lik"] == "gaussmix":
        return cpu_baseline_port(wl)
    cores = os.cpu_count() or 1
    R = min(cores, 64)              # remote proposals cost O(N^2) in the reference: bound the rank count
    t0 = time.time()
    v = cpu_reference_run(wl, R, 4, 500, 1000)
    if v is None:
        return {"value": None, "unit": UNIT, "cores": R, "kind": "reference", "sample": "oracle/_ref not built"}
    v_local = cpu_reference_run(wl, R, 4, 500, 20000, pl=1.0)
    return {"value": v, "unit": UNIT, "cores": R, "kind": "reference",
            "sample": "reference MCPar::run (own sources, shim RNG/MPI, fp64 build), %d thread-ranks x 4 chains, "
                      "nburn 500 + nsamp 1000, PLOCAL 0.9 (all-pairs remote proposals over %d chains)" % (R, 4 * R),
            "value_local_only": v_local,
            "sample_local_only": "same, PLOCAL 1.0, nsamp 20000", "host_cores": cores,
            "seconds": round(time.time() - t0, 1)}


def run_reference_arm(args):
    """The reference's own CPU implementation of the path (oracle/_ref: its unmodified sources on
    shim MPI/MKL, fp64 build) on the host cores.  MCPar::run cannot be resumed, so the K timed
    "steps" (10-step windows) and the W warm-up windows are ONE call
    run(nsamp = (W+K)*10, nburn = 500) on R thread-ranks x 4 chains; the clock is the harness's
    steady_clock around MCPar::run.  Bounded: 64 chains, so K = 1000 takes about a second."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    if WORKLOADS[wl]["lik"] == "gaussmix":
        print(json.dumps({"impl": "reference", "unavailable": "the reference has no Gaussian-mixture likelihood (only the 2-D DualGaussian)"}))
        return
    cores = os.cpu_count() or 1
    R = min(cores, 64)
    nburn, sync = 500, 10
    nsamp = (args.warmup + args.steps) * sync
    t0 = time.time()
    v = cpu_reference_run(wl, R, 4, nburn, nsamp)
    if v is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref is not built on this box"}))
        return
    secs = R * 4 * (nburn + nsamp) / v
    sample = ("one reference MCPar::run (own unmodified sources, shim RNG/MPI, fp64 build): %d thread-ranks x 4 chains, "
              "nburn %d + nsamp %d (= %d windows of %d steps), PLOCAL 0.9, all-pairs remote proposals over %d chains"
              % (R, nburn, nsamp, args.warmup + args.steps, sync, 4 * R))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / (nburn / sync + args.warmup + args.steps),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": WORKLOADS[wl]["name"], "sample": sample},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": R, "kind": "reference", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": round(time.time() - t0, 2)}
    print(json.dumps(line))


class Job:
    """One sharded (or single) engine of the job on this rank, with its exchange wiring."""

    def __init__(self, ctx, Cg, rmode, M, ring, lag=None, chains_total=None, ranks=None):
        import numpy as np
        from mcpar_b200 import engine
        from mcpar_b200.sharded import ShardedRunner, DistGroup
        a, W = ctx["args"], ctx["W"]
        self.ctx, self.Cg = ctx, Cg
        self.world = ctx["world"] if ranks is None else ranks          # ranks that take part (the first `ranks` of the job)
        self.rank = ctx["rank"]
        self.active = self.rank < self.world
        self.N = Cg * self.world if chains_total is None else chains_total
        self.sync, self.thin = a.sync, a.thin
        lag = a.lag if lag is None else lag
        self.e = None
        if not self.active:
            return
        self.e = engine.Engine(W["d"], Cg, mode="normal", nchain_total=self.N, chain0=self.rank * Cg, pl=a.pl, sync=a.sync,
                               seed=SEED, pool_m=(M if 0 < M < self.N else 0), thin=a.thin, coin_group=a.coin_group,
                               history_steps=ring, device=ctx["local"], remote_mode=rmode, pool_lag=lag)
        self.e.set_stream(ctx["stream"].cuda_stream)                   # engine kernels, NCCL ops and timing events share it
        self.e.set_likelihood(W["lik"], W["par"]); self.e.set_covariance(incov_for(a.workload))
        self.runner = None
        if self.world > 1:
            import torch
            dist = ctx["dist"]
            grp = ctx["groups"].get(self.world)
            as_tensor = lambda ptr: torch.as_tensor(ptr, device=ctx["dev"])
            self.runner = ShardedRunner(self.e, DistGroup(dist, grp), as_tensor)
            if a.exchange == "p2p":
                def gather_bytes(b, grp=grp, n=self.world):
                    out = [None] * n
                    dist.all_gather_object(out, b, group=grp)
                    return out
                self.runner.enable_p2p(self.rank, self.world, gather_bytes)

    def pinit(self):
        """this rank's rows of the job's initial points: the reference mains' four points tiled by GLOBAL chain id
        (conftest.tiled_pinit: chain g starts at P[g mod 4]); GaussMix: chain g at mu_{g mod K}"""
        import numpy as np
        from conftest import tiled_pinit
        W = self.ctx["W"]
        g0 = self.rank * self.Cg                                       # a multiple of 4 and of K
        if "pinit" in W:
            return np.ascontiguousarray(W["pinit"](np.arange(g0, g0 + self.Cg)))
        assert g0 % 4 == 0
        return tiled_pinit(self.Cg, W["d"])

    def burn(self, n):
        if self.runner is None:
            self.e.burnin(n)
        else:
            self.runner.burnin(n)

    def window(self):
        if self.runner is None:
            self.e.sample(self.sync)
        else:
            self.runner.window(self.sync)

    def barrier(self):
        if self.world > 1:
            self.ctx["dist"].barrier(group=self.ctx["groups"].get(self.world))

    def close(self):
        if self.e is not None:
            self.e.synchronize()
            self.barrier()                                             # peers may still map this engine's exchange region
            self.e.close()
            self.e = None


def timed_windows(ctx, job, K, flush):
    """K windows, one CUDA-event pair each on the launching stream, the L2 flushed between them (outside the
    pairs).  Returns (ms max over ranks, per-rank ms list, stats delta)."""
    import torch
    stream, dist = ctx["stream"], ctx["dist"]
    torch.cuda.synchronize()
    s0 = job.e.stats()
    job.barrier()
    torch.cuda.synchronize()
    evs = []
    for _ in range(K):
        if flush is not None:
            flush.zero_()                                              # L2 flush, outside the event pair
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(stream); job.window(); b.record(stream)
        evs.append((a, b))
    torch.cuda.synchronize()
    job.barrier()
    ms = sum(a.elapsed_time(b) for a, b in evs)
    per_rank = [ms / K]
    if job.world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=ctx["dev"])
        allt = [torch.zeros_like(t) for _ in range(job.world)]
        dist.all_gather(allt, t, group=ctx["groups"].get(job.world))
        per_rank = [float(x.item()) / K for x in allt]
        ms = max(per_rank) * K
    s1 = job.e.stats()
    delta = {k: s1[k] - s0[k] for k in s1 if isinstance(s1[k], int)}
    return ms, per_rank, delta


DUMP_BYTES = 60 * 1000 * 1000       # --dump-outputs: array bytes over every rank (under 64 MB with the .npy headers)
DUMP_SEED = 20260101


def dump_outputs(job, path):
    """Write what the timed path hands its caller after its last window -- the chains' state (p, ly) and running moments
    (mu, sig, psum2), and the newest kept history row (rows: parameters + logL, the MCout element) -- as float64 .npy files.
    Over the byte budget, a fixed seeded sample of chains (the same chains in every run of the same arguments) is kept."""
    import numpy as np
    st = job.e.state()
    kept = job.e.stats()["history_rows"] // job.Cg
    if kept > 0:
        st["rows"] = job.e.history(first=kept - 1, count=1)[0]
    per_chain = sum(a[0].nbytes for a in st.values())
    n = min(job.Cg, DUMP_BYTES // job.world // per_chain)
    idx = slice(None) if n == job.Cg else np.sort(np.random.default_rng(DUMP_SEED).choice(job.Cg, n, replace=False))
    os.makedirs(path, exist_ok=True)
    tag = "" if job.world == 1 else "rank%d_" % job.rank
    for name, a in st.items():
        np.save(os.path.join(path, tag + name + ".npy"), np.ascontiguousarray(a[idx], dtype=np.float64))
    return n


def measure(ctx, Cg, rmode, M, K, advance, warmup, flush, lag=None, ranks=None, clocks=None, dump=None):
    """Resident throughput of one configuration: burn-in 500, `advance` untimed windows, `warmup` untimed
    windows, K timed windows.  Returns a dict (on every active rank)."""
    a = ctx["args"]
    job = Job(ctx, Cg, rmode, M, ring=max(8, 4 * ((a.sync + a.thin - 1) // a.thin)), lag=lag, ranks=ranks)
    if not job.active:
        return None
    job.e.set_state(job.pinit())
    job.burn(500)
    job.e.sample_begin((advance + warmup + K) * a.sync)
    if clocks is not None:
        clocks.mark()                                                  # the GPU is busy from here to the end of the timed region
    for _ in range(advance + warmup):
        job.window()
    ms, per_rank, d = timed_windows(ctx, job, K, flush)
    ck = clocks.stop() if clocks is not None else None
    dumped = dump_outputs(job, dump) if dump else None
    mean, cov = job.e.moments()
    st = job.e.stats()
    out = {"value": job.N * a.sync * K / (ms * 1e-3), "ms_per_step": ms / K, "per_rank_ms_per_step": per_rank,
           "chains_total": job.N, "n_gpus": job.world, "pool_m": M if 0 < M < job.N else job.N,
           "remote_mode": "summix" if rmode else "reference", "lag": a.lag if lag is None else lag, "steps": K, "advance": advance,
           "launches": d["kernel_launches"] + (K if job.world > 1 and a.exchange == "nccl" else 0),
           "remote_fraction": d["remote_steps"] / max(1, d["tried"]),
           "remote_iterations_mean": d["remote_iterations"] / max(1, d["remote_steps"]),
           "exact_fallback_rate": d["exact_fallbacks"] / max(1, d["remote_iterations"]),
           "accept_rate": d["accepted"] / max(1, d["tried"]),
           "exchange_wait_ms_per_step": d["exchange_wait_ns"] * 1e-6 / K, "exchange_waits": d["exchange_waits"],
           "posterior_mean": [float(x) for x in mean[:4]], "posterior_var": [float(cov[i, i]) for i in range(min(4, len(mean)))],
           "clocks": ck, "dumped_chains": dumped}
    job.close()
    return out


def sharded_equals_single(ctx):
    """Untimed check at N > 1: a short sharded run (all ranks, the bench's exchange) against the same run on ONE
    engine hosting every chain (rank 0): final states must be bit-identical."""
    import numpy as np
    import torch
    a, world, rank, dist = ctx["args"], ctx["world"], ctx["rank"], ctx["dist"]
    Cg, M, nburn, nsamp = 1 << 14, 16, 110, 60
    import hashlib
    res = {}
    for rmode in (0, 1):
        job = Job(ctx, Cg, rmode, M, ring=8)
        job.e.set_state(job.pinit())
        job.burn(nburn)
        job.e.sample_begin(nsamp)
        for _ in range(nsamp // a.sync):
            job.window()
        job.e.synchronize()
        st = job.e.state()
        mine = np.concatenate([st["p"].ravel(), st["ly"], st["mu"].ravel(), st["psum2"].ravel()])
        parts = [None] * world
        dist.all_gather_object(parts, mine.tobytes())
        job.close()
        if rank == 0:
            one = Job(ctx, Cg * world, rmode, M, ring=8, ranks=1, chains_total=Cg * world)
            one.e.set_state(one.pinit())
            one.burn(nburn)
            one.e.sample_begin(nsamp); one.e.sample(nsamp); one.e.synchronize()
            s1 = one.e.state()
            one.e.close(); one.e = None
            ok = True
            for r in range(world):
                sl = slice(r * Cg, (r + 1) * Cg)
                ref = np.concatenate([s1["p"][sl].ravel(), s1["ly"][sl], s1["mu"][sl].ravel(), s1["psum2"][sl].ravel()])
                ok = ok and parts[r] == ref.tobytes()
            res["summix" if rmode else "reference"] = bool(ok)
            res["state_sha1_" + ("summix" if rmode else "reference")] = hashlib.sha1(b"".join(parts)).hexdigest()[:16]
        dist.barrier()
    return res


def e2e_job(ctx, Cg, rmode, M, f32, reps):
    """MCPar::run-shaped job through the C ABI with HOST buffers (H2D of pinit, D2H of the rows and the final
    logL inside the clock).  Returns best seconds, construction seconds, bytes."""
    import numpy as np
    import torch
    a, W = ctx["args"], ctx["W"]
    nb_e, ns_e = 500, 1000
    kept_e = (ns_e + a.thin - 1) // a.thin
    d = W["d"]
    sink = torch.empty((kept_e, Cg, d + 1), dtype=torch.float32 if f32 else torch.float64).pin_memory().numpy()
    best, best_c, fin, all_secs = None, None, None, []
    warm = 2                                        # untimed repetitions first: on a fresh box the first jobs pay one-time costs
    for rep in range(warm + reps):                  # (lazy kernel loading, first touch of the pinned sink: 2.3 s and 0.8 s observed)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        job = Job(ctx, Cg, rmode, M, ring=min(kept_e, 16))             # device history: a ring of 16 kept steps
        host_pin = torch.from_numpy(job.pinit()).pin_memory().numpy()
        job.barrier()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        job.e.set_state(host_pin)                                      # H2D inside the timed region
        job.e.attach_host_sink(sink)                                   # D2H drains on a side stream per window
        job.burn(nb_e)
        job.e.sample_begin(ns_e)
        for _ in range(ns_e // a.sync):
            job.window()
        fin = job.e.state()["ly"]
        job.e.synchronize()                                            # compute + drain finished
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        job.close()
        tt = torch.tensor([t2 - t1, t1 - t0], dtype=torch.float64, device=ctx["dev"])
        if ctx["world"] > 1:
            ctx["dist"].all_reduce(tt, op=ctx["dist"].ReduceOp.MAX)
        sec, con = float(tt[0].item()), float(tt[1].item())
        all_secs.append(round(sec, 5))
        if rep >= warm and (best is None or sec < best):
            best, best_c = sec, con
    nwin = (nb_e + ns_e) // a.sync
    return {"seconds": best, "construction_seconds": best_c, "all_seconds": all_secs, "chain_steps": Cg * ctx["world"] * (nb_e + ns_e),
            "h2d": int(Cg * d * 8 // nwin), "d2h": int((sink.nbytes + fin.nbytes) // nwin), "nwin": nwin}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="dgauss", choices=sorted(WORKLOADS))
    ap.add_argument("--chains", type=int, default=1 << 20, help="chains per GPU")
    ap.add_argument("--pool", type=int, default=16, help="remote-mixture pool size M")
    ap.add_argument("--remote-mode", default="reference", choices=sorted(RMODE),
                    help="reference: the reference's max-mixture rejection loop; summix: normalised sum-mixture proposal")
    ap.add_argument("--lag", type=int, default=1, choices=[0, 1],
                    help="1: a window reads the pool published two windows earlier (exchange off the critical path)")
    ap.add_argument("--pl", type=float, default=0.9)
    ap.add_argument("--coin-group", type=int, default=0, help="0: one local/remote coin per step for the whole job; 1..32: per group of chains")
    ap.add_argument("--thin", type=int, default=10)
    ap.add_argument("--sync", type=int, default=10)
    ap.add_argument("--advance", type=int, default=-1, help="untimed windows before the timed region (-1: the workload's default)")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: in-kernel peer-to-peer stores over NVLink (default) or an NCCL all-gather call per window")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-modes", action="store_true", help="skip the secondary measurements of the other remote modes")
    ap.add_argument("--no-check", action="store_true", help="N>1: skip the sharded == single-engine check")
    ap.add_argument("--no-place", action="store_true", help="do not move the timed region to a representative share of remote steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed windows, write the headline run's state, running moments and newest history row as "
                         "DIR/<name>.npy (float64; a fixed seeded sample of chains when all of them would exceed 64 MB)")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3                         # timing rule: W >= 3

    if args.impl == "reference":
        return run_reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from mcpar_b200 import engine

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = pin_to_gpu_numa(local)
    clocks = ClockSampler(local)                 # every rank, before anything is timed
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = dict(WORKLOADS[args.workload])
    if W["par"] == "gmix64":
        K_, d_, gmu, gs2, gw = gmix64_params()
        W["par"] = np.concatenate([[float(K_)], gmu.ravel(), gs2.ravel(), gw])
        W["pinit"] = lambda g_: gmu[g_ % K_]                       # chain g starts at mu_{g mod K}
    if "sync" in W and args.sync == 10:
        args.sync = W["sync"]
    if "thin" in W and args.thin == 10:
        args.thin = W["thin"]
    if args.advance < 0:
        args.advance = W["advance"]
    d, Cg, sync, thin = W["d"], args.chains, args.sync, args.thin
    placed_share = None
    if args.coin_group == 0 and not args.no_place:
        args.advance, placed_share = place_timed_region(SEED, d, 500, sync, args.lag, args.pl, args.advance, args.warmup, args.steps)
    N = Cg * world
    K, Wu = args.steps, args.warmup
    rmode = RMODE[args.remote_mode]

    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = {"args": args, "W": W, "rank": rank, "world": world, "local": local, "dev": dev, "stream": stream, "dist": dist,
           "groups": {world: None}}

    if world > 1 and args.exchange == "p2p":
        # probe with a throwaway engine that every rank can map every peer's exchange region (CUDA IPC +
        # peer access); all ranks then take the same path.  Both paths are GPU paths of the engine.
        pe, h = None, b""
        try:
            pe = engine.Engine(2, 64, nchain_total=64 * world, chain0=64 * rank, pool_m=world, device=local)
            h = pe.p2p_export()
        except engine.McgpuError as ex:
            sys.stderr.write("rank %d: peer-to-peer export failed (%s)\n" % (rank, ex))
        hs = [None] * world
        dist.all_gather_object(hs, h)
        ok = int(all(len(x) == engine.P2P_HANDLE_BYTES for x in hs))
        if ok:
            try:
                pe.p2p_attach(world, rank, hs)
            except engine.McgpuError as ex:
                ok = 0
                sys.stderr.write("rank %d: peer-to-peer attach failed (%s)\n" % (rank, ex))
        flag = torch.tensor([ok], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        dist.barrier()
        if pe is not None:
            pe.close()
        if int(flag.item()) == 0:
            args.exchange = "nccl"
            if rank == 0:
                sys.stderr.write("peer-to-peer exchange unavailable on this box: using the NCCL all-gather exchange\n")

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
    head = measure(ctx, Cg, rmode, args.pool, K, args.advance, Wu, flush, clocks=clocks, dump=args.dump_outputs)
    ck = head["clocks"]

    # ---- the other remote-proposal configurations, measured the same way (shorter)
    modes = None
    if not args.no_modes:
        modes = {}
        Km = min(K, 200)
        todo = [("summix_M16", 1, 16), ("summix_M256", 1, 256)] if W["d"] <= 16 else [("summix_M256", 1, 256)]
        if rmode == 1:
            todo = [("reference_M16", 0, 16)] + [t for t in todo if t[2] != args.pool]
        for name, rm, M in todo:
            r = measure(ctx, Cg, rm, M, Km, min(args.advance, 300), Wu, flush)
            modes[name] = {k: r[k] for k in ("value", "ms_per_step", "pool_m", "remote_mode", "steps", "advance", "remote_fraction",
                                             "remote_iterations_mean", "exact_fallback_rate", "accept_rate", "posterior_mean",
                                             "exchange_wait_ms_per_step")}

    check = None
    if world > 1 and not args.no_check:
        check = sharded_equals_single(ctx)

    # ---- end to end: MCPar::run-shaped job through the C ABI with HOST buffers
    e2e = None
    if not args.no_e2e:
        del flush; torch.cuda.empty_cache()
        f32 = e2e_job(ctx, Cg, rmode, args.pool, True, 3)              # rows in the reference MCout's element type (float)
        f64 = e2e_job(ctx, Cg, rmode, args.pool, False, 3)
        e2e = {"value": f32["chain_steps"] / f32["seconds"], "unit": UNIT,
               "h2d_bytes_per_step": f32["h2d"], "d2h_bytes_per_step": f32["d2h"],
               "job": "set_state(host pinit) + burnin 500 + 1000 steps + history(thin %d, fp32 rows = the reference MCout's element "
                      "type, narrowed on the device; device history = a ring of 16 kept steps drained on a side stream) and final logL "
                      "to pinned host; bytes are per %d-step window of the %d-window job; best of 3 after 2 untimed repetitions (all in all_seconds)" % (thin, sync, f32["nwin"]),
               "seconds": f32["seconds"], "all_seconds": f32["all_seconds"], "construction_seconds": f32["construction_seconds"],
               "construction": "engine create + likelihood/covariance upload + exchange wiring (CUDA IPC attach), outside the e2e clock, max over ranks",
               "host_numa": numa,
               "fp64_sink": {"value": f64["chain_steps"] / f64["seconds"], "seconds": f64["seconds"], "all_seconds": f64["all_seconds"], "d2h_bytes_per_step": f64["d2h"],
                             "note": "same job with fp64 rows on the host (twice the PCIe bytes)"}}

    if rank == 0:
        peak = engine.measure_fp64_peak(local)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        per_gpu = head["value"] / world
        bytes_step = 2 * (3 * d + 1) * 8 / sync + (d + 1) * 8 / thin     # state round trip + history, SURVEY 8(d)
        key = "%s/%s/M%d" % (args.workload, args.remote_mode, args.pool)
        prof = {}
        try:
            allprof = json.load(open(os.path.join(ROOT, "profiles", "fp64_work.json")))
            prof = allprof.get(key) or allprof.get("%s/local" % args.workload, {})      # no count for the mode: the local step's (a lower bound)
        except Exception:
            pass
        F = prof.get("fp64_flops_per_chain_step")
        ach = per_gpu * (F if F else W["F_hw"]) / 1e12
        roof = {"bound": "fp64", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak if peak else None,
                "traffic": prof.get("dram_bytes_per_launch"),
                "flops_per_chain_step": F if F else W["F_hw"],
                "flops_source": ("ncu: (dadd + dmul + 2 dfma) thread instructions of the window kernels / chain-steps, %s" % prof.get("source", "profiles/fp64_work.json")
                                 if F else "SURVEY.md 8(d) a-priori estimate (no ncu count committed for %s)" % key),
                "fp64_pipe_util_ncu": prof.get("fp64_pipe_pct"), "issue_slot_util_ncu": prof.get("issue_active_pct"),
                "warp_instructions_per_chain_step_ncu": prof.get("warp_instructions_per_chain_step"),
                "note": "achieved = chain-steps/s/GPU x fp64 flops per chain-step; peak = DFMA micro-kernel measured in this run "
                        "(MEASURED_PEAKS.json has no fp64 figure); kernel time = CUDA events around each window launch; traffic and the "
                        "pipe / issue-slot utilisation come from the committed ncu capture of this configuration (profiles/README.md), null if none.  "
                        "The step kernels are bound by issue slots and two half-rate integer pipes beside the FP64 pipe (DESIGN.md section 5): "
                        "the remote proposals' pool tests run in fp32 under rigorous bounds and add no fp64 work",
                "achieved_textbook_tflops": per_gpu * W["F_alg"] / 1e12,
                "hbm": {"achieved": per_gpu * bytes_step / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": per_gpu * bytes_step / 1e9 / hbm_peak, "bytes_per_chain_step": bytes_step,
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}}
        cpu = None if (args.no_cpu or world > 1) else cpu_baseline(args.workload)   # rank 0 at N = 1 only
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wu,
                "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "%s: %s d=%d, %d chains/GPU x %d GPU, PLOCAL %.2f, SYNCSTEP %d, remote mode %s, pool M=%d, pool lag %d, %s, "
                                       "thin %d, seed %d; step = one %d-step exchange window; %d untimed windows before the timed region (placed where the "
                                       "region's share of remote steps is closest to 1 - PLOCAL: the coins are counter-based)" % (
                                           W["name"], W["lik"], d, Cg, world, args.pl, sync, args.remote_mode, args.pool, args.lag,
                                           "one local/remote coin per step" if args.coin_group == 0 else "coin per %d chains" % args.coin_group,
                                           thin, SEED, sync, args.advance + Wu),
                           "l2": "flushed between timed steps (256 MiB memset outside the event pair)",
                           "parallelism": ("single GPU" if world == 1 else
                                           "chains sharded by global id; pool exchanged inside the window kernel by peer-to-peer stores over NVLink"
                                           if args.exchange == "p2p" else
                                           "chains sharded by global id; pool all-gather over NCCL each window")},
                "clocks": ck, "e2e": e2e, "gpu_launches": int(head["launches"]), "roofline": roof, "cpu_baseline": cpu,
                "per_rank_ms_per_step": head["per_rank_ms_per_step"], "accept_rate": head["accept_rate"],
                "remote_fraction": head["remote_fraction"], "remote_iterations_mean": head["remote_iterations_mean"],
                "exact_fallback_rate": head["exact_fallback_rate"],
                "exchange_wait_ms_per_step": head["exchange_wait_ms_per_step"],
                "posterior_mean": head["posterior_mean"], "posterior_var": head["posterior_var"],
                "modes": modes, "sharded_equals_single": check}
        if args.dump_outputs:
            line["dump_outputs"] = {"dir": args.dump_outputs, "chains_per_gpu": head["dumped_chains"], "of": Cg}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
