"""The runs that compare the production step kernels with the CPU oracle, each with the kernel instantiations it launches.

Every `mh_steps_kernel`, `mh_wide_kernel` and `mh_coop_kernel` instantiation in libmcgpu.so is separately compiled code.
Each case below names, in `claims`, the instantiations its run launches:
  ("steps", unit, LIK, D, RNG, PHASE)      thread-per-chain kernel of the fast or exact unit
  ("wide", LIK, D, NCH, PHASE)             wide kernel, D/2 lanes and NCH chains per lane group
  ("coop", D, NCW, PHASE, POOLSM)          CTA-cooperative GaussMix kernel
test_kernel_coverage.py checks that these claims and the library's kernels are the same set, and
test_gpu_kernel_routing.py that each run launches exactly its claims.  test_gpu_parity.py compares every case with
the oracle, and recomputes every kept log-likelihood in extended precision (`loglik_ld`)."""
import re
from collections import namedtuple

import numpy as np

from conftest import tiled_pinit

LIKS = {0: "ROSENBROCK1", 2: "GAUSSIAN", 3: "DUALGAUSSIAN", 4: "GAUSSMIX", 101: "PLUGIN"}
PHASES = ("BURN", "MIXED", "LOCAL", "REMOTE", "MIXED_SUM", "REMOTE_SUM")      # mh_launch.h
RNGS = ("PHILOX", "REPLAY")

_MANGLED = re.compile(r"_ZN5mcgpu(4fast|5exact)\d+(mh_steps_kernel|mh_wide_kernel|mh_coop_kernel)I((?:L[ib]\d+E)+)E")
_DEMANGLED = re.compile(r"mcgpu::(fast|exact)::(mh_steps_kernel|mh_wide_kernel|mh_coop_kernel)<([^>]*)>")


def kernel_key(name):
    """Key of a step-kernel instantiation from its mangled (cuobjdump) or demangled (profiler) name; None otherwise."""
    m = _MANGLED.search(name)
    if m:
        unit, kind = m.group(1)[1:], m.group(2)
        args = [int(a) for a in re.findall(r"L[ib](\d+)E", m.group(3))]
    else:
        m = _DEMANGLED.search(name)
        if not m:
            return None
        unit, kind = m.group(1), m.group(2)
        args = [{"true": 1, "false": 0}.get(a, None) for a in (s.strip() for s in m.group(3).split(","))]
        args = [int(s) if a is None else a for s, a in zip(m.group(3).split(","), args)]
    if kind == "mh_steps_kernel":
        lik, d, rng, ph = args
        return ("steps", unit, LIKS[lik], d, RNGS[rng], PHASES[ph])
    if kind == "mh_wide_kernel":
        lik, d, nch, ph = args
        return ("wide", LIKS[lik], d, nch, PHASES[ph])
    d, ncw, ph, poolsm = args
    return ("coop", d, ncw, PHASES[ph], poolsm)


# ---------------------------------------------------------------- claim helpers
def steps(lik, d, *phases, unit="fast"):
    rng = "PHILOX" if unit == "fast" else "REPLAY"
    return {("steps", unit, lik, d, rng, ph) for ph in phases}


def wide(lik, d, *phases):
    nch = 1 if d < 32 else (2 if d < 64 else 4)          # WideNch (mh_wide.cuh)
    return {("wide", lik, d, nch, ph) for ph in phases}


def coop(*phases):                                        # launch_coop_phase (mh_fast.cu): remote kernels one chain per owner warp
    return {("coop", 64, 1 if ph == "REMOTE_SUM" else 4, ph, 1) for ph in phases}


R1, GA, DG, GM = "ROSENBROCK1", "GAUSSIAN", "DUALGAUSSIAN", "GAUSSMIX"
B, M_, L_, R_, MS, RS = PHASES[0], PHASES[1], PHASES[2], PHASES[3], PHASES[4], PHASES[5]

# ---------------------------------------------------------------- models
# GaussMix specs: name -> (K, unequal weights, mean offset).  Components k are drawn from one generator (seed 8): means
# uniform in [-5, 5], variances in [0.5, 2]; unequal weights uniform in [0.2, 3]; the offset moves even components by
# +offset and odd ones by -offset in every parameter (far means: the expanded exponent of the wide kernels cancels).
GMIX = {"gmix64": (64, False, 0.0), "gmix16": (5, False, 0.0), "gmix2": (3, True, 0.0), "gmix4": (5, True, 0.0),
        "gmix8": (3, True, 0.0), "gmix16w": (5, True, 0.0), "gmix32far": (20, True, 40.0), "gmix64k80": (80, True, 0.0)}


def rosen_factor(d):
    """Full lower proposal covariance: the Rosenbrock pair's posterior covariance, one 2x2 block per pair."""
    return np.kron(np.eye(d // 2), (2.38 ** 2 / d) * np.array([[0.5, 1.0], [1.0, 2.505]]))


def model(lik, d, N, par):
    """(par, incov, pinit) of a case: `par` is a parameter list, None, or the name of a spec above."""
    from oracle import mh
    pin, incov = tiled_pinit(N, d), None
    if isinstance(par, str) and par.startswith("rosen"):
        par, incov = None, rosen_factor(d)
    elif isinstance(par, str):                       # K-component mixture in d dimensions, chains start on the means
        K, unequal, off = GMIX[par]
        rng = np.random.default_rng(8)
        gmu = rng.uniform(-5, 5, (K, d)); gs2 = rng.uniform(0.5, 2.0, (K, d))
        w = rng.uniform(0.2, 3.0, K) if unequal else np.ones(K)
        gmu = gmu + off * np.where(np.arange(K) % 2 == 0, 1.0, -1.0)[:, None]
        par = mh.gaussmix_params(K, d, gmu, gs2, w)
        pin = gmu[np.arange(N) % K].copy()
        incov = np.eye(d) * (2.38 ** 2 / d)
    return par, incov, pin


# ---------------------------------------------------------------- normal-mode cases
Case = namedtuple("Case", "id lik d N par pool_m pl cg rmode lag sync thin nsamp claims")
NBURN = 120


def _legacy(i, lik, d, N, par, pool_m, pl, cg, rmode, lag, claims):
    """A case of the original oracle parametrization, under its original test id."""
    pid = "par%d" % i if isinstance(par, list) else str(par)
    cid = "-".join([lik, str(d), str(N), pid, str(pool_m), str(pl), str(cg), str(rmode), str(lag)])
    return Case(cid, lik, d, N, par, pool_m, pl, cg, rmode, lag, 10, 1, 60, frozenset(claims))


def _case(cid, lik, d, N, par, pool_m, pl, cg, rmode, lag, sync, thin, nsamp, claims):
    return Case(cid, lik, d, N, par, pool_m, pl, cg, rmode, lag, sync, thin, nsamp, frozenset(claims))


_L = [
    ("rosenbrock1", 2, 256, None, 0, 0.9, 32, 0, 0, steps(R1, 2, B, M_)),
    ("rosenbrock1", 2, 512, None, 16, 0.7, 32, 0, 0, steps(R1, 2, B, M_)),
    ("dualgaussian", 2, 256, [5.0], 8, 0.8, 32, 0, 0, steps(DG, 2, B, M_)),
    ("rosenbrock1", 4, 128, None, 8, 0.8, 32, 0, 0, steps(R1, 4, B, M_)),
    ("dualgaussian", 2, 256, [5.0], 8, 0.8, 4, 0, 0, steps(DG, 2, B, M_)),        # rank-sized coin groups (mixed warps)
    ("dualgaussian", 2, 512, [5.0], 16, 0.7, 0, 0, 0, steps(DG, 2, B, L_, M_)),   # job-wide coin: host-planned windows
    ("rosenbrock1", 2, 200, None, 10, 0.6, 0, 0, 0, steps(R1, 2, B, L_, M_)),     # ragged: chains not a multiple of 32, pool not of 8
    ("rosenbrock1", 16, 72, "rosen16", 8, 0.7, 0, 0, 0, wide(R1, 16, B, L_, R_)),  # wide kernel: 8 lanes per chain, full lower factor
    ("rosenbrock1", 8, 40, None, 5, 0.7, 0, 0, 0, wide(R1, 8, B, L_, R_)),        # wide kernel: 4 lanes per chain, diagonal factor
    ("gaussmix", 64, 24, "gmix64", 6, 0.7, 0, 0, 0, coop(B, L_) | wide(GM, 64, R_)),   # K = 64: cooperative kernel; pool M < D/2 lanes
    ("gaussmix", 16, 48, "gmix16", 8, 0.8, 0, 0, 0, wide(GM, 16, B, L_, R_)),
    ("dualgaussian", 2, 512, [5.0], 16, 0.7, 0, 0, 1, steps(DG, 2, B, L_, M_)),   # pool read one exchange late
    ("rosenbrock1", 2, 256, None, 8, 0.7, 32, 0, 1, steps(R1, 2, B, M_)),
    # remote mode 1: sum-mixture independence proposal with normalised components (no rejection loop)
    ("dualgaussian", 2, 512, [5.0], 16, 0.7, 0, 1, 0, steps(DG, 2, B, L_, MS)),
    ("dualgaussian", 2, 512, [5.0], 64, 0.6, 0, 1, 1, steps(DG, 2, B, L_, MS)),
    ("rosenbrock1", 2, 200, None, 10, 0.6, 0, 1, 0, steps(R1, 2, B, L_, MS)),     # ragged
    ("rosenbrock1", 2, 256, None, 0, 0.8, 32, 1, 0, steps(R1, 2, B, MS)),         # every chain in the pool, per-group coins
    ("dualgaussian", 2, 256, [5.0], 8, 0.8, 4, 1, 1, steps(DG, 2, B, MS)),        # rank-sized coin groups, lagged pool
    ("rosenbrock1", 4, 128, None, 8, 0.8, 32, 1, 0, steps(R1, 4, B, MS)),
    ("rosenbrock1", 16, 72, "rosen16", 8, 0.7, 0, 1, 0, wide(R1, 16, B, L_, RS)),
    ("rosenbrock1", 8, 40, None, 5, 0.7, 0, 1, 1, wide(R1, 8, B, L_, RS)),
    ("gaussmix", 64, 24, "gmix64", 6, 0.7, 0, 1, 0, coop(B, L_, RS)),
    ("gaussmix", 64, 136, "gmix64", 40, 0.7, 0, 1, 1, coop(B, L_, RS)),
    ("gaussmix", 64, 256, "gmix64", 0, 0.7, 0, 1, 0, coop(B, L_, RS)),            # every chain in the pool: M = 256
    ("gaussmix", 16, 48, "gmix16", 8, 0.8, 0, 1, 0, wide(GM, 16, B, L_, RS)),
]
CASES = [_legacy(i, *c) for i, c in enumerate(_L)]

# Thread-per-chain kernels in all their phases.  A window longer than 32 steps under the job-wide coin runs as chunks of at
# most 32 steps (the width of the plan mask), each one LOCAL or MIXED(_SUM) launch: sync 40 (chunks of 32 + 8), 160 main
# steps after the sync (1 + lag) local lead-in.
for _lik, _d, _N, _par in [("gaussian", 2, 96, [1.0, -1.0, 0.5, 2.0]), ("gaussmix", 2, 96, "gmix2"), ("gaussmix", 4, 80, "gmix4")]:
    _k = {"gaussian": GA, "gaussmix": GM}[_lik]
    _n = "%s%d" % (_lik, _d)
    CASES += [
        _case(_n + "-sync40-ref", _lik, _d, _N, _par, 8, 0.7, 0, 0, 0, 40, 1, 160, steps(_k, _d, B, L_, M_)),
        _case(_n + "-sync40-sum-lag1", _lik, _d, _N, _par, 8, 0.7, 0, 1, 1, 40, 1, 160, steps(_k, _d, B, L_, MS)),
        _case(_n + "-groups-ref", _lik, _d, _N, _par, 8, 0.7, 8, 0, 0, 10, 1, 60, steps(_k, _d, B, M_)),
        _case(_n + "-groups-sum", _lik, _d, _N, _par, 8, 0.7, 8, 1, 0, 10, 1, 60, steps(_k, _d, B, MS)),
    ]
# the same windows for the other thread-per-chain likelihoods, and sync 70: chunks of 32 + 32 + 6 steps, so a middle chunk
# that neither starts nor ends its window, with thin 3 putting the chunks' first steps off the kept rows (t0 = 32, 64)
CASES += [
    _case("rosenbrock12-sync40-ref", "rosenbrock1", 2, 128, None, 8, 0.7, 0, 0, 0, 40, 1, 160, steps(R1, 2, B, L_, M_)),
    _case("rosenbrock12-sync40-sum", "rosenbrock1", 2, 128, None, 8, 0.7, 0, 1, 0, 40, 1, 160, steps(R1, 2, B, L_, MS)),
    _case("rosenbrock14-sync40-ref", "rosenbrock1", 4, 96, None, 8, 0.7, 0, 0, 0, 40, 1, 160, steps(R1, 4, B, L_, M_)),
    _case("rosenbrock14-sync40-sum-lag1", "rosenbrock1", 4, 96, None, 8, 0.7, 0, 1, 1, 40, 1, 160, steps(R1, 4, B, L_, MS)),
    _case("dualgaussian2-sync40-ref", "dualgaussian", 2, 128, [5.0], 8, 0.7, 0, 0, 0, 40, 1, 160, steps(DG, 2, B, L_, M_)),
    _case("dualgaussian2-sync40-sum", "dualgaussian", 2, 128, [5.0], 8, 0.7, 0, 1, 0, 40, 1, 160, steps(DG, 2, B, L_, MS)),
    _case("rosenbrock12-sync70-thin3", "rosenbrock1", 2, 200, None, 10, 0.6, 0, 0, 0, 70, 3, 210, steps(R1, 2, B, L_, M_)),
]
# thread-per-chain kernels at d >= 8: only per-group coins launch them (the job-wide coin takes the wide kernels)
for _lik, _d, _par in [("rosenbrock1", 8, None), ("rosenbrock1", 16, "rosen16"), ("gaussmix", 8, "gmix8"), ("gaussmix", 16, "gmix16w")]:
    _k = {"rosenbrock1": R1, "gaussmix": GM}[_lik]
    CASES += [
        _case("%s%d-groups-ref" % (_lik, _d), _lik, _d, 64, _par, 8, 0.7, 8, 0, 0, 10, 1, 60, steps(_k, _d, B, M_)),
        _case("%s%d-groups-sum" % (_lik, _d), _lik, _d, 64, _par, 8, 0.7, 8, 1, 0, 10, 1, 60, steps(_k, _d, B, MS)),
    ]
# wide kernels with 2 and 4 chains per lane group, the last group partly live (70 = 35 x 2, 42 = 10 x 4 + 2)
CASES += [
    _case("rosenbrock132-wide-ref", "rosenbrock1", 32, 70, "rosen32", 8, 0.7, 0, 0, 0, 10, 1, 60, wide(R1, 32, B, L_, R_)),
    _case("rosenbrock132-wide-sum-lag1", "rosenbrock1", 32, 70, "rosen32", 8, 0.7, 0, 1, 1, 10, 1, 60, wide(R1, 32, B, L_, RS)),
    _case("rosenbrock164-wide-ref", "rosenbrock1", 64, 42, "rosen64", 8, 0.7, 0, 0, 0, 10, 1, 60, wide(R1, 64, B, L_, R_)),
    _case("rosenbrock164-wide-sum-lag1", "rosenbrock1", 64, 42, "rosen64", 8, 0.7, 0, 1, 1, 10, 1, 60, wide(R1, 64, B, L_, RS)),
]
# wide GaussMix: padding components (K = 3 in kpad 8), far means (K = 20), and K = 80 at d = 64 (kpad 128: the wide kernel,
# not the cooperative one, which takes kpad = 64 only)
for _d, _N, _par in [(8, 40, "gmix8"), (32, 70, "gmix32far"), (64, 42, "gmix64k80")]:
    CASES += [
        _case("gaussmix%d-wide-%s-ref" % (_d, _par), "gaussmix", _d, _N, _par, 8, 0.7, 0, 0, 0, 10, 1, 60, wide(GM, _d, B, L_, R_)),
        _case("gaussmix%d-wide-%s-sum" % (_d, _par), "gaussmix", _d, _N, _par, 8, 0.7, 0, 1, 0, 10, 1, 60, wide(GM, _d, B, L_, RS)),
    ]
CASES += [
    # cooperative burn-in and local steps, wide sum-mixture remote steps: pool M = 300 (mpad 304 > 256)
    _case("gaussmix64-coop-wide-M300", "gaussmix", 64, 320, "gmix64", 300, 0.7, 0, 1, 0, 10, 1, 60, coop(B, L_) | wide(GM, 64, RS)),
    # one-step windows (BASELINE config 4's shape) and thinning that does not align with the windows
    _case("gaussmix64-sync1-sum-lag1", "gaussmix", 64, 64, "gmix64", 16, 0.7, 0, 1, 1, 1, 1, 60, coop(B, L_, RS)),
    _case("rosenbrock116-wide-sync1", "rosenbrock1", 16, 72, "rosen16", 8, 0.7, 0, 0, 0, 1, 1, 60, wide(R1, 16, B, L_, R_)),
    _case("rosenbrock12-thin3", "rosenbrock1", 2, 200, None, 10, 0.6, 0, 0, 0, 10, 3, 61, steps(R1, 2, B, L_, M_)),
    _case("rosenbrock18-wide-thin3-sum", "rosenbrock1", 8, 40, None, 5, 0.7, 0, 1, 0, 10, 3, 61, wide(R1, 8, B, L_, RS)),
]

# ---------------------------------------------------------------- replay-mode cases (exact unit, all-local)
Replay = namedtuple("Replay", "id lik d C par incov claims")


def _replay(i, lik, d, C, par, incov):
    k = {"rosenbrock1": R1, "dualgaussian": DG, "gaussian": GA, "gaussmix": GM}[lik]
    pid = "par%d" % i if isinstance(par, list) else str(par)
    return Replay("-".join([lik, str(d), str(C), pid, str(incov)]), lik, d, C, par, incov,
                  frozenset(steps(k, d, B, L_, unit="exact")))


REPLAY = [_replay(i, *c) for i, c in enumerate([
    ("rosenbrock1", 2, 96, None, None),
    ("dualgaussian", 2, 200, [5.0], None),
    ("rosenbrock1", 16, 64, None, "rosen16"),
    ("gaussian", 2, 33, [0.5, -0.5, 1.5, 0.7], None),
    ("rosenbrock1", 4, 64, None, None),
    ("rosenbrock1", 8, 64, None, None),
    ("gaussmix", 2, 40, "gmix2", None),
    ("gaussmix", 4, 40, "gmix4", None),
    ("gaussmix", 8, 40, "gmix8", None),
    ("gaussmix", 16, 40, "gmix16w", None),
])]


def all_claims():
    out = set()
    for c in CASES + REPLAY:
        out |= c.claims
    return out


# ---------------------------------------------------------------- extended-precision log-likelihood
EPS = 2.0 ** -53             # unit roundoff of fp64


def loglik_ld(lik, d, x, par, expanded):
    """(L, S, c) per row of x: log L(x) in x86 extended precision, and the error bound c*EPS*S of the kernels' fp64
    evaluation.  S sums the magnitudes of the intermediate terms the kernel's own formula forms; c counts the roundings
    each term passes through (first order; an FMA only removes roundings).  `expanded`: GaussMix in the wide and
    cooperative kernels' expanded form c_k + sum_i x_i (a_ki x_i + b_ki) instead of the direct (x - mu)^2 form."""
    assert np.finfo(np.longdouble).nmant >= 63, "needs x86 80-bit long double"
    X = np.asarray(x, dtype=np.longdouble).reshape(-1, d)
    one = np.longdouble(1)
    if lik == "rosenbrock1":
        # pair (x0, x1): t1 = 1 - x0 (one rounding), t2 = x1 - x0^2 (error <= eps (x0^2 + |t2|)), then t1^2 + 100 t2^2:
        # <= eps (4 t1^2 + 600 t2^2 + 200 |t2| x0^2) <= 6 eps S_pair, S_pair = t1^2 + 100 t2^2 + 200 |t2| x0^2;
        # the d/2 pair values are summed in d/2 - 1 additions (sequential or butterfly): c = 6 + d/2
        x0, x1 = X[:, 0::2], X[:, 1::2]
        t1, t2 = one - x0, x1 - x0 * x0
        v = t1 * t1 + 100 * t2 * t2
        return -v.sum(1), (v + 200 * np.abs(t2) * x0 * x0).sum(1), 6 + d // 2
    if lik == "gaussian":
        # term 0.5 (x - mu)^2 / s2 with 1/s2 rounded on upload: subtraction (2 eps after squaring), two products,
        # the reciprocal: 5 eps per term, + 1 for the two-term sum: c = 7
        mu, s2 = np.asarray(par[:2], np.longdouble), np.asarray(par[2:4], np.longdouble)
        g = 0.5 * (X - mu) ** 2 / s2
        return -g.sum(1), g.sum(1), 7
    if lik == "dualgaussian":
        # one-exponential form M + log(1 + e^-|t1 - t2|), t1 = log w - a1, t2 = -a2: a1 = |x|^2/2 carries 3 eps a1,
        # a2 4 eps a2, log w (host libm) 2 eps |log w|, t1 and dt one rounding each, the table exp and log <= 1.5 ulp
        # and the argument's rounding <= 10 eps in all, the final sum eps |L|: <= 9 a1 + 9 a2 + 7 |log w| + |L| + 10
        # in units of eps, so S = a1 + a2 + |log w| + |L| + 1 and c = 12.  Both exponentials below e^-708: -inf.
        w = np.longdouble(par[0] if par else 5.0)
        a1 = 0.5 * (X ** 2).sum(1)
        a2 = 0.5 * ((X - 5) ** 2).sum(1)
        L = np.log(w * np.exp(-a1) + np.exp(-a2))
        L[(a1 >= 708) & (a2 >= 708)] = -np.inf
        return L, a1 + a2 + np.abs(np.log(w)) + np.abs(L) + 1, 12
    assert lik == "gaussmix"
    K = int(par[0])
    p = np.asarray(par[1:], np.longdouble)
    mu, s2, w = p[:K * d].reshape(K, d), p[K * d:2 * K * d].reshape(K, d), p[2 * K * d:]
    lw = np.log(w)
    a = np.empty((X.shape[0], K), np.longdouble)
    t = np.empty_like(a)
    for k in range(K):
        q = 0.5 * ((X - mu[k]) ** 2 / s2[k]).sum(1)
        a[:, k] = lw[k] - q
        if expanded:
            # c_k + sum_i x_i (A x_i + B), A = -1/(2 s2), B = mu / s2, c_k = log w - 1/2 sum mu^2 / s2 (rounded once on
            # upload): the inner FMA and the reciprocal/product of A and B cost <= 4 eps of |A| x^2 + |B x|, the D-term
            # FMA chain (D - 1) eps of the same, c_k and log w one rounding each
            ck = lw[k] - 0.5 * (mu[k] ** 2 / s2[k]).sum()
            t[:, k] = np.abs(ck) + (X * X / (2 * s2[k]) + np.abs(X * mu[k] / s2[k])).sum(1) + np.abs(lw[k]) + np.abs(a[:, k])
        else:
            # lw - 1/2 sum (x - mu)^2 / s2: 5 eps per term (as Gaussian), the D-term sum, log w and the difference
            t[:, k] = q + np.abs(lw[k]) + np.abs(a[:, k])
    m = a.max(1)
    e = np.exp(a - m[:, None])
    s = e.sum(1)
    L = m + np.log(s)
    pk = e / s[:, None]
    # log-sum-exp: the error of component k's exponent reaches L with weight p_k <= 1, <= (D + 5) eps T_k; the running
    # sum of K exponentials (each <= 1.5 ulp, rescaled at most K times) and the butterfly over the lanes <= 5 K eps
    # relative, the log 3 eps, the last sum eps |L|: S = sum_k p_k T_k + |L| + 1, c = D + 5 K + 8
    return L, (pk * t).sum(1) + np.abs(L) + 1, d + 5 * K + 8
