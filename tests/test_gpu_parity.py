"""GPU parity tests: the CUDA engine, called through the C ABI (libmcgpu.so via ctypes),
against the CPU oracle (oracle/mh_oracle.c, itself pinned to the reference build).

Bar: verification mode -- identical accept/reject sequences, identical stream
consumption, states and polynomial log-likelihoods bit-identical, transcendental
log-likelihoods within 1e-12 relative (north star).
"""
import numpy as np
import pytest

import kernel_matrix as km
from conftest import make_streams, tiled_pinit
from oracle import mh

pytestmark = pytest.mark.gpu

RTOL = 1e-12          # north star: log-likelihoods within 1e-12 relative in fp64
ATOL = 1e-14          # floor for values that cross zero (log of a quantity near 1)


def _engine():
    from mcpar_b200 import engine
    return engine


def _close(a, b, rtol=RTOL, atol=ATOL):
    a = np.asarray(a, float); b = np.asarray(b, float)
    both_inf = np.isinf(a) & np.isinf(b) & (np.sign(a) == np.sign(b))
    ok = both_inf | (np.abs(a - b) <= atol + rtol * np.abs(b))
    return bool(np.all(ok))


# ---------------------------------------------------------------- likelihoods
@pytest.mark.parametrize("lik,d,par", [
    ("rosenbrock1", 2, None), ("rosenbrock1", 16, None), ("rosenbrock2", 4, None),
    ("gaussian", 2, [1.0, -1.0, 0.5, 2.0]), ("dualgaussian", 2, [5.0]),
])
def test_loglik_matches_oracle(lik, d, par):
    eng = _engine()
    rng = np.random.default_rng(7)
    x = rng.normal(1.0, 2.0, size=(100003, d))
    y = eng.loglik(lik, d, x, par)
    yo = mh.loglik(lik, d, x, par)
    if lik.startswith("rosenbrock") or lik == "gaussian":
        assert np.array_equal(y, yo)          # polynomial: bit-identical
    else:
        assert _close(y, yo)


def test_loglik_known_answers():
    eng = _engine()
    assert np.array_equal(eng.loglik("rosenbrock1", 2, [[1, 1], [0, 0], [2, 2]]), [0.0, -1.0, -401.0])
    y = eng.loglik("dualgaussian", 2, [[0, 0], [5, 5], [100, 100]], [5.0])
    assert _close(y[:2], [np.log(5 + np.exp(-25)), np.log(5 * np.exp(-25) + 1)])
    assert y[2] == -np.inf                    # no log-sum-exp guard, as in the reference


def test_loglik_gaussmix():
    eng = _engine()
    rng = np.random.default_rng(3)
    K, d = 5, 4
    par = mh.gaussmix_params(K, d, rng.normal(0, 3, (K, d)), rng.uniform(0.5, 2, (K, d)), rng.uniform(0.5, 2, K))
    x = rng.normal(0, 4, size=(5000, d))
    assert _close(eng.loglik("gaussmix", d, x, par), mh.loglik("gaussmix", d, x, par), rtol=1e-11)


def test_loglik_rejects_bad_shapes():
    eng = _engine()
    with pytest.raises(eng.McgpuError):
        eng.loglik("rosenbrock1", 3, np.zeros((2, 3)))
    with pytest.raises(eng.McgpuError):
        eng.loglik("gaussian", 3, np.zeros((2, 3)))


# ---------------------------------------------------------------- verification mode
def _run_verify(lik, d, C, R, nsamp, nburn, par=None, incov=None, pl=0.9, sync=10, seed=1, split=None):
    eng = _engine()
    pin = tiled_pinit(C, d)
    Z, U, I = make_streams(R, C, d, nsamp + nburn, seed)
    o = mh.run_replay(lik, d, C, R, nsamp, nburn, pin, Z, U, I, incov=incov, par=par, pl=pl, sync=sync, trace=True)
    e = eng.Engine(d, R * C, mode="verify", chains_per_rank=C, pl=pl, sync=sync, trace=nburn + nsamp,
                   history_steps=nsamp)
    e.set_likelihood(lik, par)
    e.set_covariance(incov)
    e.set_state(np.tile(pin, (R, 1)))
    for r in range(R):
        e.set_streams(r, Z[r], U[r], I[r])
    e.burnin(nburn)
    e.sample_begin(nsamp)
    if split:
        done = 0
        for n in split:
            e.sample(n); done += n
        e.sample(nsamp - done)
    else:
        e.sample(nsamp)
    e.synchronize()
    return o, e


@pytest.mark.parametrize("lik,d,C,R,nsamp,nburn,par,incov,pl,sync", [
    ("rosenbrock1", 2, 4, 1, 200, 120, None, None, 0.9, 10),
    ("rosenbrock1", 2, 4, 3, 300, 200, None, None, 0.9, 10),
    ("dualgaussian", 2, 4, 2, 200, 120, [5.0], None, 0.9, 10),
    ("gaussian", 2, 8, 2, 100, 120, [1.0, -1.0, 0.5, 2.0], None, 0.9, 10),
    ("rosenbrock2", 4, 4, 2, 100, 120, None, None, 0.9, 10),
    ("rosenbrock1", 4, 5, 2, 100, 520, None, "spd4", 0.9, 10),
    ("rosenbrock1", 2, 1, 1, 100, 120, None, None, 0.9, 10),
    ("rosenbrock1", 2, 4, 2, 55, 0, None, None, 0.5, 3),
    ("rosenbrock1", 2, 40, 2, 60, 60, None, None, 0.7, 10),
])
def test_verify_mode_matches_oracle(lik, d, C, R, nsamp, nburn, par, incov, pl, sync):
    if incov == "spd4":
        incov = np.diag([0.5, 2, 0.5, 2.0]) + 0.1
    o, e = _run_verify(lik, d, C, R, nsamp, nburn, par, incov, pl, sync)
    T = nburn + nsamp
    poly = lik in ("rosenbrock1", "rosenbrock2", "gaussian")
    st = e.state()
    for r in range(R):
        tr = e.trace(r, T)
        otr = o["trace"]
        assert np.array_equal(tr["accept"].astype(bool), o["accept"][r]), "accept/reject sequence differs"
        assert np.array_equal(tr["remote"], otr["remote"][r])
        assert np.array_equal(tr["iters"], otr["iters"][r])
        assert np.array_equal(tr["cursors"], o["used"][r][:3]), "stream consumption differs"
        assert np.array_equal(tr["trial_p"], otr["trial_p"][r]), "trial points are not bit-identical"
        if poly:
            assert np.array_equal(tr["trial_ly"], otr["trial_ly"][r])
        else:
            assert _close(tr["trial_ly"], otr["trial_ly"][r])
        assert _close(tr["cfac"], otr["cfac"][r], rtol=1e-11)
        assert np.array_equal(e.factor(r), o["cov"][r])
        sl = slice(r * C, (r + 1) * C)
        assert np.array_equal(st["p"][sl], o["p"][r])
        assert np.array_equal(st["mu"][sl], o["mu"][r]) and np.array_equal(st["psum2"][sl], o["psum2"][r])
        assert np.array_equal(st["sig"][sl], o["sig"][r])
        assert np.array_equal(e.musig(r), o["musig"][r])
        (np.testing.assert_array_equal if poly else np.testing.assert_allclose)(st["ly"][sl], o["ly"][r])
    # MCout contents: [step][rank*C + chain][d+1]  ->  reference per-rank row order
    h = e.history().reshape(nsamp, R, C, d + 1).transpose(1, 0, 2, 3).reshape(R, nsamp * C, d + 1)
    assert np.array_equal(h[..., :d], o["rows"][..., :d])
    assert _close(h[..., d], o["rows"][..., d])
    pm, lm = e.maxlike()
    assert _close(lm, o["maxl"][d]) and (not poly or np.array_equal(pm, o["maxl"][:d]))
    s = e.stats()
    assert s["remote_steps"] == int(otr["remote"].sum()) and s["remote_iterations"] == int(otr["iters"].sum())
    e.close()


def test_verify_mode_split_sample_calls():
    """Advancing in uneven pieces must not change anything (exchange boundaries are internal)."""
    o, e = _run_verify("rosenbrock1", 2, 4, 2, 95, 60, split=[3, 7, 15, 4])
    st = e.state()
    assert np.array_equal(st["p"].reshape(2, 4, 2), o["p"])
    assert np.array_equal(e.musig(1), o["musig"][1])
    e.close()


def test_stream_overrun_is_an_error():
    eng = _engine()
    e = eng.Engine(2, 4, mode="verify", chains_per_rank=4, trace=0, history_steps=0)
    e.set_likelihood("rosenbrock1")
    e.set_state(tiled_pinit(4, 2))
    e.set_streams(0, np.zeros(10), np.full(10, 0.5), np.zeros(10, np.int32))
    with pytest.raises(eng.McgpuError, match="ESTREAM"):
        e.burnin(50)
    e.close()


# ---------------------------------------------------------------- production kernel, replayed
@pytest.mark.parametrize("lik,d,C,par,incov", [pytest.param(c.lik, c.d, c.C, c.par, c.incov, id=c.id) for c in km.REPLAY])
def test_production_kernel_replay_local(lik, d, C, par, incov):
    """The production step kernel (exact-arithmetic instantiation) fed the reference's
    streams at the reference's offsets, all-local run (pl = 1): one rank of C chains."""
    eng = _engine()
    pin = tiled_pinit(C, d)
    if incov == "rosen16":
        incov = km.rosen_factor(16)
    if isinstance(par, str):                         # GaussMix spec: chains start on the means
        par, incov, pin = km.model(lik, d, C, par)
    nburn, nsamp = 230, 75
    Z, U, I = make_streams(1, C, d, nsamp + nburn, 11, mult=2)
    o = mh.run_replay(lik, d, C, 1, nsamp, nburn, pin, Z, U, I, incov=incov, par=par, pl=1.0, trace=True)
    e = eng.Engine(d, C, mode="replay_local", pl=1.0, history_steps=nsamp)
    e.set_likelihood(lik, par); e.set_covariance(incov); e.set_state(pin)
    e.set_streams(0, Z[0], U[0])
    e.burnin(nburn); e.sample_begin(nsamp); e.sample(nsamp); e.synchronize()
    st = e.state()
    poly = lik not in ("dualgaussian", "gaussmix")
    assert np.array_equal(st["p"], o["p"][0])
    assert np.array_equal(e.factor(), o["cov"][0]), "burn-in tuning history differs"
    assert np.array_equal(st["mu"], o["mu"][0]) and np.array_equal(st["psum2"], o["psum2"][0])
    h = e.history().reshape(nsamp * C, d + 1)
    assert np.array_equal(h[:, :d], o["rows"][0][:, :d])
    assert np.array_equal(h[:, d], o["rows"][0][:, d]) if poly else _close(h[:, d], o["rows"][0][:, d])
    s = e.stats()
    assert s["accepted"] == int(o["accept"][0][nburn:].sum()) and s["tried"] == nsamp * C
    e.close()


# ---------------------------------------------------------------- normal mode vs counter oracle
@pytest.mark.parametrize("lik,d,N,par,pool_m,pl,cg,rmode,lag,sync,thin,nsamp,expanded", [
    pytest.param(c.lik, c.d, c.N, c.par, c.pool_m, c.pl, c.cg, c.rmode, c.lag, c.sync, c.thin, c.nsamp,
                 any(k[0] != "steps" for k in c.claims), id=c.id) for c in km.CASES])
def test_normal_mode_matches_counter_oracle(lik, d, N, par, pool_m, pl, cg, rmode, lag, sync, thin, nsamp, expanded):
    """Same Philox draws on both sides: identical accept sequences; values agree to
    rounding (host libm vs CUDA libm differ in the last ulp of log/sin/cos/exp).  Every kept
    log-likelihood and the final state's are the likelihood of their own row, to the kernel's
    fp64 error bound against an extended-precision evaluation.  The cases and the kernels
    each one launches: tests/kernel_matrix.py (`expanded`: a wide or cooperative kernel evaluates the run's
    GaussMix in the expanded form)."""
    eng = _engine()
    nburn = km.NBURN
    kept = (nsamp + thin - 1) // thin
    par, incov, pin = km.model(lik, d, N, par)
    o = mh.run_counter(lik, d, N, nsamp, nburn, pin, incov=incov, par=par, pool_m=pool_m, pl=pl, coin_group=cg, trace=True,
                       remote_mode=rmode, pool_lag=lag, sync=sync, thin=thin)
    e = eng.Engine(d, N, mode="normal", pool_m=pool_m, pl=pl, coin_group=cg, history_steps=kept, remote_mode=rmode,
                   pool_lag=lag, sync=sync, thin=thin)
    e.run(nsamp, nburn, pin, lik, par, incov)
    st = e.state()
    h = e.history()
    # accept pattern of the main phase from the history: a row changed iff accepted
    same_state = np.all(np.isclose(h[:, :, :d], o["rows"][:, :, :d], rtol=1e-7, atol=1e-9), axis=-1)
    print("rows agreeing with the oracle: %.5f" % same_state.mean())
    assert same_state.mean() > 0.999, "trajectories diverged: %.4f agree" % same_state.mean()
    # log-likelihood column of the rows whose state agrees: the kernels' table-driven fp64 math (and the
    # one-exponential form of DualGaussian) against the host libm evaluation of the reference's formula
    ll, lo = h[:, :, d][same_state], o["rows"][:, :, d][same_state]
    fin = np.isfinite(lo)
    assert np.array_equal(np.isfinite(ll), fin)
    assert np.allclose(ll[fin], lo[fin], rtol=1e-7, atol=1e-9)
    tight = np.isclose(h[:, :, :d], o["rows"][:, :, :d], rtol=0, atol=0).all(axis=-1) & same_state   # bit-equal states
    if tight.any():
        assert _close(h[:, :, d][tight], o["rows"][:, :, d][tight], rtol=1e-12, atol=1e-13)
    assert np.allclose(st["p"], o["p"], rtol=1e-6, atol=1e-8) or same_state[-1].mean() > 0.995
    assert np.allclose(e.factor(), o["cov"]), "global burn-in tuning differs"
    s = e.stats()
    assert abs(s["accepted"] - int(o["counts"][0])) <= max(2, nsamp * N // 5000)
    assert o["remote"][nburn:].any(), "test must exercise the remote branch"
    # the kernels count the remote chain-steps and the candidates their rejection loops tried
    # (mcpar.cc:331-409); trajectories that diverge by an ulp may shift the candidate count slightly
    assert s["remote_steps"] == int(o["remote"][nburn:].sum())
    ri = int(o["remote_iters"][0])
    assert abs(s["remote_iterations"] - ri) <= max(2, ri // 200), (s["remote_iterations"], ri)
    if rmode == 1:
        assert s["remote_iterations"] == s["remote_steps"]       # one candidate per remote step: no rejection loop
    # (the exact-path fallbacks of the fp32-bounded tests are counted in s["exact_fallbacks"]: in a run this short
    # they are dominated by the first windows' narrow pools, sigma ~ 1e-7; the rate that matters is asserted at
    # full size in test_full_size_stationarity and printed by bench.py)
    assert s["exact_fallbacks"] >= 0
    pool = e.musig()
    assert np.allclose(pool, o["pool"], rtol=1e-6, atol=1e-8) or same_state[-1].mean() > 0.995
    # every kept row and the final state: ly is log L of the row's own point, within the kernel's rounding bound
    # (a kernel that stores x' with the old log-likelihood, or a partly live lane group that writes stale values, fails)
    x = np.concatenate([h[:, :, :d].reshape(-1, d), st["p"]])
    y = np.concatenate([h[:, :, d].ravel(), st["ly"]])
    L, S, c = km.loglik_ld(lik, d, x, par, expanded)
    inf = np.isinf(L)
    assert np.array_equal(np.isinf(y), inf) and np.all(y[inf] == L[inf])
    ratio = (np.abs(y[~inf] - L[~inf]) / (c * km.EPS * S[~inf])).astype(float)
    print("max |ly - L| / (c eps S) = %.3g  (c = %d, max S = %.3g)" % (ratio.max(), c, float(S.max())))
    assert ratio.max() <= 1.0, "log-likelihood off its row by %.3g times its rounding bound" % ratio.max()
    e.close()


# ---------------------------------------------------------------- sharding
def test_two_sharded_engines_equal_one_engine():
    """Chains sharded over two engines (host-driven exchange + summed tuning counters, the
    protocol mcpar_b200/sharded.py runs over NCCL) reproduce the single-engine run bit for
    bit: Philox is keyed on the global chain id, tuning is global, the pool is all-gathered."""
    import torch
    _two_vs_one(32)


def test_two_sharded_engines_equal_one_engine_jobwide_coin():
    _two_vs_one(0)


def test_two_sharded_engines_equal_one_engine_at_full_size():
    """BASELINE configs[1] at its full size (DualGaussian, 2^20 chains, PLOCAL 0.9, pool 16, job-wide
    coin, thin 10): sharding invariance is the size-independent property -- two engines of 2^19 chains
    reproduce the 2^20-chain engine bit for bit (states, moments, kept rows, tuned factor)."""
    _two_vs_one(0, N=1 << 20, lik="dualgaussian", par=[5.0], nburn=110, nsamp=40, pl=0.9, thin=10)


def _two_vs_one(cg, N=512, lik="rosenbrock1", par=None, nburn=130, nsamp=60, pl=0.7, thin=1):
    import torch
    eng = _engine()
    d, M = 2, 16
    kept = (nsamp + thin - 1) // thin
    pin = tiled_pinit(N, d)
    one = eng.Engine(d, N, mode="normal", pool_m=M, pl=pl, coin_group=cg, thin=thin, history_steps=kept)
    one.run(nsamp, nburn, pin, lik, par)
    ref_state, ref_hist, ref_factor = one.state(), one.history(), one.factor()
    one.close()

    half = N // 2
    es = [eng.Engine(d, half, mode="normal", nchain_total=N, chain0=r * half, pool_m=M, pl=pl, coin_group=cg, thin=thin,
                     history_steps=kept) for r in range(2)]
    for r, e in enumerate(es):
        e.set_likelihood(lik, par); e.set_covariance(None); e.set_state(pin[r * half:(r + 1) * half])
    dev = torch.device("cuda", 0)
    cnts = [torch.as_tensor(e.tuning_counters(), device=dev) for e in es]
    left = nburn
    while left > 0:                                              # burn-in with all-reduced counters
        done = [e.burnin_some(left) for e in es]
        assert done[0] == done[1]
        left -= done[0][0]
        if done[0][1]:
            [e.synchronize() for e in es]
            tot = cnts[0] + cnts[1]
            cnts[0].copy_(tot); cnts[1].copy_(tot)
            torch.cuda.synchronize()
            [e.tune() for e in es]
    [e.sample_begin(nsamp) for e in es]
    t = 0
    while t < nsamp:
        n = min(10, nsamp - t)
        [e.sample(n) for e in es]
        t += n
        if t % 10 == 0:                                          # "all-gather": copy each owner's slice to the peer
            [e.synchronize() for e in es]
            bufs = [e.exchange_begin() for e in es]
            views = [torch.as_tensor(b[0], device=dev) for b in bufs]
            for r in range(2):
                off, own = bufs[r][1] // 8, bufs[r][2] // 8
                views[1 - r][off:off + own].copy_(views[r][off:off + own])
            torch.cuda.synchronize()
            [e.exchange_end() for e in es]
    [e.synchronize() for e in es]
    st = [e.state() for e in es]
    assert np.array_equal(np.concatenate([s["p"] for s in st]), ref_state["p"])
    assert np.array_equal(np.concatenate([s["psum2"] for s in st]), ref_state["psum2"])
    assert np.array_equal(np.concatenate([e.history() for e in es], axis=1), ref_hist)
    assert np.array_equal(es[0].factor(), ref_factor) and np.array_equal(es[1].factor(), ref_factor)
    [e.close() for e in es]


# ---------------------------------------------------------------- statistics (normal mode)
def _stationary_rosenbrock(N, rng):
    x = rng.normal(1.0, np.sqrt(0.5), N)
    y = rng.normal(x * x, np.sqrt(1.0 / 200.0))
    return np.stack([x, y], axis=1)


def test_posterior_moments_local_only_rosenbrock():
    """PLOCAL = 1, chains started from exact draws of the target: the MH kernel must leave the
    Rosenbrock posterior invariant -- analytic moments x ~ N(1,1/2), E y = 1.5, Var y = 2.505,
    Cov = 1 (SURVEY.md section 4) hold at every later time."""
    eng = _engine()
    N = 1 << 16
    pin = _stationary_rosenbrock(N, np.random.default_rng(2))
    e = eng.Engine(2, N, mode="normal", pl=1.0, thin=250, history_steps=8)
    e.run(2000, 500, pin, "rosenbrock1")
    for k in (3, 7):
        r = e.history()[k]
        se = 1.0 / np.sqrt(N)
        assert abs(r[:, 0].mean() - 1.0) < 5 * se * np.sqrt(0.5) and abs(r[:, 1].mean() - 1.5) < 5 * se * np.sqrt(2.505)
        assert abs(r[:, 0].var() - 0.5) < 0.02 and abs(r[:, 1].var() - 2.505) < 0.12
        assert abs(np.cov(r[:, 0], r[:, 1])[0, 1] - 1.0) < 0.05
    mean, cov = e.moments()                                      # device reduction agrees with the host one
    hh = e.history().reshape(-1, 3)
    assert np.allclose(mean, hh[:, :2].mean(0), rtol=1e-9) and np.allclose(cov, np.cov(hh[:, :2].T, bias=True), rtol=1e-7)
    e.close()


def test_ks_local_only_dualgaussian_marginal():
    """PLOCAL = 1, stationary start: each chain's marginal stays the mixture
    5/6 N(0,1) + 1/6 N(5,1) (rosenbrock.cc:69-75 with w = 5); chains are independent, so a
    one-sample KS against the mixture CDF applies (p > 0.01, north star)."""
    from scipy import stats
    eng = _engine()
    N = 1 << 14
    rng = np.random.default_rng(3)
    comp = rng.random(N) < 1.0 / 6.0
    pin = rng.standard_normal((N, 2)) + 5.0 * comp[:, None]
    e = eng.Engine(2, N, mode="normal", pl=1.0, thin=500, history_steps=3)
    e.run(1500, 500, pin, "dualgaussian", [5.0])
    cdf = lambda v: (5.0 * stats.norm.cdf(v) + stats.norm.cdf(v - 5.0)) / 6.0
    h = e.history()[2]
    assert stats.kstest(h[:, 0], cdf).pvalue > 0.01 and stats.kstest(h[:, 1], cdf).pvalue > 0.01
    assert abs((h[:, 0] > 2.5).mean() - 1.0 / 6.0) < 0.02
    e.close()


@pytest.mark.parametrize("pl,rmode,M", [(1.0, 0, 16), (0.9, 0, 16), (0.9, 1, 16), (0.9, 1, 256)])
def test_full_size_stationarity(pl, rmode, M):
    """BASELINE configs[1] at full size (2^20 chains, pool 16, job-wide coin), chains started from exact
    draws of the target 5/6 N(0,I) + 1/6 N((5,5),I).
    PLOCAL 1: Metropolis steps leave the target invariant exactly; with 2^20 chains the mean is pinned to
    +-0.01 and the mass of the small mode to +-0.002 (5 standard errors), and a KS test applies.
    PLOCAL 0.9: the reference's remote proposal is an independence proposal from the max-mixture of the
    pool corrected by cfac = max_i Q_i(x) / max_i Q_i(x') with UNNORMALISED Q_i = exp(-1/2 sum (x-mu)^2/sig^2)
    (src/mcpar.cc:367-390, :412-439): the correction is exact only when all components have the same
    widths, so the reference's own algorithm carries a small bias that 2^20 chains resolve.  The engine
    reproduces that algorithm (it matches the oracle trajectory for trajectory at small sizes), so here
    only coarse bounds are asserted and the deviation is printed.
    PLOCAL 0.9, remote mode 1 (sum-mixture proposal, NORMALISED components, Hastings factor q(x)/q(x')): an exact
    independence sampler whatever the pool holds, so the full bar of the PLOCAL 1 case applies -- mean, mode
    mass and KS within 5 standard errors at 2^20 chains (the north star's normal-mode bar)."""
    from scipy import stats
    eng = _engine()
    N = 1 << 20
    rng = np.random.default_rng(11)
    comp = rng.random(N) < 1.0 / 6.0
    pin = rng.standard_normal((N, 2)) + 5.0 * comp[:, None]
    e = eng.Engine(2, N, mode="normal", pl=pl, pool_m=M, coin_group=0, thin=100, history_steps=3, remote_mode=rmode)
    e.run(300, 100, pin, "dualgaussian", [5.0])
    s = e.stats()
    assert (s["remote_steps"] > 20 * N) == (pl < 1.0)
    exact = pl >= 1.0 or rmode == 1
    if pl < 1.0:
        print("remote mode %d, M = %d: %.2f candidates per remote step, exact-path fallbacks %.2e of them"
              % (rmode, M, s["remote_iterations"] / s["remote_steps"], s["exact_fallbacks"] / s["remote_iterations"]))
        assert s["exact_fallbacks"] < 0.02 * s["remote_iterations"]
    cdf = lambda v: (5.0 * stats.norm.cdf(v) + stats.norm.cdf(v - 5.0)) / 6.0
    var = 1.0 + 25.0 * (5.0 / 36.0)
    for k in (1, 2):
        h = e.history()[k]
        dm = [h[:, i].mean() - 5.0 / 6.0 for i in (0, 1)]
        pright = (5.0 * stats.norm.sf(2.5) + stats.norm.cdf(2.5)) / 6.0       # P(x0 > 2.5) under the mixture: 0.1708
        df = (h[:, 0] > 2.5).mean() - pright
        print("pl=%g mode %d M=%d kept step %d: mean - 5/6 = %+.5f %+.5f   P(x0 > 2.5) - exact = %+.5f" % (pl, rmode, M, k, dm[0], dm[1], df))
        if exact:
            for i in (0, 1):
                assert abs(dm[i]) < 5.0 * np.sqrt(var / N)
                assert abs(h[:, i].var() - var) < 0.03
                # KS over all 2^20 chains (four tests in this case: family-wise 0.4 %) and over the p-values of the 16 stride-16
                # sub-samples, which a correct sampler leaves uniform.  A single stride-64 sub-sample is not a sound probe: runs that
                # share the Philox streams of their local steps share their fluctuations (profiles/r02_ks_diag.md).
                assert stats.kstest(h[:, i], cdf).pvalue > 1.0e-3
                sub = [stats.kstest(h[j::16, i], cdf).pvalue for j in range(16)]
                assert stats.kstest(sub, "uniform").pvalue > 1.0e-3
            assert abs(df) < 5.0 * np.sqrt(pright * (1.0 - pright) / N)
        else:                                  # measured: profiles/r02_bias_curve.md (the reference algorithm's own drift)
            assert max(abs(dm[0]), abs(dm[1])) < 0.25 and abs(df) < 0.05
        assert abs(((h[:, 0] > 2.5) != (h[:, 1] > 2.5)).mean()) < 0.02      # both coordinates sit in the same mode
    e.close()


def test_remote_proposals_match_reference_distribution():
    """PLOCAL = 0.9 (remote proposals on): the engine's normal mode against the reference's
    algorithm (oracle/mh_oracle.c, which test_oracle.py pins bit for bit to the reference's own
    outputs stored in tests/golden/) on the reference's own launch shape (4 ranks x 4 chains,
    all 16 chains in the mixture), the reference side on seeded replay streams.  Chains of one
    run are coupled through the exchange, so the unit of comparison is the RUN: per-run
    posterior summaries over 48 independent seeds each, two-sample KS at p > 0.01."""
    from scipy import stats
    eng = _engine()
    R, C, d, nburn, nsamp, nrep = 4, 4, 2, 300, 1500, 48
    pin = tiled_pinit(C, d)
    ref_stat, gpu_stat = [], []
    for k in range(nrep):
        Z, U, I = make_streams(R, C, d, nburn + nsamp, 1000 + k)
        o = mh.run_replay("dualgaussian", d, C, R, nsamp, nburn, pin, Z, U, I, par=[5.0])
        assert o["used"][:, 3].sum() == 0                                # no stream overrun
        rows = o["rows"].reshape(-1, 3)
        ref_stat.append((rows[:, 0].mean(), (rows[:, 0] > 2.5).mean(), rows[:, 0].var()))
        e = eng.Engine(d, R * C, mode="normal", coin_group=4, pool_m=0, seed=5000 + k, history_steps=nsamp)
        e.run(nsamp, nburn, np.tile(pin, (R, 1)), "dualgaussian", [5.0])
        rows = e.history().reshape(-1, 3)
        gpu_stat.append((rows[:, 0].mean(), (rows[:, 0] > 2.5).mean(), rows[:, 0].var()))
        e.close()
    ref_stat, gpu_stat = np.array(ref_stat), np.array(gpu_stat)
    for j in range(3):
        assert stats.ks_2samp(ref_stat[:, j], gpu_stat[:, j]).pvalue > 0.01, (j, ref_stat[:, j].mean(), gpu_stat[:, j].mean())


# ---------------------------------------------------------------- edge cases
def test_far_start_is_stuck_as_in_the_reference():
    """DualGaussian has no log-sum-exp guard (rosenbrock.cc:75): far from both modes logL = -inf,
    exp(-inf - -inf) = NaN, `acpt < NaN` is false, so such a chain rejects until a proposal lands
    where logL is finite.  Verification mode and the production kernel must both follow that."""
    eng = _engine()
    d, C, R, nburn, nsamp = 2, 4, 1, 60, 40
    pin = np.array([[60.0, 60.0], [0.0, 0.0], [-45.0, 50.0], [2.0, 2.0]])
    Z, U, I = make_streams(R, C, d, nburn + nsamp, 21)
    o = mh.run_replay("dualgaussian", d, C, R, nsamp, nburn, pin, Z, U, I, par=[5.0], trace=True)
    # chain 0 cannot move during burn-in (local proposals only); a remote proposal may free it later
    assert np.isinf(o["trace"]["pre_ly"][0, 0, 0]) and not o["accept"][0, :nburn, 0].any()
    e = eng.Engine(d, C, mode="verify", chains_per_rank=C, trace=nburn + nsamp, history_steps=nsamp)
    e.set_likelihood("dualgaussian", [5.0]); e.set_state(pin); e.set_streams(0, Z[0], U[0], I[0])
    e.burnin(nburn); e.sample_begin(nsamp); e.sample(nsamp); e.synchronize()
    tr = e.trace(0, nburn + nsamp)
    assert np.array_equal(tr["accept"].astype(bool), o["accept"][0])
    assert np.array_equal(e.state()["p"], o["p"][0])
    e.close()
    oc = mh.run_counter("dualgaussian", d, 64, 30, 60, np.tile(pin, (16, 1)), par=[5.0], pool_m=8, coin_group=0)
    e = eng.Engine(d, 64, mode="normal", pool_m=8, coin_group=0, history_steps=30)
    e.run(30, 60, np.tile(pin, (16, 1)), "dualgaussian", [5.0])
    st = e.state()
    assert np.allclose(st["p"], oc["p"], rtol=1e-7, atol=1e-9)
    assert np.array_equal(np.isinf(st["ly"]), np.isinf(oc["ly"]))
    e.close()


@pytest.mark.parametrize("nburn,nsamp", [(0, 0), (0, 7), (37, 0), (51, 3), (52, 1)])
def test_degenerate_lengths(nburn, nsamp):
    """Empty phases and runs that end exactly on / next to a tuning boundary (isamp = 51)."""
    eng = _engine()
    d, C, R = 2, 4, 2
    pin = tiled_pinit(C, d)
    Z, U, I = make_streams(R, C, d, nburn + nsamp + 1, 31)
    o = mh.run_replay("rosenbrock1", d, C, R, nsamp, nburn, pin, Z, U, I, trace=True)
    e = eng.Engine(d, R * C, mode="verify", chains_per_rank=C, history_steps=max(nsamp, 1))
    e.set_likelihood("rosenbrock1"); e.set_state(np.tile(pin, (R, 1)))
    for r in range(R):
        e.set_streams(r, Z[r], U[r], I[r])
    e.burnin(nburn); e.sample_begin(nsamp); e.sample(nsamp); e.synchronize()
    st = e.state()
    assert np.array_equal(st["p"].reshape(R, C, d), o["p"]) and np.array_equal(st["ly"].reshape(R, C), o["ly"])
    for r in range(R):
        assert np.array_equal(e.factor(r), o["cov"][r])
    assert e.stats()["history_rows"] == nsamp * R * C
    e.close()
    en = eng.Engine(d, 96, mode="normal", coin_group=0, pool_m=8, history_steps=max(nsamp, 1))
    en.run(nsamp, nburn, tiled_pinit(96, d), "rosenbrock1")
    oc = mh.run_counter("rosenbrock1", d, 96, nsamp, nburn, tiled_pinit(96, d), pool_m=8, coin_group=0)
    assert np.allclose(en.state()["p"], oc["p"], rtol=1e-9, atol=1e-12) and np.array_equal(en.factor(), oc["cov"])
    en.close()


def test_single_chain_and_large_rank():
    """C = 1 (one thread per CTA) and C = 1024 (the verify kernel's maximum CTA)."""
    eng = _engine()
    for C, nburn, nsamp in [(1, 120, 40), (1024, 60, 12)]:
        pin = tiled_pinit(C, 2)
        Z, U, I = make_streams(1, C, 2, nburn + nsamp, 41, mult=12)
        o = mh.run_replay("rosenbrock1", 2, C, 1, nsamp, nburn, pin, Z, U, I, pl=0.5, trace=True)
        e = eng.Engine(2, C, mode="verify", chains_per_rank=C, pl=0.5, trace=nburn + nsamp, history_steps=nsamp)
        e.set_likelihood("rosenbrock1"); e.set_state(pin); e.set_streams(0, Z[0], U[0], I[0])
        e.burnin(nburn); e.sample_begin(nsamp); e.sample(nsamp); e.synchronize()
        tr = e.trace(0, nburn + nsamp)
        assert np.array_equal(tr["accept"].astype(bool), o["accept"][0])
        assert np.array_equal(tr["cursors"], o["used"][0][:3])
        assert np.array_equal(e.state()["p"], o["p"][0]) and np.array_equal(e.musig(0), o["musig"][0])
        e.close()


def test_qriguess_matches_oracle():
    """mcutil::qriguess on the device (Sobol points in a box, rank skip-ahead, mcutil.cc:16-31)."""
    eng = _engine()
    plo, phi = [0.0, -1.0, 2.0, 10.0, -3.0], [1.0, 1.0, 4.0, 11.0, 3.0]
    for rank, npset in [(0, 1000), (3, 257), (1, 1)]:
        assert np.array_equal(eng.qriguess(rank, npset, 5, plo, phi), mh.qriguess(rank, npset, 5, plo, phi))
    with pytest.raises(eng.McgpuError):
        eng.qriguess(0, 4, 65, [0] * 65, [1] * 65)
    assert np.array_equal(eng.qriguess(2, 300, 40, [0] * 40, [1] * 40), mh.qriguess(2, 300, 40, [0] * 40, [1] * 40))


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_host_sink_receives_the_history(dtype):
    """mcgpu_history_attach_host[_f32]: rows drained on the side stream during sampling equal a
    read-back (fp32 sink: the read-back narrowed to the reference MCout's element type)."""
    eng = _engine()
    N, nsamp, thin = 4096, 120, 4
    e = eng.Engine(2, N, mode="normal", coin_group=0, pool_m=8, thin=thin, history_steps=nsamp // thin)
    e.set_likelihood("dualgaussian", [5.0]); e.set_covariance(None); e.set_state(tiled_pinit(N, 2))
    e.burnin(60)
    sink = np.full((nsamp // thin, N, 3), np.nan, dtype=dtype)
    e.attach_host_sink(sink)
    e.sample_begin(nsamp)
    for _ in range(nsamp // 10):
        e.sample(10)
    e.synchronize()
    assert np.array_equal(sink, e.history().astype(dtype))
    e.attach_host_sink(None)
    e.close()


def test_api_misuse_is_reported():
    eng = _engine()
    e = eng.Engine(2, 64, mode="normal", history_steps=40)
    with pytest.raises(eng.McgpuError, match="ESTATE"):
        e.set_state(np.zeros((64, 2)))                 # likelihood first
    e.set_likelihood("rosenbrock1")
    with pytest.raises(eng.McgpuError, match="ESTATE"):
        e.burnin(10)                                   # state first
    e.set_state(np.zeros((64, 2)))
    with pytest.raises(eng.McgpuError, match="ESTATE"):
        e.sample(5)                                    # sample_begin first
    e.sample_begin(40)
    with pytest.raises(eng.McgpuError, match="EINVAL"):
        e.sample(41)
    with pytest.raises(eng.McgpuError, match="EINVAL"):
        e.set_likelihood("rosenbrock2")                # couples neighbouring chains: verify mode only
    e.close()
    with pytest.raises(eng.McgpuError, match="EINVAL"):
        eng.Engine(3, 64, mode="normal").set_likelihood("rosenbrock1")    # odd n (rosenbrock.hh:13-16)
    with pytest.raises(eng.McgpuError, match="EINVAL"):
        eng.Engine(2, 64, mode="normal", coin_group=3)


# ---------------------------------------------------------------- history ring, Sobol start
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_history_ring_drains_a_long_run(dtype):
    """history_steps smaller than the run's kept steps: the device keeps a RING and every row still reaches the
    host sink (the drain of a ring row is awaited before the row is overwritten); a full-history engine is the
    reference.  history() then returns the last history_steps kept steps."""
    eng = _engine()
    N, nsamp, thin, cap = 2048, 400, 2, 12
    pin = tiled_pinit(N, 2)
    full = eng.Engine(2, N, mode="normal", coin_group=0, pool_m=8, thin=thin, history_steps=nsamp // thin)
    full.run(nsamp, 60, pin, "dualgaussian", [5.0])
    ref = full.history(); rmean, rcov = full.moments(); rml = full.maxlike()
    full.close()
    e = eng.Engine(2, N, mode="normal", coin_group=0, pool_m=8, thin=thin, history_steps=cap)
    e.set_likelihood("dualgaussian", [5.0]); e.set_covariance(None); e.set_state(pin)
    e.burnin(60)
    sink = np.full((nsamp // thin, N, 3), np.nan, dtype=dtype)
    e.attach_host_sink(sink)
    e.sample_begin(nsamp)
    for n in (7, 13, 180, 200):                       # uneven pieces, several windows per call
        e.sample(n)
    e.synchronize()
    assert np.array_equal(sink, ref.astype(dtype))
    tail = e.history()
    assert tail.shape[0] == cap and np.array_equal(tail, ref[-cap:])
    assert np.array_equal(e.history(first=nsamp // thin - 5, count=5), ref[-5:])
    with pytest.raises(eng.McgpuError, match="no longer on the device"):
        e.history(first=0, count=1)
    mean, cov = e.moments()                            # device reductions see the rows the ring still holds
    hh = ref[-cap:].reshape(-1, 3)
    assert np.allclose(mean, hh[:, :2].mean(0), rtol=1e-9) and np.allclose(cov, np.cov(hh[:, :2].T, bias=True), rtol=1e-7)
    assert e.maxlike()[1] == hh[:, 2].max()
    e.attach_host_sink(None)
    e.close()


def test_ring_without_sink_keeps_the_last_rows():
    eng = _engine()
    N, nsamp = 512, 95
    pin = tiled_pinit(N, 2)
    full = eng.Engine(2, N, mode="normal", coin_group=32, pool_m=8, history_steps=nsamp)
    full.run(nsamp, 30, pin, "rosenbrock1")
    ref = full.history()
    full.close()
    e = eng.Engine(2, N, mode="normal", coin_group=32, pool_m=8, history_steps=7)
    e.run(nsamp, 30, pin, "rosenbrock1")
    assert np.array_equal(e.history(), ref[-7:])
    assert e.stats()["history_rows"] == nsamp * N
    e.close()


@pytest.mark.parametrize("d,N,cg,lik", [(64, 1 << 20, 0, "rosenbrock1"), (16, 4096, 32, "rosenbrock1"), (2, 100000, 0, "dualgaussian")])
def test_set_state_sobol_matches_oracle_qriguess(d, N, cg, lik):
    """mcgpu_set_state_sobol: qriguess (mcutil.cc:16-31) straight into the engine's state, bit for bit against
    the oracle at 2^20 x 64 (BASELINE config 4's shape); a sharded engine continues the sequence at chain0."""
    eng = _engine()
    rng = np.random.default_rng(5)
    plo = rng.uniform(-3, 0, d); phi = plo + rng.uniform(0.5, 4, d)
    want = mh.qriguess(0, N, d, plo, phi)
    e = eng.Engine(d, N, mode="normal", coin_group=cg, pool_m=16, history_steps=0)
    e.set_likelihood(lik, [5.0] if lik == "dualgaussian" else None)
    e.set_state_sobol(plo, phi)
    st = e.state()
    assert np.array_equal(st["p"], want)
    assert np.allclose(st["ly"][:1000], mh.loglik(lik, d, want[:1000], [5.0] if lik == "dualgaussian" else None), rtol=1e-12, atol=1e-12)
    e.close()
    half = N // 2 // 32 * 32
    e2 = eng.Engine(d, N - half, mode="normal", nchain_total=N, chain0=half, coin_group=cg, pool_m=16, history_steps=0)
    e2.set_likelihood(lik, [5.0] if lik == "dualgaussian" else None)
    e2.set_state_sobol(plo, phi)
    assert np.array_equal(e2.state()["p"], want[half:])
    e2.close()
    if d <= 16:
        assert np.array_equal(eng.qriguess(1, 257, d, plo, phi), mh.qriguess(1, 257, d, plo, phi))


def test_second_run_on_one_engine_is_reproducible():
    """mcgpu_set_state starts a fresh run: tuning counters and the pending-boundary flag are reset (ADVICE r1)."""
    eng = _engine()
    pin = tiled_pinit(256, 2)
    e = eng.Engine(2, 256, mode="normal", coin_group=0, pool_m=8, history_steps=20)
    e.run(20, 77, pin, "rosenbrock1")                  # ends between two tuning boundaries, counters half full
    e.set_covariance(None); e.set_state(pin)
    e.burnin(120); e.sample_begin(20); e.sample(20); e.synchronize()
    second = (e.state()["p"], e.factor())
    e.close()
    f = eng.Engine(2, 256, mode="normal", coin_group=0, pool_m=8, history_steps=20)
    f.run(20, 120, pin, "rosenbrock1")
    assert np.array_equal(second[0], f.state()["p"]) and np.array_equal(second[1], f.factor())
    f.close()
