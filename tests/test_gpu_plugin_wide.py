"""Wide device likelihood plugins (MCGPU_PLUGIN_WIDE, include/mcgpu_plugin.cuh): a user functor that returns one share
of the log-likelihood per lane, run inside the wide step kernels (d = 8, 16, 32, 64, d/2 lanes per chain).  The
restated-Rosenbrock plugin is the built-in wide Rosenbrock1 typed in again, so a run with it must equal the built-in
run bit for bit, apart from the last bits of the initial log-likelihoods (the built-in takes them from the exact unit
in serial order, the plugin from its group-ordered batched evaluation); the logistic-regression plugin (d = 32) must
follow the host-callback path with the same model written in numpy."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import tiled_pinit

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STATS = ("accepted", "remote_steps", "remote_iterations", "exact_fallbacks")


def _shipped(name):
    from mcpar_b200 import plugin
    path = plugin.shipped(name)
    assert os.path.exists(path), "%s is built by build(): run the package build first" % path
    return path


def _rosen(d, tmp_dir=None):
    """The restated wide Rosenbrock at d: shipped at 16 and 64, built on demand at 8 and 32."""
    if d in (16, 64):
        return _shipped("rosen1_wide_d%d.cubin" % d)
    from mcpar_b200 import plugin
    return plugin.build(os.path.join(ROOT, "tests", "plugins", "rosen1_wide.cuh"), nparam=d,
                        out=os.path.join(str(tmp_dir), "rosen1_wide_d%d.cubin" % d))


def logistic_wide_data(n=64, seed=7):
    """par = [n, 1/sigma^2_prior, X (n x 31), y (n)] of examples/likelihoods/logistic_wide.cuh, and the parts."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, 31)) * 0.5
    beta = rng.normal(0.0, 0.5, 32)
    y = (rng.random(n) < 1.0 / (1.0 + np.exp(-(beta[0] + X @ beta[1:])))).astype(np.float64)
    prec = 0.25
    return np.concatenate([[n, prec], X.ravel(), y]), X, y, prec


def logistic_wide_np(B, X, y, prec):
    B = np.asarray(B, dtype=np.float64).reshape(-1, 32)
    eta = B[:, :1] + B[:, 1:] @ X.T
    sp = np.maximum(eta, 0.0) + np.log1p(np.exp(-np.abs(eta)))
    return (y * eta - sp).sum(axis=1) - 0.5 * prec * (B * B).sum(axis=1)


def _collect(e):
    s = e.stats()
    out = dict(hist=e.history(), factor=e.factor(), **e.state())
    out.update({k: s[k] for k in STATS})
    return out


def _run(d, N, lik, par=None, plugin=None, nburn=120, nsamp=80, scale=1.0, **kw):
    from mcpar_b200 import engine
    kw.setdefault("history_steps", nsamp)
    e = engine.Engine(d, N, **kw)
    e.run(nsamp, nburn, tiled_pinit(N, d) * scale, lik, par, plugin=plugin)
    out = _collect(e)
    e.close()
    return out


def _assert_same(a, b, d):
    """Bit for bit except the log-likelihoods, which may keep an initial value's last-bit difference."""
    for k in ("p", "mu", "sig", "psum2", "factor") + STATS:
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["hist"][:, :, :d], b["hist"][:, :, :d])
    np.testing.assert_allclose(a["ly"], b["ly"], rtol=1e-15, atol=0)
    np.testing.assert_allclose(a["hist"][:, :, d], b["hist"][:, :, d], rtol=1e-15, atol=0)


@pytest.mark.parametrize("d,mode,lag", [
    (8, 0, 0), (8, 1, 1),
    (16, 0, 1), (16, 1, 0),
    (32, 0, 0), (32, 1, 1),
    (64, 0, 1), (64, 1, 0),
])
def test_restated_wide_rosenbrock_matches_builtin(tmp_path, d, mode, lag):
    from mcpar_b200 import engine
    cubin = _rosen(d, tmp_path)
    N = 998                                       # ragged over CTAs and over the 2 or 4 chains of a lane group
    kw = dict(pool_m=16, pl=0.7, coin_group=0, remote_mode=mode, pool_lag=lag)
    a = _run(d, N, "rosenbrock1", **kw)
    b = _run(d, N, "plugin", plugin=cubin, **kw)
    assert a["remote_steps"] > 0
    _assert_same(a, b, d)
    # the batched evaluation is the step kernels' sum: bit for bit on the final states
    assert np.array_equal(engine.loglik("plugin", d, b["p"], plugin=cubin), b["ly"])


def test_logistic_wide_batched_evaluation():
    from mcpar_b200 import engine
    par, X, y, prec = logistic_wide_data()
    cubin = _shipped("logistic_wide.cubin")
    x = np.random.default_rng(5).normal(0.0, 0.5, (1001, 32))   # 1001: the last CTA is partly idle
    got = engine.loglik("plugin", 32, x, par, plugin=cubin)
    want = logistic_wide_np(x, X, y, prec)
    assert np.allclose(got, want, rtol=1e-12, atol=0.0), np.max(np.abs(got / want - 1))
    with pytest.raises(engine.McgpuError, match="EINVAL"):
        engine.loglik("plugin", 16, x[:, :16], par, plugin=cubin)


@pytest.mark.parametrize("mode", [0, 1])
def test_logistic_wide_follows_host_path(mode):
    from mcpar_b200 import engine
    par, X, y, prec = logistic_wide_data()
    cubin = _shipped("logistic_wide.cubin")
    d, N, nburn, nsamp = 32, 256, 110, 45
    pin = tiled_pinit(N, d) * 0.25
    kw = dict(pool_m=8, pl=0.7, coin_group=0, history_steps=nsamp, remote_mode=mode)
    e = engine.Engine(d, N, **kw)
    e.run(nsamp, nburn, pin, "plugin", par, plugin=cubin)
    a = _collect(e)
    e.close()
    h = engine.Engine(d, N, **kw)
    h.run_host(nsamp, nburn, pin, lambda x: logistic_wide_np(x, X, y, prec))
    b = _collect(h)
    h.close()
    same = np.all(np.isclose(a["hist"][:, :, :d], b["hist"][:, :, :d], rtol=1e-9, atol=1e-11), axis=-1)
    assert same.mean() >= 0.995, same.mean()
    assert np.array_equal(a["factor"], b["factor"]), "burn-in tuning differs"
    assert a["remote_steps"] == b["remote_steps"] > 0


_AUDIT_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
from conftest import tiled_pinit
from mcpar_b200 import engine
from test_gpu_plugin_wide import logistic_wide_data
par = logistic_wide_data()[0]
N, nsamp = 512, 60
e = engine.Engine(32, N, pool_m=16, pl=0.7, coin_group=0, history_steps=nsamp, remote_mode=int(sys.argv[4]))
e.run(nsamp, 100, tiled_pinit(N, 32) * 0.25, "plugin", par, plugin=sys.argv[2])
np.save(sys.argv[3], e.history())
"""


@pytest.mark.parametrize("mode", [0, 1])
def test_logistic_wide_audit_mode_is_bit_identical(tmp_path, mode):
    """MCGPU_EXACT_TESTS=1 settles every accept / rejection / Hastings-factor decision in fp64; the decisions, hence
    the histories, are the same.  The variable is read once per process, so each run gets a fresh interpreter."""
    cubin = _shipped("logistic_wide.cubin")
    out = {}
    for flag in ("0", "1"):
        f = str(tmp_path / ("h%s.npy" % flag))
        env = dict(os.environ, MCGPU_EXACT_TESTS=flag)
        r = subprocess.run([sys.executable, "-c", _AUDIT_CHILD, ROOT, cubin, f, str(mode)], env=env,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        out[flag] = np.load(f)
    assert np.array_equal(out["0"], out["1"])


@pytest.mark.parametrize("mode", [0, 1])
def test_wide_plugin_sharded_p2p_equals_single_engine(mode):
    from mcpar_b200 import engine as eng
    par = logistic_wide_data()[0]
    cubin = _shipped("logistic_wide.cubin")
    d, Cg, world, nburn, nsamp, sync = 32, 256, 2, 110, 50, 10
    N = Cg * world
    pin = tiled_pinit(N, d) * 0.25
    kw = dict(pool_m=16, pl=0.7, sync=sync, coin_group=0, history_steps=nsamp, remote_mode=mode)
    ndev = eng.device_count()
    es = [eng.Engine(d, Cg, nchain_total=N, chain0=r * Cg, device=r % ndev, **kw) for r in range(world)]
    for r, e in enumerate(es):
        e.set_likelihood("plugin", par, plugin=cubin); e.set_covariance(None); e.set_state(pin[r * Cg:(r + 1) * Cg])
    eng.p2p_attach_local(es)
    eng.burnin_group(es, nburn)
    for e in es:
        e.sample_begin(nsamp)
    for _ in range(nsamp // sync):
        eng.sample_group(es, sync)
    for e in es:
        e.synchronize()
    parts = [_collect(e) for e in es]
    for e in es:
        e.close()
    one = _run(d, N, "plugin", par, plugin=cubin, nburn=nburn, nsamp=nsamp, scale=0.25, **kw)
    assert one["remote_steps"] > 0
    assert np.array_equal(np.concatenate([p["hist"] for p in parts], axis=1), one["hist"])
    for k in ("p", "ly", "mu", "sig", "psum2"):
        assert np.array_equal(np.concatenate([p[k] for p in parts]), one[k]), k
    for p in parts:
        assert np.array_equal(p["factor"], one["factor"])
    for k in ("accepted", "remote_steps"):
        assert sum(p[k] for p in parts) == one[k], k


def test_wide_plugin_checkpoint_continues_bit_for_bit():
    from mcpar_b200 import engine as eng
    cubin = _shipped("rosen1_wide_d64.cubin")
    d, N, nburn, nsamp, cut = 64, 500, 120, 60, 30          # cut: an exchange-window boundary (sync = 10)
    pin = tiled_pinit(N, d)
    kw = dict(pool_m=16, pl=0.7, coin_group=0, history_steps=nsamp, remote_mode=1)
    ref = _run(d, N, "plugin", plugin=cubin, nburn=nburn, nsamp=nsamp, **kw)
    b = eng.Engine(d, N, **kw)
    b.set_likelihood("plugin", plugin=cubin); b.set_covariance(None); b.set_state(pin)
    b.burnin(nburn); b.sample_begin(nsamp); b.sample(cut)
    head = b.history()
    blob = b.checkpoint()
    b.close()
    c = eng.Engine(d, N, **kw)
    c.set_likelihood("plugin", plugin=cubin)
    c.restore(blob)
    c.sample(nsamp - cut); c.synchronize()
    st = c.state()
    for k in ("p", "ly", "mu", "sig", "psum2"):
        assert np.array_equal(st[k], ref[k]), k
    assert np.array_equal(head, ref["hist"][:cut]) and np.array_equal(c.history(first=cut), ref["hist"][cut:])
    assert np.array_equal(c.factor(), ref["factor"])
    s = c.stats()
    assert (s["accepted"], s["remote_steps"]) == (ref["accepted"], ref["remote_steps"]) and s["remote_steps"] > 0
    c.close()


def test_wide_plugin_sobol_start():
    from mcpar_b200 import engine as eng
    par = logistic_wide_data()[0]
    cubin = _shipped("logistic_wide.cubin")
    d, N = 32, 300
    e = eng.Engine(d, N, pool_m=16, pl=0.7, coin_group=0, history_steps=20)
    e.set_likelihood("plugin", par, plugin=cubin)
    e.set_state_sobol(-np.ones(d), np.ones(d))
    st = e.state()
    assert np.all(np.abs(st["p"]) <= 1.0) and np.unique(st["p"][:, 0]).size > N // 2
    assert np.array_equal(st["ly"], eng.loglik("plugin", d, st["p"], par, plugin=cubin))
    e.set_covariance(None); e.burnin(30); e.sample_begin(20); e.sample(20); e.synchronize()
    assert np.all(np.isfinite(e.state()["ly"]))
    e.close()


def test_wide_plugin_rejections_launch_nothing(tmp_path):
    from mcpar_b200 import engine as eng, plugin, build
    r16 = _shipped("rosen1_wide_d16.cubin")
    stale = plugin.build(os.path.join(ROOT, "tests", "plugins", "rosen1_wide.cuh"), nparam=16,
                         out=str(tmp_path / "stale.cubin"), stamp=build.kernel_stamp() ^ 1)
    cases = [
        (dict(coin_group=4), r16, "EINVAL.*coin_group = 0"),                    # wide kernels: job-wide coin only
        (dict(coin_group=0, nparam=64), r16, "EINVAL.*nparam = 16"),            # built for d = 16, engine has d = 64
        (dict(coin_group=0), stale, "EINVAL.*stamp"),                           # other kernel sources
        (dict(mode="verify", chains_per_rank=4), r16, "EINVAL.*NORMAL mode only"),
    ]
    for kw, path, msg in cases:
        d = kw.pop("nparam", 16)
        e = eng.Engine(d, 64, **kw)
        with pytest.raises(eng.McgpuError, match=msg):
            e.set_likelihood("plugin", plugin=path)
        assert e.stats()["kernel_launches"] == 0
        e.set_likelihood("rosenbrock1")                                          # the engine is still usable
        e.close()
    # state installed with a thread-per-chain likelihood (the d = 16 restated plugin with a job-wide coin), then a
    # wide plugin: the state layout would change
    e = eng.Engine(16, 64, coin_group=0, pool_m=8, pl=0.7)
    e.set_likelihood("plugin", plugin=_shipped("rosen1_restated_d16.cubin")); e.set_covariance(None)
    e.set_state(tiled_pinit(64, 16))
    n0 = e.stats()["kernel_launches"]
    with pytest.raises(eng.McgpuError, match="ESTATE"):
        e.set_likelihood("plugin", plugin=r16)
    assert e.stats()["kernel_launches"] == n0
    e.burnin(10); e.synchronize()                                                # still usable, with the old plugin
    assert e.stats()["kernel_launches"] > n0
    e.close()


@pytest.mark.parametrize("ngpu,mode", [(1, "0"), (2, "1"), (1, "refuse")])
def test_cpp_wide_device_plugin_through_mcpar(tmp_path, ngpu, mode):
    host = os.path.join(ROOT, "mcpar_b200", "host")
    exe = str(tmp_path / "plugin_wide_mcpar_check")
    subprocess.check_call(["/usr/bin/g++", "-std=c++11", "-O2", "-I", host, "-I", os.path.join(ROOT, "include"), "-o", exe,
                           os.path.join(ROOT, "tests", "plugin_wide_mcpar_check.cc"), "-L", os.path.join(ROOT, "mcpar_b200"),
                           "-lmcpar", "-lmcgpu", "-Wl,-rpath," + os.path.join(ROOT, "mcpar_b200")])
    r = subprocess.run([exe, _shipped("rosen1_wide_d16.cubin"), "16", str(ngpu), mode], cwd=tmp_path,
                       capture_output=True, text=True, timeout=300)
    if mode == "refuse":
        assert r.returncode == 3 and "coin_group = 0" in r.stderr, r.stdout + r.stderr
    else:
        assert r.returncode == 0 and r.stdout.startswith("ok "), r.stdout + r.stderr
