"""Device likelihood plugins (include/mcgpu_plugin.cuh, mcgpu_set_likelihood_plugin): a user functor compiled into
the production step kernels.  The restated-Rosenbrock plugin is the built-in Rosenbrock1 typed in again, so every run
with it must equal the built-in run bit for bit; the logistic-regression plugin (a model and a dimension no built-in
has) must follow the host-callback path with the same model written in numpy."""
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


def logistic_data(n=40, seed=3):
    """par = [n, 1/sigma^2_prior, X (n x 5), y (n)] of examples/likelihoods/logistic.cuh, and the parts."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, 5))
    beta = np.array([0.5, -1.0, 0.8, 0.0, 0.3, -0.5])
    y = (rng.random(n) < 1.0 / (1.0 + np.exp(-(beta[0] + X @ beta[1:])))).astype(np.float64)
    prec = 0.25
    return np.concatenate([[n, prec], X.ravel(), y]), X, y, prec


def logistic_np(B, X, y, prec):
    B = np.asarray(B, dtype=np.float64).reshape(-1, 6)
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


def _assert_same(a, b):
    for k in ("hist", "p", "ly", "mu", "sig", "psum2", "factor") + STATS:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("d,N,cg,mode,lag", [
    (2, 1000, 0, 0, 0),           # ragged N, job-wide coin: lean local / planned mixed kernels
    (2, 1000, 4, 1, 1),           # per-group coins, sum-mixture proposal, lagged pool
    (2, 256, 0, 1, 0),
    (2, 256, 4, 0, 1),
    (16, 256, 32, 0, 0),          # coin_group 32 keeps the built-in on the thread-per-chain kernel
    (16, 256, 32, 1, 1),
])
def test_restated_rosenbrock_is_bit_identical_to_builtin(d, N, cg, mode, lag):
    cubin = _shipped("rosen1_restated_d%d.cubin" % d)
    kw = dict(pool_m=16, pl=0.7, coin_group=cg, remote_mode=mode, pool_lag=lag)
    a = _run(d, N, "rosenbrock1", **kw)
    b = _run(d, N, "plugin", plugin=cubin, **kw)
    assert a["remote_steps"] > 0
    _assert_same(a, b)


@pytest.mark.parametrize("cg,mode,lag", [(0, 0, 0), (4, 1, 1)])
def test_logistic_plugin_follows_host_path(cg, mode, lag):
    from mcpar_b200 import engine
    par, X, y, prec = logistic_data()
    cubin = _shipped("logistic.cubin")
    d, N, nburn, nsamp = 6, 256, 110, 45
    pin = tiled_pinit(N, d) * 0.25
    kw = dict(pool_m=8, pl=0.7, coin_group=cg, history_steps=nsamp, remote_mode=mode, pool_lag=lag)
    e = engine.Engine(d, N, **kw)
    e.run(nsamp, nburn, pin, "plugin", par, plugin=cubin)
    a = _collect(e)
    e.close()
    h = engine.Engine(d, N, **kw)
    h.run_host(nsamp, nburn, pin, lambda x: logistic_np(x, X, y, prec))
    b = _collect(h)
    h.close()
    same = np.all(np.isclose(a["hist"][:, :, :d], b["hist"][:, :, :d], rtol=1e-9, atol=1e-11), axis=-1)
    assert same.mean() >= 0.995, same.mean()
    assert np.array_equal(a["factor"], b["factor"]), "burn-in tuning differs"
    assert a["remote_steps"] == b["remote_steps"] > 0


def test_logistic_plugin_batched_evaluation():
    from mcpar_b200 import engine
    par, X, y, prec = logistic_data()
    x = np.random.default_rng(5).normal(0.0, 1.5, (1000, 6))
    got = engine.loglik("plugin", 6, x, par, plugin=_shipped("logistic.cubin"))
    want = logistic_np(x, X, y, prec)
    assert np.allclose(got, want, rtol=1e-12, atol=0.0), np.max(np.abs(got / want - 1))
    with pytest.raises(ValueError):
        engine.loglik("plugin", 6, x, par)
    with pytest.raises(engine.McgpuError, match="EINVAL"):
        engine.loglik("plugin", 4, x[:, :4], par, plugin=_shipped("logistic.cubin"))


_AUDIT_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
from conftest import tiled_pinit
from mcpar_b200 import engine
from test_gpu_plugin import logistic_data
par = logistic_data()[0]
N, nsamp = 512, 60
e = engine.Engine(6, N, pool_m=16, pl=0.7, coin_group=0, history_steps=nsamp, remote_mode=int(sys.argv[4]))
e.run(nsamp, 100, tiled_pinit(N, 6) * 0.25, "plugin", par, plugin=sys.argv[2])
np.save(sys.argv[3], e.history())
"""


@pytest.mark.parametrize("mode", [0, 1])
def test_logistic_plugin_audit_mode_is_bit_identical(tmp_path, mode):
    """MCGPU_EXACT_TESTS=1 settles every accept / rejection test in fp64; the decisions, hence the histories, are
    the same.  The variable is read once per process, so each run gets a fresh interpreter."""
    cubin = _shipped("logistic.cubin")
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
def test_plugin_sharded_p2p_equals_single_engine(mode):
    from mcpar_b200 import engine as eng
    par = logistic_data()[0]
    cubin = _shipped("logistic.cubin")
    d, Cg, world, nburn, nsamp, sync = 6, 256, 2, 110, 50, 10
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
    assert np.array_equal(np.concatenate([p["hist"] for p in parts], axis=1), one["hist"])
    for k in ("p", "ly", "mu", "sig", "psum2"):
        assert np.array_equal(np.concatenate([p[k] for p in parts]), one[k]), k
    for p in parts:
        assert np.array_equal(p["factor"], one["factor"])
    for k in ("accepted", "remote_steps"):
        assert sum(p[k] for p in parts) == one[k], k


def test_plugin_checkpoint_continues_bit_for_bit():
    from mcpar_b200 import engine as eng
    par = logistic_data()[0]
    cubin = _shipped("logistic.cubin")
    d, N, nburn, nsamp, cut = 6, 500, 120, 60, 30          # cut: an exchange-window boundary (sync = 10)
    pin = tiled_pinit(N, d) * 0.25
    kw = dict(pool_m=16, pl=0.7, coin_group=8, history_steps=nsamp, remote_mode=1)
    ref = _run(d, N, "plugin", par, plugin=cubin, nburn=nburn, nsamp=nsamp, scale=0.25, **kw)
    b = eng.Engine(d, N, **kw)
    b.set_likelihood("plugin", par, plugin=cubin); b.set_covariance(None); b.set_state(pin)
    b.burnin(nburn); b.sample_begin(nsamp); b.sample(cut)
    head = b.history()
    blob = b.checkpoint()
    b.close()
    c = eng.Engine(d, N, **kw)
    c.set_likelihood("plugin", par, plugin=cubin)
    c.restore(blob)
    c.sample(nsamp - cut); c.synchronize()
    st = c.state()
    for k in ("p", "ly", "mu", "sig", "psum2"):
        assert np.array_equal(st[k], ref[k]), k
    assert np.array_equal(head, ref["hist"][:cut]) and np.array_equal(c.history(first=cut), ref["hist"][cut:])
    assert np.array_equal(c.factor(), ref["factor"])
    s = c.stats()
    assert (s["accepted"], s["remote_steps"]) == (ref["accepted"], ref["remote_steps"])
    c.close()


def test_plugin_rejections_launch_nothing(tmp_path):
    from mcpar_b200 import engine as eng, plugin, build
    logi = _shipped("logistic.cubin")
    other = plugin.build(os.path.join(ROOT, "tests", "plugins", "rosen1_restated.cuh"), nparam=4,
                         out=str(tmp_path / "stale.cubin"), stamp=build.kernel_stamp() ^ 1)
    cases = [
        (dict(nparam=4), str(tmp_path / "missing.cubin"), "cannot open"),
        (dict(nparam=4), logi, "nparam = 6"),                        # built for d = 6, engine has d = 4
        (dict(nparam=4), other, "stamp"),                            # other kernel sources
        (dict(nparam=4, mode="verify", chains_per_rank=4), logi, "NORMAL mode only"),
        (dict(nparam=4, mode="replay_local"), logi, "NORMAL mode only"),
    ]
    for kw, path, msg in cases:
        d = kw.pop("nparam")
        e = eng.Engine(d, 64, **kw)
        with pytest.raises(eng.McgpuError, match="EINVAL.*" + msg):
            e.set_likelihood("plugin", [1.0], plugin=path)
        assert e.stats()["kernel_launches"] == 0
        e.set_likelihood("rosenbrock1")                              # the engine is still usable
        e.close()
    with pytest.raises(ValueError):
        eng.Engine(2, 64).set_likelihood("plugin")


@pytest.mark.parametrize("ngpu,mode", [(1, 0), (2, 0), (2, 1)])
def test_cpp_device_plugin_through_mcpar(tmp_path, ngpu, mode):
    host = os.path.join(ROOT, "mcpar_b200", "host")
    exe = str(tmp_path / "plugin_mcpar_check")
    subprocess.check_call(["/usr/bin/g++", "-std=c++11", "-O2", "-I", host, "-I", os.path.join(ROOT, "include"), "-o", exe,
                           os.path.join(ROOT, "tests", "plugin_mcpar_check.cc"), "-L", os.path.join(ROOT, "mcpar_b200"),
                           "-lmcpar", "-lmcgpu", "-Wl,-rpath," + os.path.join(ROOT, "mcpar_b200")])
    r = subprocess.run([exe, _shipped("rosen1_restated_d2.cubin"), str(ngpu), str(mode)], cwd=tmp_path,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.startswith("ok "), r.stdout + r.stderr
