"""Rank-normalised R-hat, bulk ESS and tail ESS of the device history (mcgpu_history_rank_diag) against the port of
ArviZ (tests/rank_ref.py) over the same rows read back with history()."""
import os
import sys

import numpy as np
import pytest

from conftest import tiled_pinit

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import rank_ref  # noqa: E402

pytestmark = pytest.mark.gpu


def check(e, rows, rtol=1e-10):
    """Device report = the port of `rows` (the valid history) to rtol; a repeated call gives the same bits."""
    got = e.rank_diagnostics()
    rank_ref.assert_reports_close(got, rank_ref.report(rows), rtol)
    again = e.rank_diagnostics()
    for k in rank_ref.FIELDS:
        assert np.array_equal(got[k], again[k], equal_nan=True), "a repeated call changed bits (%s)" % k
    return got


def _run(eng, d, C, lik, par, nsamp, nburn=100, history_steps=None, incov=None, plugin=None, pin=None, **kw):
    e = eng.Engine(d, C, history_steps=history_steps or nsamp // kw.get("thin", 1), **kw)
    e.run(nsamp, nburn, tiled_pinit(C, d) if pin is None else pin, lik, par, incov, plugin=plugin)
    return e


@pytest.mark.parametrize("mode", [0, 1])
def test_dualgaussian_both_remote_modes(mode):
    from mcpar_b200 import engine as eng
    e = _run(eng, 2, 4096, "dualgaussian", [5.0], 60, pool_m=16, pl=0.7, remote_mode=mode)
    check(e, e.history())
    e.close()


def test_odd_n_thinned_and_wrapped():
    from mcpar_b200 import engine as eng
    e = _run(eng, 2, 1024, "rosenbrock1", None, 90, thin=2, pool_m=8)         # 45 kept steps
    rows = e.history()
    assert rows.shape[0] == 45
    check(e, rows)
    e.close()
    e = _run(eng, 2, 1024, "dualgaussian", [5.0], 100, history_steps=37, pool_m=8)   # ring wrapped: last 37 of 100
    rows = e.history()
    assert rows.shape[0] == 37 and e.stats()["history_rows"] == 100 * 1024
    check(e, rows)
    e.close()


def test_cross_chain_ties_from_the_first_main_step():
    """A wide proposal rejects most steps: the chains keep their tiled starting points, so draws tie across chains."""
    from mcpar_b200 import engine as eng
    C = 2048
    e = _run(eng, 2, C, "dualgaussian", [5.0], 40, nburn=2, incov=np.eye(2) * 400.0, pool_m=0, pl=1.0)
    rows = e.history()
    s = e.stats()
    assert s["accepted"] / s["tried"] < 0.2
    assert len(np.unique(rows[0, :, 0])) < C // 4                              # ties across chains
    assert len(np.unique(rows[:, :, 0])) < rows[:, :, 0].size // 4
    check(e, rows)
    e.close()


def test_wide_rosenbrock_d16():
    from mcpar_b200 import engine as eng
    e = _run(eng, 16, 1024, "rosenbrock1", None, 50, pool_m=8, pl=0.7, coin_group=0)
    check(e, e.history())
    e.close()


def test_gaussmix_d64_cooperative():
    from mcpar_b200 import engine as eng
    from oracle import mh
    K, d, N = 64, 64, 256
    rng = np.random.default_rng(8)
    gmu = rng.uniform(-5, 5, (K, d)); gs2 = rng.uniform(0.5, 2.0, (K, d))
    par = mh.gaussmix_params(K, d, gmu, gs2, np.ones(K))
    pin = gmu[np.arange(N) % K].copy()
    e = _run(eng, d, N, "gaussmix", par, 30, nburn=60, incov=np.eye(d) * (2.38 ** 2 / d), pin=pin,
             pool_m=12, pl=0.7, coin_group=0, remote_mode=1, pool_lag=1)
    rows = e.history()
    assert rows.shape[2] == 65
    check(e, rows)
    e.close()


def test_logistic_plugin():
    from mcpar_b200 import engine as eng, plugin
    from test_gpu_plugin import logistic_data
    par = logistic_data()[0]
    e = _run(eng, 6, 512, "plugin", par, 40, nburn=110, plugin=plugin.shipped("logistic.cubin"),
             pin=tiled_pinit(512, 6) * 0.25, pool_m=8, pl=0.7)
    check(e, e.history())
    e.close()


def test_host_callback_nan_loglik():
    """Chains whose log-likelihood is NaN hold NaN in the logL column: that column reports its count only."""
    from mcpar_b200 import engine as eng
    C = 512

    def loglik(x):
        y = -0.5 * np.sum(x * x, axis=1)
        y[::7] = np.nan
        return y

    e = eng.Engine(2, C, pool_m=8, pl=0.7, history_steps=40)
    e.run_host(40, 60, tiled_pinit(C, 2), loglik)
    rows = e.history()
    nf = np.count_nonzero(~np.isfinite(rows[:, :, 2]))
    assert nf > 0
    got = check(e, rows)
    assert got["nonfinite"][2] == nf and np.isnan(got["rhat"][2]) and np.isnan(got["ess_tail"][2])
    assert np.isfinite(got["ess_bulk"][:2]).all()
    e.close()


def test_restored_engine_counts_rows_from_the_load():
    from mcpar_b200 import engine as eng
    kw = dict(pool_m=8, pl=0.7, coin_group=0, history_steps=80)
    a = eng.Engine(2, 1024, **kw)
    a.set_likelihood("dualgaussian", [5.0]); a.set_covariance(None); a.set_state(tiled_pinit(1024, 2))
    a.burnin(100); a.sample_begin(80); a.sample(30)
    blob = a.checkpoint()
    a.close()
    b = eng.Engine(2, 1024, **kw)
    b.set_likelihood("dualgaussian", [5.0])
    b.restore(blob)
    b.sample(50); b.synchronize()
    rows = b.history(first=30)
    assert rows.shape[0] == 50
    check(b, rows)
    b.close()


def test_each_shard_reports_over_its_own_chains():
    from mcpar_b200 import engine as eng
    d, Cg, nsamp = 2, 2048, 70
    ndev = eng.device_count()
    pin = tiled_pinit(2 * Cg, d)
    es = [eng.Engine(d, Cg, nchain_total=2 * Cg, chain0=r * Cg, pool_m=16, pl=0.7, sync=10, coin_group=0,
                     history_steps=nsamp, device=r % ndev) for r in range(2)]
    for r, e in enumerate(es):
        e.set_likelihood("dualgaussian", [5.0]); e.set_covariance(None); e.set_state(pin[r * Cg:(r + 1) * Cg])
    eng.p2p_attach_local(es)
    eng.burnin_group(es, 130)
    for e in es:
        e.sample_begin(nsamp)
    for _ in range(nsamp // 10):
        eng.sample_group(es, 10)
    for e in es:
        e.synchronize()
    for e in es:
        check(e, e.history())
    for e in es:
        e.close()


def test_refusals_launch_nothing_and_leave_the_engine_usable():
    from mcpar_b200 import engine as eng
    e = eng.Engine(2, 64, pool_m=8, history_steps=20)
    with pytest.raises(eng.McgpuError, match="ESTATE"):
        e.rank_diagnostics(1)                                    # empty history
    none = eng.Engine(2, 64, pool_m=8)
    none.run(10, 10, tiled_pinit(64, 2), "dualgaussian", [5.0])
    with pytest.raises(eng.McgpuError, match="ESTATE"):          # no history
        none.rank_diagnostics(1)
    none.close()
    e.set_likelihood("dualgaussian", [5.0]); e.set_covariance(None); e.set_state(tiled_pinit(64, 2))
    e.burnin(20); e.sample_begin(20); e.sample(3); e.synchronize()
    with pytest.raises(eng.McgpuError, match="EINVAL"):          # n = 3 < 4
        e.rank_diagnostics(1)
    e.sample(17); e.synchronize()                                # n = 20, N = 10
    launches = e.stats()["kernel_launches"]
    for L in (0, 10, -3):
        with pytest.raises(eng.McgpuError, match="EINVAL"):
            e.rank_diagnostics(L)
    lib = eng.load()
    assert lib.mcgpu_history_rank_diag(e.h, 5, None) == -1
    assert e.stats()["kernel_launches"] == launches, "a refusal launched a kernel"
    e.rank_diagnostics(9)
    assert e.stats()["kernel_launches"] > launches
    e.sample_begin(20); e.sample(20); e.synchronize()           # the engine still samples afterwards
    check(e, e.history())
    e.close()


def test_full_size_dualgaussian():
    """2^20 chains, n = 100 kept steps: every column's report is finite and column 0 equals the port."""
    from mcpar_b200 import engine as eng
    C = 1 << 20
    e = eng.Engine(2, C, pool_m=16, history_steps=100)
    e.set_likelihood("dualgaussian", [5.0]); e.set_covariance(None)
    e.set_state_sobol([-3.0, -3.0], [3.0, 3.0])
    e.burnin(100); e.sample_begin(100); e.sample(100); e.synchronize()
    got = e.rank_diagnostics()
    again = e.rank_diagnostics()
    for k in rank_ref.FIELDS:
        assert np.array_equal(got[k], again[k], equal_nan=True), k
    assert all(np.isfinite(got[k]).all() for k in rank_ref.FIELDS)
    x = e.history()[:, :, :1]
    e.close()
    rank_ref.assert_reports_close({k: got[k][:1] for k in rank_ref.FIELDS}, rank_ref.report(x), 1e-10)
