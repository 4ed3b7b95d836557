"""Convergence diagnostics and quantiles of the device history (mcgpu_history_diag_partials, mcgpu_diag_finalize,
mcgpu_history_quantiles) against the numpy reference of the same rows read back with history() (tests/diag_ref.py)."""
import os
import sys

import numpy as np
import pytest

from conftest import tiled_pinit

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import diag_ref  # noqa: E402

pytestmark = pytest.mark.gpu

PROBS = (0.0, 0.05, 0.37, 0.5, 0.95, 1.0)


def check_engine(e, rows, Gs=(1,), full_report=True):
    """Device partials = host partials of `rows` (the valid history) to 1e-12, the finalized report = the ArviZ port,
    a repeated call gives the same bits, quantiles = numpy."""
    from mcpar_b200 import engine as eng
    for G in Gs:
        blk = e.diag_partials(G)
        diag_ref.assert_blocks_close(blk, diag_ref.partials(rows, G, int(blk[2])))
        assert np.array_equal(blk, e.diag_partials(G)), "a repeated call changed bits"
        if full_report:
            diag_ref.assert_reports_close(eng.diag_finalize([blk]), diag_ref.report(rows, G), rtol=1e-10)
    check_quantiles(e, rows)


def check_quantiles(e, rows):
    q = e.quantiles(PROBS)
    assert np.array_equal(q, e.quantiles(PROBS))
    S = rows.shape[0] * rows.shape[1]
    # probabilities whose h = (S - 1) p is whole return the order statistic itself
    ranks = [i for i in (0, 1, S // 3, S // 2, S - 2, S - 1) if (S - 1) * (i / (S - 1)) == i]
    qo = e.quantiles([i / (S - 1) for i in ranks])
    for j in range(rows.shape[2]):
        flat = rows[:, :, j].ravel()
        want = np.quantile(flat, PROBS, method="linear")
        assert np.all(np.abs(q[j] - want) <= 2 * np.spacing(np.abs(want))), (j, q[j], want)
        assert np.array_equal(qo[j], np.partition(flat, ranks)[ranks]), (j, ranks)


def _run(eng, d, C, lik, par, nsamp, nburn=100, history_steps=None, incov=None, plugin=None, pin=None, **kw):
    e = eng.Engine(d, C, history_steps=history_steps or nsamp // kw.get("thin", 1), **kw)
    e.run(nsamp, nburn, tiled_pinit(C, d) if pin is None else pin, lik, par, incov, plugin=plugin)
    return e


@pytest.mark.parametrize("mode", [0, 1])
def test_dualgaussian_both_remote_modes(mode):
    from mcpar_b200 import engine as eng
    e = _run(eng, 2, 4096, "dualgaussian", [5.0], 60, pool_m=16, pl=0.7, remote_mode=mode)
    rows = e.history()
    assert np.mean(rows[1:] == rows[:-1]) > 0.05                 # rejected steps repeat rows: ties in the quantiles
    check_engine(e, rows, Gs=(1, 8, 4096))
    e.close()


def test_wide_rosenbrock_d16():
    from mcpar_b200 import engine as eng
    e = _run(eng, 16, 1024, "rosenbrock1", None, 50, pool_m=8, pl=0.7, coin_group=0)
    check_engine(e, e.history(), Gs=(1, 32))
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
    check_engine(e, e.history(), Gs=(1, 4))
    e.close()


def test_logistic_plugin():
    from mcpar_b200 import engine as eng, plugin
    from test_gpu_plugin import logistic_data
    par = logistic_data()[0]
    e = _run(eng, 6, 512, "plugin", par, 40, nburn=110, plugin=plugin.shipped("logistic.cubin"),
             pin=tiled_pinit(512, 6) * 0.25, pool_m=8, pl=0.7)
    check_engine(e, e.history(), Gs=(1, 16))
    e.close()


def test_thinned_and_wrapped_histories():
    from mcpar_b200 import engine as eng
    e = _run(eng, 2, 1024, "rosenbrock1", None, 90, thin=3, pool_m=8)        # 30 kept steps
    rows = e.history()
    assert rows.shape[0] == 30
    check_engine(e, rows, Gs=(1, 4))
    e.close()
    e = _run(eng, 2, 1024, "dualgaussian", [5.0], 100, history_steps=37, pool_m=8)   # ring wrapped: last 37 of 100
    rows = e.history()
    assert rows.shape[0] == 37 and e.stats()["history_rows"] == 100 * 1024
    check_engine(e, rows, Gs=(1, 2))
    e.close()


def test_after_restore_counts_rows_from_the_load():
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
    check_engine(b, rows, Gs=(1, 8))
    b.close()


def test_host_callback_engine():
    from mcpar_b200 import engine as eng
    e = eng.Engine(2, 512, pool_m=8, pl=0.7, history_steps=40)
    e.run_host(40, 60, tiled_pinit(512, 2), lambda x: -0.5 * np.sum(x * x, axis=1))
    check_engine(e, e.history(), Gs=(1, 8))
    e.close()


def test_sharded_blocks_match_one_engine():
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
    blocks = [e.diag_partials(64) for e in es]
    hist = np.concatenate([e.history() for e in es], axis=1)
    for e in es:
        e.close()
    one = eng.Engine(d, 2 * Cg, pool_m=16, pl=0.7, sync=10, coin_group=0, history_steps=nsamp)
    one.run(nsamp, 130, pin, "dualgaussian", [5.0])
    assert np.array_equal(one.history(), hist)                  # the same chains, bit for bit
    single = eng.diag_finalize([one.diag_partials(64)])
    one.close()
    diag_ref.assert_reports_close(eng.diag_finalize(blocks), single)


def test_refusals_leave_the_engine_usable():
    from mcpar_b200 import engine as eng
    e = eng.Engine(2, 64, pool_m=8, history_steps=20)
    with pytest.raises(eng.McgpuError, match="ESTATE"):
        e.diag_partials(1, 1)                                    # empty history
    with pytest.raises(eng.McgpuError, match="ESTATE"):
        e.quantiles([0.5])
    none = eng.Engine(2, 64, pool_m=8)
    none.run(10, 10, tiled_pinit(64, 2), "dualgaussian", [5.0])
    with pytest.raises(eng.McgpuError, match="ESTATE"):          # no history
        none.diag_partials(1, 1)
    none.close()
    e.set_likelihood("dualgaussian", [5.0]); e.set_covariance(None); e.set_state(tiled_pinit(64, 2))
    e.burnin(20); e.sample_begin(20); e.sample(3); e.synchronize()
    with pytest.raises(eng.McgpuError, match="EINVAL"):          # n = 3 < 4
        e.diag_partials(1, 1)
    e.sample(17); e.synchronize()                                # n = 20, N = 10
    launches = e.stats()["kernel_launches"]
    for G, L in ((0, 5), (3, 5), (128, 5), (1, 0), (1, 10)):
        with pytest.raises(eng.McgpuError, match="EINVAL"):
            e.diag_partials(G, L)
    for p in ([], [0.5] * 17, [-0.1], [1.5], [np.nan]):
        with pytest.raises(eng.McgpuError, match="EINVAL"):
            e.quantiles(p)
    lib = eng.load()
    assert lib.mcgpu_history_diag_partials(e.h, 1, 5, None) == -1
    assert lib.mcgpu_history_quantiles(e.h, None, 1, None) == -1
    assert e.stats()["kernel_launches"] == launches, "a refusal launched a kernel"
    e.diag_partials(1, 9); e.quantiles()
    e.sample_begin(20); e.sample(20); e.synchronize()           # the engine still samples afterwards
    check_engine(e, e.history(), Gs=(1, 2, 64))
    e.close()


def test_superchain_must_divide_chain0():
    """A shard of chains [32, 128) of a 128-chain job: G = 3 divides its 96 chains but not chain0."""
    from mcpar_b200 import engine as eng
    e = eng.Engine(2, 96, chain0=32, nchain_total=128, pool_m=0, pl=1.0, sync=10, history_steps=20)
    e.set_likelihood("dualgaussian", [5.0]); e.set_covariance(None); e.set_state(tiled_pinit(96, 2))
    left = 20
    while left:
        done, pending = e.burnin_some(left)
        left -= done
        if pending:
            e.tune()
    e.sample_begin(20)
    for _ in range(2):
        e.sample(10)
        e.exchange_begin(); e.exchange_end()
    e.synchronize()
    with pytest.raises(eng.McgpuError, match="EINVAL"):
        e.diag_partials(3, 5)
    check_engine(e, e.history(), Gs=(1, 32), full_report=False)
    e.close()


def test_full_size_dualgaussian():
    """2^20 chains, n = 100 kept steps: device partials and quantiles against the host reference."""
    from mcpar_b200 import engine as eng
    C = 1 << 20
    e = eng.Engine(2, C, pool_m=16, history_steps=100)
    e.set_likelihood("dualgaussian", [5.0]); e.set_covariance(None)
    e.set_state_sobol([-3.0, -3.0], [3.0, 3.0])
    e.burnin(100); e.sample_begin(100); e.sample(100); e.synchronize()
    rows = e.history()
    blk = e.diag_partials(16)
    diag_ref.assert_blocks_close(blk, diag_ref.partials(rows, 16, int(blk[2])))
    # two separated modes over 100 steps: R-hat well above 1 is the right answer here, not a failure
    diag_ref.assert_reports_close(eng.diag_finalize([blk]), eng.diag_finalize([diag_ref.partials(rows, 16)]))
    q = e.quantiles((0.05, 0.5, 0.95))
    for j in range(3):
        want = np.quantile(rows[:, :, j].ravel(), (0.05, 0.5, 0.95), method="linear")
        assert np.all(np.abs(q[j] - want) <= 2 * np.spacing(np.abs(want))), (j, q[j], want)
    e.close()
