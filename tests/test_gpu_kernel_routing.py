"""Each case of kernel_matrix.py launches exactly the step kernels it claims, as the CUDA profiler records them.  With
test_kernel_coverage.py this ties every instantiation in libmcgpu.so to a case that test_gpu_parity.py compares with
the CPU oracle."""
import numpy as np
import pytest

import kernel_matrix as km
from conftest import make_streams

pytestmark = pytest.mark.gpu


def _launched(fn):
    """Keys of the step kernels launched while fn() runs (CUPTI records the library's launches made through ctypes)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {k for k in (km.kernel_key(ev.name) for ev in prof.events()) if k is not None}


@pytest.mark.parametrize("case", km.CASES, ids=[c.id for c in km.CASES])
def test_normal_mode_case_launches_its_claims(case):
    from mcpar_b200 import engine
    c = case
    par, incov, pin = km.model(c.lik, c.d, c.N, c.par)
    e = engine.Engine(c.d, c.N, mode="normal", pool_m=c.pool_m, pl=c.pl, coin_group=c.cg, remote_mode=c.rmode,
                      pool_lag=c.lag, sync=c.sync, thin=c.thin, history_steps=(c.nsamp + c.thin - 1) // c.thin)
    try:
        got = _launched(lambda: e.run(c.nsamp, km.NBURN, pin, c.lik, par, incov))
    finally:
        e.close()
    assert got == set(c.claims), "launched but not claimed: %s; claimed but not launched: %s" % (
        sorted(got - c.claims), sorted(c.claims - got))


@pytest.mark.parametrize("case", km.REPLAY, ids=[c.id for c in km.REPLAY])
def test_replay_case_launches_its_claims(case):
    from mcpar_b200 import engine
    c = case
    par, incov, pin = km.model(c.lik, c.d, c.C, c.par)
    if c.incov == "rosen16":
        incov = km.rosen_factor(16)
    nburn, nsamp = 60, 20
    Z, U, _ = make_streams(1, c.C, c.d, nsamp + nburn, 11, mult=2)
    e = engine.Engine(c.d, c.C, mode="replay_local", pl=1.0, history_steps=nsamp)

    def run():
        e.set_likelihood(c.lik, par); e.set_covariance(incov); e.set_state(pin)
        e.set_streams(0, Z[0], U[0])
        e.burnin(nburn); e.sample_begin(nsamp); e.sample(nsamp); e.synchronize()
    try:
        got = _launched(run)
    finally:
        e.close()
    assert got == set(c.claims), (sorted(got - c.claims), sorted(c.claims - got))
