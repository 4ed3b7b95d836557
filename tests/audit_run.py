"""Helper of tests/test_gpu_audit.py: one normal-mode run, history + final state saved to an .npz.
Run in a fresh process because MCGPU_EXACT_TESTS is read once per process."""
import os
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import tiled_pinit                        # noqa: E402
from mcpar_b200 import engine                           # noqa: E402


def run(lik, par, d, N, M, pl, cg, nburn, nsamp, rmode=0, sync=10, K=64):
    pin, incov = tiled_pinit(N, d), None
    if lik == "gaussmix":                               # K-component mixture in d = 64 (K = 64: the cooperative kernel), chains start on the means
        from oracle import mh
        rng = np.random.default_rng(8)
        gmu = rng.uniform(-5, 5, (K, d)); gs2 = rng.uniform(0.5, 2.0, (K, d))
        par = mh.gaussmix_params(K, d, gmu, gs2, np.ones(K))
        pin = gmu[np.arange(N) % K].copy()
        incov = np.eye(d) * (2.38 ** 2 / d)
    e = engine.Engine(d, N, mode="normal", pool_m=M, pl=pl, coin_group=cg, history_steps=nsamp, remote_mode=rmode, sync=sync)
    e.run(nsamp, nburn, pin, lik, par, incov)
    out = dict(hist=e.history(), p=e.state()["p"], pool=e.musig(), acc=np.array(e.stats()["accepted"]),
               rit=np.array(e.stats()["remote_iterations"]))
    e.close()
    return out


CASES = {
    "dgauss": ("dualgaussian", [5.0], 2, 8192, 16, 0.5, 0, 150, 300),
    "rosen2": ("rosenbrock1", None, 2, 4096, 32, 0.5, 0, 150, 300),
    "rosen2_groups": ("rosenbrock1", None, 2, 4096, 12, 0.6, 8, 150, 200),
    "rosen4": ("rosenbrock1", None, 4, 2048, 8, 0.5, 0, 150, 200),
    # remote mode 1 (sum-mixture proposal): the fp32 bounds on q(x)/q(x') against the all-fp64 evaluation
    "dgauss_sum": ("dualgaussian", [5.0], 2, 8192, 64, 0.5, 0, 150, 300, 1),
    "rosen2_sum256": ("rosenbrock1", None, 2, 4096, 256, 0.5, 0, 150, 300, 1),
    "rosen2_sum_groups": ("rosenbrock1", None, 2, 4096, 12, 0.6, 8, 150, 200, 1),
    "rosen4_sum": ("rosenbrock1", None, 4, 2048, 8, 0.5, 0, 150, 200, 1),
    # wide kernels (d = 16: 8 lanes per chain) and the cooperative d = 64 kernel
    "rosen16_ref": ("rosenbrock1", None, 16, 512, 8, 0.5, 0, 150, 100, 0),
    "rosen16_sum": ("rosenbrock1", None, 16, 512, 16, 0.5, 0, 150, 100, 1),
    "gmix64_sum": ("gaussmix", None, 64, 200, 40, 0.5, 0, 100, 100, 1),
    "gmix64_sum256": ("gaussmix", None, 64, 256, 0, 0.5, 0, 100, 100, 1),
    # wide kernels with 2 and 4 chains per lane group (d = 32, 64), and at d = 64 with K = 80 (kpad 128: not cooperative)
    "rosen32_ref": ("rosenbrock1", None, 32, 500, 8, 0.5, 0, 150, 100, 0),
    "rosen32_sum": ("rosenbrock1", None, 32, 500, 16, 0.5, 0, 150, 100, 1),
    "rosen64_ref": ("rosenbrock1", None, 64, 250, 8, 0.5, 0, 150, 100, 0),
    "rosen64_sum": ("rosenbrock1", None, 64, 250, 16, 0.5, 0, 150, 100, 1),
    "gmix64_k80_ref": ("gaussmix", None, 64, 200, 40, 0.5, 0, 100, 100, 0, 10, 80),
    "gmix64_k80_sum": ("gaussmix", None, 64, 200, 40, 0.5, 0, 100, 100, 1, 10, 80),
    # thread-per-chain at d = 16 (per-group coins), and windows > 32 steps (job-wide coin: chunks of up to 32 steps)
    "rosen16_groups_ref": ("rosenbrock1", None, 16, 512, 8, 0.5, 8, 150, 100, 0),
    "rosen16_groups_sum": ("rosenbrock1", None, 16, 512, 8, 0.5, 8, 150, 100, 1),
    "rosen2_sync40_ref": ("rosenbrock1", None, 2, 4096, 32, 0.5, 0, 150, 200, 0, 40),
    "rosen2_sync40_sum": ("rosenbrock1", None, 2, 4096, 32, 0.5, 0, 150, 200, 1, 40),
}

if __name__ == "__main__":
    name, path = sys.argv[1], sys.argv[2]
    np.savez(path, **run(*CASES[name]))
