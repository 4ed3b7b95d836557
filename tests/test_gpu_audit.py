"""Audit of the fp32-bounded decisions of the production kernels.

The accept test u < exp(delta) cfac (mcpar.cc:67-69, :167-169) and the rejection test of the remote
proposal u < max_i Q_i / sum_i Q_i (mcpar.cc:355-406) are settled by rigorous fp32 bounds and
evaluated in fp64 only when the bounds straddle u.  With MCGPU_EXACT_TESTS=1 the same kernels always
take the fp64 route.  If the bounds are right, no decision differs and the two runs are identical
bit for bit -- every state of every chain at every step."""
import os
import subprocess
import sys
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize("case", ["dgauss", "rosen2", "rosen2_groups", "rosen4",
                                  "dgauss_sum", "rosen2_sum256", "rosen2_sum_groups", "rosen4_sum",
                                  "rosen16_ref", "rosen16_sum", "gmix64_sum", "gmix64_sum256",
                                  "rosen32_ref", "rosen32_sum", "rosen64_ref", "rosen64_sum", "gmix64_k80_ref", "gmix64_k80_sum",
                                  "rosen16_groups_ref", "rosen16_groups_sum", "rosen2_sync40_ref", "rosen2_sync40_sum"])
def test_fp32_bounded_decisions_equal_fp64_decisions(case, tmp_path):
    outs = {}
    for mode in ("0", "1"):
        path = str(tmp_path / ("run%s.npz" % mode))
        env = dict(os.environ, MCGPU_EXACT_TESTS=mode)
        r = subprocess.run([sys.executable, os.path.join(HERE, "audit_run.py"), case, path], env=env,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        outs[mode] = np.load(path)
    fast, exact = outs["0"], outs["1"]
    assert int(exact["rit"]) > 0, "the case must exercise remote proposals"
    for k in ("hist", "p", "pool", "acc", "rit"):
        assert np.array_equal(fast[k], exact[k]), "fp32-bounded run differs from the fp64 run in %s" % k
