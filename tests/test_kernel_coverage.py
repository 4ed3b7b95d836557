"""Every step-kernel instantiation that libmcgpu.so ships is launched by a case of kernel_matrix.py (and so compared
with the CPU oracle), and every kernel a case claims exists in the library."""
import os
import subprocess

import pytest

from kernel_matrix import all_claims, kernel_key

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUOBJDUMP = os.path.join(os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")), "cuobjdump")
LIB = os.path.join(ROOT, "mcpar_b200", "libmcgpu.so")


@pytest.fixture(scope="module")
def shipped():
    """Keys of the library's mh_steps_kernel, mh_wide_kernel and mh_coop_kernel entries."""
    from mcpar_b200 import build
    if build.stale():
        build.build_lib()
    r = subprocess.run([CUOBJDUMP, "-symbols", LIB], capture_output=True, text=True, check=True)
    names = [ln.split()[-1] for ln in r.stdout.splitlines() if "STO_ENTRY" in ln]
    keys = [kernel_key(n) for n in names]
    assert sum(k is not None for k in keys) > 0, "no step kernels found in libmcgpu.so"
    return {k for k in keys if k is not None}


def test_every_shipped_step_kernel_is_claimed_by_a_case(shipped):
    unclaimed = sorted(shipped - all_claims())
    assert not unclaimed, "%d kernels no case launches:\n  %s" % (len(unclaimed), "\n  ".join(map(str, unclaimed)))


def test_every_claimed_kernel_is_shipped(shipped):
    missing = sorted(all_claims() - shipped)
    assert not missing, "%d claimed kernels are not in libmcgpu.so:\n  %s" % (len(missing), "\n  ".join(map(str, missing)))


def test_kernel_names_parse_in_both_forms():
    assert kernel_key("_ZN5mcgpu4fast15mh_steps_kernelILi4ELi16ELi0ELi5EEEvNS_10StepParamsE") == \
        kernel_key("void mcgpu::fast::mh_steps_kernel<4, 16, 0, 5>(mcgpu::StepParams)") == \
        ("steps", "fast", "GAUSSMIX", 16, "PHILOX", "REMOTE_SUM")
    assert kernel_key("_ZN5mcgpu5exact15mh_steps_kernelILi0ELi8ELi1ELi2EEEvNS_10StepParamsE") == \
        ("steps", "exact", "ROSENBROCK1", 8, "REPLAY", "LOCAL")
    assert kernel_key("_ZN5mcgpu4fast14mh_wide_kernelILi0ELi64ELi4ELi3EEEvNS_10WideParamsE") == \
        kernel_key("void mcgpu::fast::mh_wide_kernel<0, 64, 4, 3>(mcgpu::WideParams)") == ("wide", "ROSENBROCK1", 64, 4, "REMOTE")
    assert kernel_key("_ZN5mcgpu4fast14mh_coop_kernelILi64ELi1ELi5ELb1EEEvNS_10WideParamsEiii") == \
        kernel_key("void mcgpu::fast::mh_coop_kernel<64, 1, 5, true>(mcgpu::WideParams, int, int, int)") == \
        ("coop", 64, 1, "REMOTE_SUM", 1)
    assert kernel_key("void mcgpu::fast::tune_kernel(unsigned long long*)") is None
