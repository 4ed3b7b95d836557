"""Wide device likelihood plugins (MCGPU_PLUGIN_WIDE) on the CPU: every wide cubin holds the four wide step-kernel
phases and the batched evaluation kernel under the exact names the loader asks for, the local and burn-in kernels do
not spill at any of d = 8, 16, 32, 64, nparam outside {8, 16, 32, 64} is refused, and the wide kernel template is
part of the kernel-source stamp."""
import os
import re
import subprocess
from concurrent.futures import ThreadPoolExecutor

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUOBJDUMP = os.path.join(os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")), "cuobjdump")
LOGISTIC = os.path.join(ROOT, "examples", "likelihoods", "logistic_wide.cuh")
ROSEN = os.path.join(ROOT, "tests", "plugins", "rosen1_wide.cuh")
NCH = {8: 1, 16: 1, 32: 2, 64: 4}        # chains per lane group (WideNch, mh_wide.cuh)


# what mcgpu_api.cu (plugin_kernel_name) looks up for a wide plugin, pinned: mh_wide_kernel<101, d, nch, phase> for
# PH_BURN = 0, PH_LOCAL = 2, PH_REMOTE = 3, PH_REMOTE_SUM = 5, and the batched evaluation
def _names(d):
    return ["_ZN5mcgpu4fast14mh_wide_kernelILi101ELi%dELi%dELi%dEEEvNS_10WideParamsE" % (d, NCH[d], ph)
            for ph in (0, 2, 3, 5)] + ["mcgpu_plugin_loglik"]


NAMES_D64 = [
    "_ZN5mcgpu4fast14mh_wide_kernelILi101ELi64ELi4ELi0EEEvNS_10WideParamsE",
    "_ZN5mcgpu4fast14mh_wide_kernelILi101ELi64ELi4ELi2EEEvNS_10WideParamsE",
    "_ZN5mcgpu4fast14mh_wide_kernelILi101ELi64ELi4ELi3EEEvNS_10WideParamsE",
    "_ZN5mcgpu4fast14mh_wide_kernelILi101ELi64ELi4ELi5EEEvNS_10WideParamsE",
    "mcgpu_plugin_loglik",
]

# the shipped wide plugins (plugin.SHIPPED) and the restated Rosenbrock at the two d nothing ships
BUILDS = [(LOGISTIC, None, 32), (ROSEN, 16, 16), (ROSEN, 64, 64), (ROSEN, 8, 8), (ROSEN, 32, 32)]   # (header, nparam=, d)


@pytest.fixture(scope="module")
def built(tmp_path_factory):
    """Each build: (d, cubin path, ptxas log)."""
    from mcpar_b200 import plugin
    out = tmp_path_factory.mktemp("wide_plugins")

    def one(b):
        header, nparam, d = b
        cubin = str(out / ("%s_d%d.cubin" % (os.path.basename(header).split(".")[0], d)))
        cmd = plugin.command(header, cubin, nparam)
        r = subprocess.run(cmd[:1] + ["-Xptxas=-v"] + cmd[1:], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        return d, cubin, r.stderr

    with ThreadPoolExecutor(max_workers=len(BUILDS)) as ex:
        return list(ex.map(one, BUILDS))


def _entries(cubin):
    r = subprocess.run([CUOBJDUMP, "-symbols", cubin], capture_output=True, text=True, check=True)
    return {ln.split()[-1] for ln in r.stdout.splitlines() if "STO_ENTRY" in ln}


def test_shipped_wide_plugins_are_in_the_package_build():
    from mcpar_b200 import plugin
    shipped = {s[2]: (s[0], s[1]) for s in plugin.SHIPPED}
    assert shipped["logistic_wide.cubin"] == (LOGISTIC, None)
    assert shipped["rosen1_wide_d16.cubin"] == (ROSEN, 16) and shipped["rosen1_wide_d64.cubin"] == (ROSEN, 64)


def test_wide_plugins_hold_the_kernels_the_loader_names(built):
    assert _names(64) == NAMES_D64
    for d, cubin, _ in built:
        entries = _entries(cubin)
        missing = set(_names(d)) - entries
        assert not missing, (d, sorted(missing))
        assert not any("mh_steps_kernelILi101" in n for n in entries), d      # no thread-per-chain kernels in a wide cubin


def test_wide_plugin_burnin_and_local_kernels_do_not_spill(built):
    for d, _, log in built:
        props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", log)
        steps = {p[0]: p for p in props if "mh_wide_kernelILi101" in p[0]}
        assert len(steps) == 4, (d, sorted(steps))
        for name in _names(d)[:2]:                                   # PH_BURN, PH_LOCAL
            _, _, st, ld = steps[name]
            assert st == "0" and ld == "0", (d, name, st, ld)


@pytest.mark.parametrize("nparam", [12, 18, 48])
def test_wide_build_refuses_nparam_outside_8_16_32_64(tmp_path, nparam):
    """12 passes the early check (a thread-per-chain plugin may have it) and stops at the wide static_assert; 18 and
    48 stop at the early check.  Both messages name the wide sizes."""
    from mcpar_b200 import plugin
    with pytest.raises((ValueError, RuntimeError), match="8, 16, 32 or 64"):
        plugin.build(ROSEN, nparam=nparam, out=str(tmp_path / "x.cubin"))


def test_kernel_stamp_covers_the_wide_kernel_template():
    from mcpar_b200 import build
    assert "mcpar_b200/csrc/mh_wide.cuh" in build.STAMPED
