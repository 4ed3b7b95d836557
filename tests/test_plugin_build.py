"""Device likelihood plugins on the CPU: every shipped plugin compiles for sm_100a into a cubin that holds the
kernels the loader asks for under the exact names it asks for, without register spills at d <= 12; the
kernel-source stamp is deterministic and follows every stamped byte; bad parameter counts are refused."""
import os
import re
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUOBJDUMP = os.path.join(os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")), "cuobjdump")
LOGISTIC = os.path.join(ROOT, "examples", "likelihoods", "logistic.cuh")
ROSEN = os.path.join(ROOT, "tests", "plugins", "rosen1_restated.cuh")

# what mcgpu_api.cu (plugin_kernel_name) looks up, pinned: mh_steps_kernel<101, d, RNG_PHILOX, phase> for the six
# phases, init_loglik_kernel<101, d> and the batched evaluation
def _names(d):
    steps = ["_ZN5mcgpu4fast15mh_steps_kernelILi101ELi%dELi0ELi%dEEEvNS_10StepParamsE" % (d, ph) for ph in range(6)]
    return steps + ["_ZN5mcgpu4fast18init_loglik_kernelILi101ELi%dEEEvNS_10StepParamsE" % d, "mcgpu_plugin_loglik"]


NAMES_D6 = [
    "_ZN5mcgpu4fast15mh_steps_kernelILi101ELi6ELi0ELi0EEEvNS_10StepParamsE",
    "_ZN5mcgpu4fast15mh_steps_kernelILi101ELi6ELi0ELi1EEEvNS_10StepParamsE",
    "_ZN5mcgpu4fast15mh_steps_kernelILi101ELi6ELi0ELi2EEEvNS_10StepParamsE",
    "_ZN5mcgpu4fast15mh_steps_kernelILi101ELi6ELi0ELi3EEEvNS_10StepParamsE",
    "_ZN5mcgpu4fast15mh_steps_kernelILi101ELi6ELi0ELi4EEEvNS_10StepParamsE",
    "_ZN5mcgpu4fast15mh_steps_kernelILi101ELi6ELi0ELi5EEEvNS_10StepParamsE",
    "_ZN5mcgpu4fast18init_loglik_kernelILi101ELi6EEEvNS_10StepParamsE",
    "mcgpu_plugin_loglik",
]

BUILDS = [(LOGISTIC, None, 6), (ROSEN, 2, 2), (ROSEN, 12, 12), (ROSEN, 16, 16)]   # (header, nparam=, d)


@pytest.fixture(scope="module")
def built(tmp_path_factory):
    """Each build: (d, cubin path, ptxas log)."""
    from mcpar_b200 import plugin
    out = tmp_path_factory.mktemp("plugins")

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


def test_shipped_plugins_hold_the_kernels_the_loader_names(built):
    assert _names(6) == NAMES_D6
    for d, cubin, _ in built:
        missing = set(_names(d)) - _entries(cubin)
        assert not missing, (d, sorted(missing))


def test_plugin_step_kernels_do_not_spill(built):
    for d, _, log in built:
        if d > 12:
            continue
        props = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", log)
        steps = [p for p in props if "mh_steps_kernelILi101" in p[0]]
        assert len(steps) == 6, (d, len(steps))
        for name, _, st, ld in steps:
            assert st == "0" and ld == "0", (d, name, st, ld)


def test_build_caches_and_cli(tmp_path):
    from mcpar_b200 import plugin
    out = str(tmp_path / "r.cubin")
    r = subprocess.run([sys.executable, "-m", "mcpar_b200.plugin", ROSEN, "-o", out, "--nparam", "4"], cwd=ROOT,
                       capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == out, r.stderr
    t = os.path.getmtime(out)
    assert plugin.build(ROSEN, nparam=4, out=out) == out and os.path.getmtime(out) == t      # up to date: not rebuilt
    assert _names(4)[0] in _entries(plugin.build(ROSEN, nparam=4, out=out, force=True))


def test_kernel_stamp_is_deterministic_and_covers_every_stamped_byte(tmp_path):
    from mcpar_b200 import build
    for rel in build.STAMPED:
        os.makedirs(os.path.dirname(str(tmp_path / rel)), exist_ok=True)
        shutil.copyfile(os.path.join(ROOT, rel), str(tmp_path / rel))
    s0 = build.kernel_stamp()
    assert build.kernel_stamp(str(tmp_path)) == s0 == build.kernel_stamp()
    for rel in build.STAMPED:
        f = str(tmp_path / rel)
        data = bytearray(open(f, "rb").read())
        data[len(data) // 2] ^= 0x01
        open(f, "wb").write(bytes(data))
        assert build.kernel_stamp(str(tmp_path)) != s0, rel
        data[len(data) // 2] ^= 0x01
        open(f, "wb").write(bytes(data))
        assert build.kernel_stamp(str(tmp_path)) == s0, rel


@pytest.mark.parametrize("nparam", [0, 1, 3, 18, 5.0])
def test_build_refuses_bad_nparam_early(tmp_path, nparam):
    from mcpar_b200 import plugin
    with pytest.raises(ValueError, match="even"):
        plugin.build(ROSEN, nparam=nparam, out=str(tmp_path / "x.cubin"))


def test_build_refuses_odd_nparam_at_compile_time(tmp_path):
    from mcpar_b200 import plugin
    h = tmp_path / "odd.cuh"
    h.write_text(open(ROSEN).read().replace("#define MCGPU_PLUGIN_NPARAM 2", "#define MCGPU_PLUGIN_NPARAM 5"))
    with pytest.raises(RuntimeError, match="MCGPU_PLUGIN_NPARAM must be even"):
        plugin.build(str(h), out=str(tmp_path / "odd.cubin"))
