"""Build libmcgpu.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension), and the shipped
likelihood plugins into mcpar_b200/plugins/ (mcpar_b200/plugin.py).

  python -m mcpar_b200.build            # build if stale
  python -m mcpar_b200.build --force
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libmcgpu.so")
OBJ = os.path.join(HERE, "build")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++",
          "-I", os.path.join(ROOT, "include")]
# Sources that fix the layout and meaning of what the engine hands a plugin's kernels (StepParams and WideParams by
# value, the kernel templates they instantiate, both kernel families' launch rules).  Their hash is compiled into libmcgpu.so and into every plugin; the
# engine loads only plugins whose stamp equals its own.
STAMPED = ["include/mcgpu.h", "mcpar_b200/csrc/mcgpu_device.cuh", "mcpar_b200/csrc/mh_kernels.cuh",
           "mcpar_b200/csrc/mcgpu_math.cuh", "mcpar_b200/csrc/mcgpu_tables.h", "mcpar_b200/csrc/mh_plugin.cu",
           "mcpar_b200/csrc/mh_wide.cuh", "mcpar_b200/csrc/mcgpu_cellbound.cuh"]


def kernel_stamp(root=ROOT):
    """64-bit stamp of the STAMPED sources under `root` (contents and relative names only)."""
    h = hashlib.sha256()
    for rel in STAMPED:
        with open(os.path.join(root, rel), "rb") as f:
            data = f.read()
        h.update(rel.encode() + b"\0" + str(len(data)).encode() + b"\0" + data)
    return int.from_bytes(h.digest()[:8], "little")


def stamp_define(stamp):
    return "-DMCGPU_KERNEL_STAMP=0x%016xULL" % stamp


UNITS = {                       # translation unit -> extra flags
    "mh_fast.cu": [],
    "mh_exact.cu": ["-fmad=false"],        # operation-by-operation IEEE arithmetic (verification)
    "mcgpu_api.cu": [stamp_define(kernel_stamp())],
}


def _sources():
    out = [os.path.join(ROOT, "include", "mcgpu.h")]
    for f in os.listdir(CSRC):
        out.append(os.path.join(CSRC, f))
    for f in os.listdir(os.path.join(HERE, "host")):
        out.append(os.path.join(HERE, "host", f))
    return out


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(s) > t for s in _sources())


def build(force=False, verbose=False):
    if force or stale():
        build_lib(verbose)
    from mcpar_b200 import plugin
    plugin.build_shipped(force=force)
    return LIB


def build_lib(verbose=False):
    os.makedirs(OBJ, exist_ok=True)

    def cc(item):
        src, extra = item
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        cmd = [NVCC] + ARCH + COMMON + extra + os.environ.get("MCGPU_NVCC_FLAGS", "").split() + \
            ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        objs = list(ex.map(cc, UNITS.items()))
    cmd = [NVCC] + ARCH + ["-shared", "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++", "-o", LIB] + objs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    build_host()


HOST = os.path.join(HERE, "host")
BIN = os.path.join(HERE, "bin")
DRIVERS = ["mcpar-rosen1", "mcpar-dgauss", "mcpar-rosen2", "mcpar-gmix", "mcpar-bench"]


def build_host():
    """libmcpar.so (C++ MCPar/MCout/VLFunc/mcutil mirror above the C ABI) + the driver mains."""
    os.makedirs(BIN, exist_ok=True)
    cxx = ["/usr/bin/g++", "-std=c++11", "-O2", "-fPIC", "-I", HOST, "-I", os.path.join(ROOT, "include")]
    lib = os.path.join(HERE, "libmcpar.so")
    srcs = [os.path.join(HOST, f) for f in ("likelihoods.cc", "mcout.cc", "mcutil.cc", "mcpar.cc")]
    r = subprocess.run(cxx + ["-shared", "-o", lib] + srcs + ["-L", HERE, "-lmcgpu", "-Wl,-rpath,$ORIGIN"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("host library build failed:\n" + r.stderr)
    for d in DRIVERS:
        r = subprocess.run(cxx + ["-o", os.path.join(BIN, d), os.path.join(HOST, d + ".cc"), "-L", HERE, "-lmcpar",
                                  "-lmcgpu", "-Wl,-rpath,$ORIGIN/.."], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("driver build failed (%s):\n%s" % (d, r.stderr))


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
