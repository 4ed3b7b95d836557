"""Build a device likelihood plugin: a cubin of the production step kernels instantiated with the functor of ONE
user header (the contract is include/mcgpu_plugin.cuh).  Load it with Engine.set_likelihood("plugin", par,
plugin=path) or mcgpu_set_likelihood_plugin.

  python -m mcpar_b200.plugin mylik.cuh -o mylik.cubin [--nparam N] [--force]

The cubin is compiled from mcpar_b200/csrc/mh_plugin.cu with the nvcc, architecture and flags of libmcgpu.so's
production unit, and carries the stamp of the kernel sources (build.kernel_stamp): rebuild plugins whenever
those change -- the engine refuses a plugin with another stamp.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

from mcpar_b200 import build as b

SRC = os.path.join(b.CSRC, "mh_plugin.cu")
PLUGINS = os.path.join(b.HERE, "plugins")
# the plugins build.py ships: (header, nparam or None for the header's own, cubin name)
SHIPPED = [
    (os.path.join(b.ROOT, "examples", "likelihoods", "logistic.cuh"), None, "logistic.cubin"),
    (os.path.join(b.ROOT, "tests", "plugins", "rosen1_restated.cuh"), 2, "rosen1_restated_d2.cubin"),
    (os.path.join(b.ROOT, "tests", "plugins", "rosen1_restated.cuh"), 16, "rosen1_restated_d16.cubin"),
]


def command(header, out, nparam=None, stamp=None):
    """The nvcc command that compiles `header` into the plugin cubin `out`."""
    header = os.path.abspath(header)
    if nparam is not None and (not isinstance(nparam, int) or nparam < 2 or nparam > 16 or nparam % 2):
        raise ValueError("nparam must be an even integer in 2..16 (thread-per-chain kernels), got %r" % (nparam,))
    cmd = [b.NVCC] + b.ARCH + b.COMMON + ["-I", os.path.dirname(header), "-include", header,
                                          b.stamp_define(b.kernel_stamp() if stamp is None else stamp)]
    if nparam is not None:
        cmd.append("-DMCGPU_PLUGIN_NPARAM=%d" % nparam)
    return cmd + ["-cubin", SRC, "-o", os.path.abspath(out)]


def _key(header, cmd):
    h = hashlib.sha256(json.dumps(cmd[:-1]).encode())
    for f in [header, SRC, os.path.join(b.ROOT, "include", "mcgpu_plugin.cuh")]:
        h.update(open(f, "rb").read())
    return h.hexdigest()


def build(header, nparam=None, out=None, force=False, stamp=None):
    """Compile `header` into a plugin cubin and return its path.  nparam overrides the header's
    MCGPU_PLUGIN_NPARAM (headers that allow it guard their #define with #ifndef); stamp replaces the kernel-source
    stamp (tests of the engine's refusal).  Rebuilds only when the header, the kernel sources, the flags or the
    arguments changed since `out` was built."""
    if out is None:
        stem = os.path.splitext(os.path.abspath(header))[0]
        out = stem + ("" if nparam is None else "_d%d" % nparam) + ".cubin"
    cmd = command(header, out, nparam, stamp)
    key, keyfile = _key(header, cmd), out + ".key"
    if not force and os.path.exists(out) and os.path.exists(keyfile) and open(keyfile).read() == key:
        return out
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("plugin build failed for %s:\n%s\n%s" % (header, r.stdout, r.stderr))
    with open(keyfile, "w") as f:
        f.write(key)
    return out


def build_shipped(force=False):
    """The plugins of SHIPPED into mcpar_b200/plugins/ (build.py runs this)."""
    with ThreadPoolExecutor(max_workers=len(SHIPPED)) as ex:
        return list(ex.map(lambda s: build(s[0], s[1], os.path.join(PLUGINS, s[2]), force), SHIPPED))


def shipped(name):
    """Path of a shipped plugin cubin, e.g. shipped("logistic.cubin")."""
    return os.path.join(PLUGINS, name)


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m mcpar_b200.plugin", description=__doc__.split("\n\n")[0])
    ap.add_argument("header")
    ap.add_argument("-o", "--out", default=None)
    ap.add_argument("--nparam", type=int, default=None)
    ap.add_argument("--force", action="store_true")
    a = ap.parse_args(argv)
    print(build(a.header, a.nparam, a.out, a.force))


if __name__ == "__main__":
    sys.exit(main())
