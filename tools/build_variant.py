#!/usr/bin/env python
"""Build an A/B variant of libmcgpu.so here (no GPU needed): mh_fast.cu recompiled with extra nvcc flags and linked
with the current mh_exact.o / mcgpu_api.o / mcgpu_diag.o into mcpar_b200/variants/libmcgpu_<tag>.so (git-ignored; travels to the GPU
box).  Select it at run time with MCGPU_LIB=<path>.    python tools/build_variant.py mb9 -DMCGPU_MINB_LOCAL=9"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mcpar_b200 import build as b   # noqa: E402

tag, flags = sys.argv[1], sys.argv[2:]
b.build()                           # make sure the common objects are current
vdir = os.path.join(ROOT, "mcpar_b200", "variants")
os.makedirs(vdir, exist_ok=True)
obj = os.path.join(vdir, "mh_fast_%s.o" % tag)
cmd = [b.NVCC] + b.ARCH + b.COMMON + flags + ["-c", os.path.join(b.CSRC, "mh_fast.cu"), "-o", obj]
subprocess.check_call(cmd)
lib = os.path.join(vdir, "libmcgpu_%s.so" % tag)
subprocess.check_call([b.NVCC] + b.ARCH + ["-shared", "-Xcompiler", "-fPIC", "-ccbin", "/usr/bin/g++", "-o", lib, obj,
                       os.path.join(b.OBJ, "mh_exact.o"), os.path.join(b.OBJ, "mcgpu_api.o"),
                       os.path.join(b.OBJ, "mcgpu_diag.o")])
os.remove(obj)
print(lib)
