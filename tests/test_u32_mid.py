"""The remote candidate test reads its rejection uniform as (float)u32_mid(w).  The kernels form that float with
fp32 and integer operations (mcgpu::u32_mid_f32, __host__ __device__ in mcpar_b200/csrc/mcgpu_math.cuh); it
must equal the fp64 uniform narrowed to fp32 for every one of the 2^32 words, or decisions would change."""
import json
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_u32_mid_f32_matches_fp64_for_every_word(tmp_path):
    exe = str(tmp_path / "u32_mid_check")
    subprocess.check_call(["/usr/bin/g++", "-x", "c++", "-std=c++17", "-O2", "-ffp-contract=off", "-o", exe,
                           os.path.join(ROOT, "tests", "u32_mid_check.cc")])
    r = json.loads(subprocess.check_output([exe]).decode())
    assert r["mismatches"] == 0, r
    assert r["naive_mismatches"] > 0, r        # the check can tell a double rounding from the exact one
