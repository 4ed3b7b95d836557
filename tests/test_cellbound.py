"""The d = 2 table of acceptance-ratio bounds (mcpar_b200/csrc/mcgpu_cellbound.cuh) lets a remote candidate skip the
pool loop when its cell's bounds settle the uniform.  That keeps every decision only if the bounds hold: compile the
bound routine for the host and check it against an x86 extended-precision evaluation of remote_exact's ratio over
pools of several shapes, at random points, cell corners and the edges of the dilated cells."""
import json
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cell_bounds_contain_the_extended_precision_ratio(tmp_path):
    exe = str(tmp_path / "cellbound_check")
    subprocess.check_call(["/usr/bin/g++", "-x", "c++", "-std=c++17", "-O2", "-o", exe,
                           os.path.join(ROOT, "tests", "cellbound_check.cc")])
    rows = [json.loads(l) for l in subprocess.check_output([exe]).decode().splitlines()]
    assert len(rows) == 7
    for r in rows:
        assert r["violations"] == 0 and r["store_violations"] == 0, r
        assert r["points"] > 10000, r
    by = {r["shape"]: r for r in rows}
    # not vacuous: where the pool is alike, most cells are decidable and tight
    for name in ("plateau_like", "plateau_like_256", "random"):
        assert by[name]["decidable"] > 0.5 * by[name]["cells"], by[name]
    assert 0.0 <= by["plateau_like"]["median_rel_width"] < 0.5, by["plateau_like"]
