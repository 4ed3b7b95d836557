"""mcgpu_diag_finalize (host arithmetic, no GPU needed) against the numpy port of ArviZ's diagnostics and nested R-hat
(tests/diag_ref.py), on partial blocks computed on the host from known chains."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import diag_ref  # noqa: E402
from mcpar_b200 import engine  # noqa: E402


def ar1(rng, n, C, ncol, phi):
    """rows[n][C][ncol] of stationary AR(1) chains, unit marginal variance."""
    x = np.empty((n, C, ncol))
    x[0] = rng.standard_normal((C, ncol))
    s = np.sqrt(1 - phi * phi)
    for t in range(1, n):
        x[t] = phi * x[t - 1] + s * rng.standard_normal((C, ncol))
    return x


def finalize(rows, G=1, L=None, nsplit=1):
    """diag_finalize over the blocks of nsplit equal contiguous chain shards."""
    return engine.diag_finalize([diag_ref.partials(r, G, L) for r in np.split(rows, nsplit, axis=1)])


def shifted(rng, n, C, ncol, G, offset):
    x = rng.standard_normal((n, C, ncol))
    return x + offset * np.repeat(rng.standard_normal(C // G), G)[None, :, None]


CASES = {
    "iid": lambda r: r.standard_normal((40, 64, 3)) * [1.0, 3.0, 0.1] + [0.0, 1e3, -7.0],
    "ar1": lambda r: ar1(r, 60, 64, 3, 0.7),
    "superchain_shift": lambda r: shifted(r, 40, 64, 2, 8, 0.5),
    "odd_n": lambda r: ar1(r, 37, 32, 3, 0.4) + 2.0,
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("G", [1, 8, "C"])
def test_finalize_matches_the_arviz_port(case, G):
    rows = CASES[case](np.random.default_rng(11))
    G = rows.shape[1] if G == "C" else G
    got = finalize(rows, G)
    want = diag_ref.report(rows, G)
    diag_ref.assert_reports_close(got, want)
    assert np.all(got["ess_truncated"] == 0) and np.all(got["nonfinite"] == 0)
    if G == rows.shape[1]:
        assert np.all(np.isnan(got["rhat_nested"]))          # one superchain: K < 2


# phi = 0.9 runs longer chains: at 400 draws (N = 200 per split chain, tau = 19) ArviZ's estimator itself reads about
# 24 % low over 4096 chains -- the centred autocovariances keep the positive-sequence sum positive out to large lags,
# and the more chains, the less noise stops it early -- while finalize equals the ArviZ port on the same data
@pytest.mark.parametrize("phi,C,n", [(0.5, 4096, 400), (0.9, 1024, 1600)])
def test_ess_of_ar1_chains_matches_theory(phi, C, n):
    rows = ar1(np.random.default_rng(5), n, C, 1, phi)
    got = finalize(rows)
    theory = 2 * C * (n // 2) * (1 - phi) / (1 + phi)
    assert abs(got["ess_mean"][0] / theory - 1) < 0.10, (got["ess_mean"][0], theory)
    assert abs(got["mcse_mean"][0] - got["sd"][0] / np.sqrt(got["ess_mean"][0])) < 1e-15


def test_rhat_flags_superchain_offsets():
    rng = np.random.default_rng(2)
    iid = rng.standard_normal((100, 256, 1))
    r = finalize(iid, 8)
    assert r["rhat_split"][0] < 1.01 and r["rhat_nested"][0] < 1.01
    off = iid + np.repeat(rng.standard_normal(32), 8)[None, :, None]    # superchain offsets of 1 sd
    assert finalize(off, 8)["rhat_nested"][0] > 1.1


@pytest.mark.parametrize("nsplit", [2, 4])
def test_sharded_blocks_merge_to_the_one_block_report(nsplit):
    rows = ar1(np.random.default_rng(3), 50, 64, 3, 0.6) + [0.0, 50.0, -3.0]
    one = finalize(rows, 4)
    many = finalize(rows, 4, nsplit=nsplit)
    diag_ref.assert_reports_close(many, one)


def test_small_max_lag_sets_ess_truncated():
    rows = ar1(np.random.default_rng(4), 200, 64, 1, 0.95)
    assert finalize(rows, 1, L=4)["ess_truncated"][0] == 1
    assert finalize(rows, 1)["ess_truncated"][0] == 0


def test_constant_and_nonfinite_columns():
    rng = np.random.default_rng(6)
    rows = rng.standard_normal((20, 16, 3))
    rows[:, :, 1] = 2.5
    rows[3, 5, 2] = np.inf; rows[7, 2, 2] = np.nan
    r = finalize(rows, 4)
    assert r["ess_mean"][1] == 2 * 16 * 10 and r["mcse_mean"][1] == 0 and r["mean"][1] == 2.5
    assert np.isnan(r["rhat_split"][1]) and np.isnan(r["rhat_nested"][1])
    assert r["nonfinite"][2] == 2 and r["nonfinite"][0] == 0 and r["nonfinite"][1] == 0
    assert all(np.isnan(r[k][2]) for k in diag_ref.FIELDS if k != "nonfinite")
    assert np.isfinite(r["rhat_split"][0])


def test_mismatched_or_malformed_blocks_are_refused():
    rows = np.random.default_rng(7).standard_normal((20, 16, 2))
    a = diag_ref.partials(rows, 4, 5)
    for other in (diag_ref.partials(rows, 2, 5), diag_ref.partials(rows[:18], 4, 5)):
        with pytest.raises(engine.McgpuError, match="EINVAL"):
            engine.diag_finalize([a, other])
    for field, value in ((0, 3.0), (0, 10.5), (1, 0.0)):     # n < 4, n not whole (max_lag 5 > N - 1 = 4), G = 0
        bad = a.copy(); bad[field] = value
        with pytest.raises(engine.McgpuError, match="EINVAL"):
            engine.diag_finalize([bad])
    with pytest.raises(ValueError):
        engine.diag_finalize([a, a[:-1]])
