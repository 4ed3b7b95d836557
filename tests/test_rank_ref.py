"""The device's decomposition of ArviZ's rank-normalised diagnostics (a [2N][C][4] series of normal scores, folded
normal scores and tail indicators, reduced by the partials and mcgpu_diag_finalize) against the direct port of
ArviZ (tests/rank_ref.py).  Host arithmetic only; needs no GPU."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import diag_ref  # noqa: E402
import rank_ref  # noqa: E402


def ar1(rng, C, n, phi):
    x = np.empty((C, n))
    x[:, 0] = rng.standard_normal(C)
    for t in range(1, n):
        x[:, t] = phi * x[:, t - 1] + np.sqrt(1 - phi * phi) * rng.standard_normal(C)
    return x


def tied(rng):
    """Values rounded to 0.1 and every draw repeated once (a rejected step repeats the chain's value)."""
    x = np.round(ar1(rng, 24, 21, 0.5), 1)
    return np.repeat(x, 2, axis=1)


def scale_mixture(rng):
    """Equal means, chain scales 1 and 6: the split R-hat of the raw draws stays near 1, the folded one does not."""
    return rng.standard_normal((32, 60)) * np.repeat([1.0, 6.0], 16)[:, None]


CASES = {
    "iid": lambda r: r.standard_normal((16, 40)),
    "ar1": lambda r: ar1(r, 32, 64, 0.8) + 3.0,
    "odd_n": lambda r: ar1(r, 16, 37, 0.4),
    "tied": tied,
    "constant": lambda r: np.full((8, 20), 2.5),
    "shifted_means": lambda r: r.standard_normal((16, 30)) + 4.0 * (np.arange(16)[:, None] % 3),
    "scale_mixture": scale_mixture,
    "one_chain": lambda r: ar1(r, 1, 40, 0.3),
}


def direct(x):
    return rank_ref.report(x.T[:, :, None])


@pytest.mark.parametrize("case", sorted(CASES))
def test_decomposition_matches_the_port(case):
    x = CASES[case](np.random.default_rng(11))
    got, want = rank_ref.decomposed(x), direct(x)
    rank_ref.assert_reports_close(got, want, rtol=1e-12)


def test_case_properties():
    rng = np.random.default_rng(11)
    x = tied(rng)
    assert len(np.unique(x)) < x.size / 4                       # ties are the normal case here
    r = direct(CASES["shifted_means"](np.random.default_rng(11)))
    assert r["rhat"][0] > 2.0
    c = direct(CASES["constant"](None))
    assert np.isnan(c["rhat"][0]) and c["ess_bulk"][0] == 8 * 20 and c["ess_tail"][0] == 8 * 20
    x = scale_mixture(np.random.default_rng(11))
    r = direct(x)
    assert diag_ref._rhat(diag_ref._split_chains(x)) < 1.05 and r["rhat_bulk"][0] < 1.05
    assert r["rhat_tail"][0] > 1.2 and r["rhat"][0] == r["rhat_tail"][0]
    assert np.isnan(direct(CASES["one_chain"](np.random.default_rng(11)))["rhat"][0])


def test_bulk_is_invariant_under_a_monotone_map():
    x = ar1(np.random.default_rng(5), 16, 50, 0.6)
    ex = np.exp(x)
    assert len(np.unique(ex)) == len(np.unique(x)) == x.size   # exp creates no new ties
    a, b = rank_ref.decomposed(x), rank_ref.decomposed(ex)
    for k in ("rhat_bulk", "ess_bulk"):
        assert a[k] == pytest.approx(b[k], rel=1e-12), k


def test_nonfinite_column_reports_only_its_count():
    rows = np.random.default_rng(3).standard_normal((20, 8, 2))
    rows[4, 3, 1] = np.nan
    rows[7, 1, 1] = -np.inf
    r = rank_ref.report(rows)
    assert r["nonfinite"].tolist() == [0.0, 2.0]
    assert all(np.isnan(r[k][1]) for k in rank_ref.FIELDS[:-1]) and not np.isnan(r["rhat"][0])


def test_truncation_flag_follows_the_lag_limit():
    x = ar1(np.random.default_rng(2), 16, 80, 0.95)
    assert rank_ref.decomposed(x)["ess_truncated"] == 0.0
    assert rank_ref.decomposed(x, L=2)["ess_truncated"] == 1.0
