"""numpy reference of the rank-normalised diagnostics (include/mcgpu.h: mcgpu_history_rank_diag).

- z_scale, rhat_rank, ess_bulk, ess_quantile, ess_tail: a port of ArviZ's _z_scale + _backtransform_ranks, _rhat_rank,
  _ess_bulk, _ess_quantile (with _quantile = scipy's mquantiles(alphap=1, betap=1)) and _ess_tail
  (arviz/stats/diagnostics.py), written against the port in tests/diag_ref.py;
- series / decomposed: the device's route to the same numbers, a [2N][C][4] series of normal scores, folded normal
  scores and tail indicators whose partial block (diag_ref.partials) goes through mcgpu_diag_finalize;
- report: the per-column report of rows[n][C][ncol] (kept step, chain, column) from the direct port.

Deviation from ArviZ, as in mcgpu_diag_finalize: a column holding any non-finite value (ArviZ checks for NaN only)
reports only its count.
"""
import numpy as np
from scipy import stats
from scipy.stats.mstats import mquantiles

from diag_ref import _ess, _rhat, _split_chains, default_lag

FIELDS = ["rhat", "rhat_bulk", "rhat_tail", "ess_bulk", "ess_tail", "ess_truncated", "nonfinite"]
TAIL_PROBS = (0.05, 0.95)


def z_scale(y):
    r = stats.rankdata(y, method="average", axis=None)
    r = (r - 3 / 8) / (r.size - 2 * (3 / 8) + 1)
    return stats.norm.ppf(r).reshape(y.shape)


def fold(y):
    return np.abs(y - np.median(y))


def rhat_rank(x):
    """(rhat, rhat_bulk, rhat_tail) of x[C][n]; rhat is Python's max(): NaN if bulk is NaN, bulk if only tail is."""
    if x.shape[0] < 2:
        return np.nan, np.nan, np.nan
    y = _split_chains(x)
    with np.errstate(invalid="ignore", divide="ignore"):
        bulk = _rhat(z_scale(y))
        tail = _rhat(z_scale(fold(y)))
    return max(bulk, tail), bulk, tail


def ess_bulk(x):
    return _ess(z_scale(_split_chains(x)))


def tail_threshold(x, p):
    (q,) = mquantiles(x, [p], alphap=1, betap=1)       # over all C n draws, the middle draw of odd n included
    return q


def ess_quantile(x, p):
    return _ess(_split_chains((x <= tail_threshold(x, p)).astype(float)))


def ess_tail(x):
    return min(ess_quantile(x, TAIL_PROBS[0]), ess_quantile(x, TAIL_PROBS[1]))


def report(rows):
    """The direct port over every column of rows[n][C][ncol]: a dict of per-column arrays named by FIELDS."""
    rows = np.asarray(rows, dtype=np.float64)
    ncol = rows.shape[2]
    out = {k: np.full(ncol, np.nan) for k in FIELDS}
    for j in range(ncol):
        x = rows[:, :, j].T
        out["nonfinite"][j] = np.count_nonzero(~np.isfinite(x))
        if out["nonfinite"][j]:
            continue
        out["rhat"][j], out["rhat_bulk"][j], out["rhat_tail"][j] = rhat_rank(x)
        out["ess_bulk"][j] = ess_bulk(x)
        out["ess_tail"][j] = ess_tail(x)
        out["ess_truncated"][j] = 0.0
    return out


def series(x):
    """The device's transform of one column x[C][n]: [2N][C][4], split row r of chain c (rows N..2N-1 are draws
    n-N..n-1), columns z(y), z(|y - median y|), I(x <= q_0.05), I(x <= q_0.95)."""
    C, n = x.shape
    N = n // 2
    y = np.concatenate([x[:, :N], x[:, n - N:]], axis=1).T          # [2N][C]
    s = np.empty((2 * N, C, 4))
    s[:, :, 0] = z_scale(y)
    s[:, :, 1] = z_scale(fold(y))
    for k, p in enumerate(TAIL_PROBS):
        s[:, :, 2 + k] = (y <= tail_threshold(x, p)).astype(float)
    return s


def from_series_report(rep, C):
    """The field mapping of the 4-column report of diag_finalize (DIAG_FIELDS) into FIELDS for one column."""
    out = dict.fromkeys(FIELDS, np.nan)
    bulk, tail = rep["rhat_split"][0], rep["rhat_split"][1]
    if C >= 2:
        out["rhat_bulk"], out["rhat_tail"] = bulk, tail
        out["rhat"] = max(bulk, tail)
    out["ess_bulk"] = rep["ess_mean"][0]
    out["ess_tail"] = min(rep["ess_mean"][2], rep["ess_mean"][3])
    out["ess_truncated"] = max(rep["ess_truncated"][0], rep["ess_truncated"][2], rep["ess_truncated"][3])
    out["nonfinite"] = 0.0
    return out


def decomposed(x, L=None):
    """One column x[C][n] through the device's decomposition: series -> partials (superchain 1) -> diag_finalize."""
    import diag_ref
    from mcpar_b200 import engine
    s = series(x)
    L = default_lag(s.shape[0]) if L is None else L
    return from_series_report(engine.diag_finalize([diag_ref.partials(s, 1, L)]), x.shape[0])


def assert_reports_close(got, want, rtol):
    """Equal to rtol relative, NaN where the other is NaN."""
    for k in FIELDS:
        g, w = np.atleast_1d(np.asarray(got[k], dtype=float)), np.atleast_1d(np.asarray(want[k], dtype=float))
        assert np.array_equal(np.isnan(g), np.isnan(w)), (k, g, w)
        m = ~np.isnan(w)
        assert np.allclose(g[m], w[m], rtol=rtol, atol=0), (k, g, w)
