"""numpy reference of the history diagnostics (include/mcgpu.h: mcgpu_history_diag_partials, mcgpu_diag_finalize,
mcgpu_history_quantiles).

- partials(rows, G, L): the partial block of a host array rows[n][C][ncol], field for field;
- a line-for-line port of ArviZ's _split_chains, _rhat, _ess and _mcse_mean (arviz/stats/diagnostics.py; the
  autocovariance is the direct sum instead of ArviZ's FFT, the same quantity without its rounding);
- nested_rhat: Margossian et al., "Nested R-hat: assessing the convergence of MCMC when running many short chains".
"""
import numpy as np

FIELDS = ["mean", "sd", "mcse_mean", "rhat_split", "rhat_nested", "ess_mean", "ess_truncated", "nonfinite"]


def default_lag(n):
    return max(1, n // 2 - 2)


def partials(rows, G=1, L=None):
    """The block mcgpu_history_diag_partials computes from rows[n][C][ncol] (kept step, chain, column)."""
    rows = np.asarray(rows, dtype=np.float64)
    n, C, ncol = rows.shape
    N = n // 2
    L = default_lag(n) if L is None else L
    K = C // G
    blk = [float(n), float(G), float(L), float(ncol)]
    for j in range(ncol):
        x = rows[:, :, j].T                                   # [C][n]
        f = np.zeros(16 + L)
        fin = ~np.isnan(x)
        f[0] = np.count_nonzero(~np.isfinite(x))
        f[1] = x[fin].min() if fin.any() else np.inf
        f[2] = x[fin].max() if fin.any() else -np.inf
        xbar = x.mean(axis=1)
        s2 = x.var(axis=1, ddof=1)
        f[3], f[4] = C, xbar.mean()
        f[5], f[6] = np.sum((xbar - f[4]) ** 2), s2.sum()
        xg = xbar.reshape(K, G)
        xk = xg.mean(axis=1)
        bk = np.sum((xg - xk[:, None]) ** 2, axis=1) / (G - 1) if G > 1 else np.zeros(K)
        wk = s2.reshape(K, G).mean(axis=1)
        f[7], f[8] = K, xk.mean()
        f[9], f[10] = np.sum((xk - f[8]) ** 2), np.sum(bk + wk)
        y = _split_chains(x)
        ybar = y.mean(axis=1)
        f[11], f[12] = y.shape[0], ybar.mean()
        f[13], f[14] = np.sum((ybar - f[12]) ** 2), y.var(axis=1, ddof=1).sum()
        yc = y - ybar[:, None]
        for t in range(L + 1):
            f[15 + t] = np.sum(yc[:, :N - t] * yc[:, t:]) / N
        blk.extend(f)
    return np.array(blk)


# ---- ArviZ (arviz/stats/diagnostics.py), ary is [chain][draw] -------------------------------------------------------
def _split_chains(ary):
    ary = np.asarray(ary)
    if len(ary.shape) <= 1:
        ary = np.atleast_2d(ary)
    _, n_draw = ary.shape
    half = n_draw // 2
    return np.vstack((ary[:, :half], ary[:, -half:]))


def _autocov(ary):
    """Biased autocovariance along the draws, all lags (ArviZ autocov, by direct sums)."""
    n = ary.shape[1]
    z = ary - ary.mean(axis=1, keepdims=True)
    cov = np.empty_like(z)
    for t in range(n):
        cov[:, t] = np.sum(z[:, :n - t] * z[:, t:], axis=1)
    return cov / n


def _not_valid(ary, min_draws=1, min_chains=1):
    return (not np.all(np.isfinite(ary))) or ary.shape[0] < min_chains or ary.shape[1] < min_draws


def _rhat(ary):
    ary = np.asarray(ary, dtype=float)
    if _not_valid(ary):
        return np.nan
    _, num_samples = ary.shape
    chain_mean = np.mean(ary, axis=1)
    chain_var = np.var(ary, axis=1, ddof=1)
    between_chain_variance = num_samples * np.var(chain_mean, axis=None, ddof=1)
    within_chain_variance = np.mean(chain_var)
    return np.sqrt((between_chain_variance / within_chain_variance + num_samples - 1) / (num_samples))


def _ess(ary):
    ary = np.asarray(ary, dtype=float)
    if _not_valid(ary):
        return np.nan
    if (np.max(ary) - np.min(ary)) < np.finfo(float).resolution:
        return ary.size
    n_chain, n_draw = ary.shape
    acov = _autocov(ary)
    chain_mean = ary.mean(axis=1)
    mean_var = np.mean(acov[:, 0]) * n_draw / (n_draw - 1.0)
    var_plus = mean_var * (n_draw - 1.0) / n_draw
    if n_chain > 1:
        var_plus += np.var(chain_mean, axis=None, ddof=1)

    rho_hat_t = np.zeros(n_draw)
    rho_hat_even = 1.0
    rho_hat_t[0] = rho_hat_even
    rho_hat_odd = 1.0 - (mean_var - np.mean(acov[:, 1])) / var_plus
    rho_hat_t[1] = rho_hat_odd

    # Geyer's initial positive sequence
    t = 1
    while t < (n_draw - 3) and (rho_hat_even + rho_hat_odd) > 0.0:
        rho_hat_even = 1.0 - (mean_var - np.mean(acov[:, t + 1])) / var_plus
        rho_hat_odd = 1.0 - (mean_var - np.mean(acov[:, t + 2])) / var_plus
        if (rho_hat_even + rho_hat_odd) >= 0:
            rho_hat_t[t + 1] = rho_hat_even
            rho_hat_t[t + 2] = rho_hat_odd
        t += 2

    max_t = t - 2
    # improve estimation
    if rho_hat_even > 0:
        rho_hat_t[max_t + 1] = rho_hat_even

    # Geyer's initial monotone sequence
    t = 1
    while t <= max_t - 2:
        if (rho_hat_t[t + 1] + rho_hat_t[t + 2]) > (rho_hat_t[t - 1] + rho_hat_t[t]):
            rho_hat_t[t + 1] = (rho_hat_t[t - 1] + rho_hat_t[t]) / 2.0
            rho_hat_t[t + 2] = rho_hat_t[t + 1]
        t += 2

    ess = n_chain * n_draw
    tau_hat = -1.0 + 2.0 * np.sum(rho_hat_t[: max_t + 1]) + np.sum(rho_hat_t[max_t + 1: max_t + 2])
    tau_hat = max(tau_hat, 1 / np.log10(ess))
    ess = ess / tau_hat
    if np.isnan(rho_hat_t).any():
        ess = np.nan
    return ess


def _ess_mean(ary):
    return _ess(_split_chains(ary))


def _mcse_mean(ary):
    ary = np.asarray(ary)
    if _not_valid(ary, min_draws=4, min_chains=1):
        return np.nan
    ess = _ess_mean(ary)
    sd = np.std(ary, ddof=1)
    return sd / np.sqrt(ess)


def nested_rhat(ary, G):
    """sqrt(1 + Bhat / What) over K = chains / G superchains of G consecutive chains (NaN when K < 2)."""
    ary = np.asarray(ary, dtype=float)
    C = ary.shape[0]
    K = C // G
    if K < 2:
        return np.nan
    xbar = ary.mean(axis=1).reshape(K, G)
    s2 = ary.var(axis=1, ddof=1).reshape(K, G)
    xk = xbar.mean(axis=1)
    bt = xbar.var(axis=1, ddof=1) if G > 1 else np.zeros(K)
    wt = s2.mean(axis=1)
    return np.sqrt(1.0 + np.var(xk, ddof=1) / np.mean(bt + wt))


def report(rows, G=1):
    """The per-column report from the raw rows[n][C][ncol] through the ArviZ port (no truncation)."""
    rows = np.asarray(rows, dtype=np.float64)
    ncol = rows.shape[2]
    out = {k: np.empty(ncol) for k in FIELDS}
    for j in range(ncol):
        x = rows[:, :, j].T
        nf = np.count_nonzero(~np.isfinite(x))
        out["nonfinite"][j] = nf
        if nf:
            for k in FIELDS[:-1]:
                out[k][j] = np.nan
            continue
        out["mean"][j] = x.mean()
        out["sd"][j] = np.std(x, ddof=1)
        out["ess_truncated"][j] = 0.0
        if x.max() - x.min() < np.finfo(float).resolution:
            out["ess_mean"][j] = _split_chains(x).size
            out["mcse_mean"][j] = 0.0
            out["rhat_split"][j] = out["rhat_nested"][j] = np.nan
            continue
        out["rhat_split"][j] = _rhat(_split_chains(x))
        out["rhat_nested"][j] = nested_rhat(x, G)
        out["ess_mean"][j] = _ess_mean(x)
        out["mcse_mean"][j] = _mcse_mean(x)
    return out


def assert_blocks_close(got, want, rtol=1e-12):
    """Equal to rtol relative, each field's tolerance floored at rtol times the largest magnitude of that field over
    the columns (sums that nearly cancel, such as long-lag autocovariances, carry absolute rounding)."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and np.array_equal(got[:4], want[:4]), (got[:4], want[:4])
    ncol, L = int(want[3]), int(want[2])
    g, w = got[4:].reshape(ncol, 16 + L), want[4:].reshape(ncol, 16 + L)
    scale = np.nanmax(np.where(np.isfinite(w), np.abs(w), 0), axis=0, keepdims=True)
    lag_scale = np.max(np.abs(w[:, 15:]), axis=1, keepdims=True)
    scale = np.maximum(scale, np.concatenate([np.zeros((ncol, 15)), np.broadcast_to(lag_scale, (ncol, L + 1))], axis=1))
    ok = (g == w) | (np.abs(g - w) <= rtol * np.maximum(np.abs(w), scale))
    assert ok.all(), "fields differ at (column, field) %s: got %s want %s" % (
        np.argwhere(~ok)[:5].tolist(), g[~ok][:5], w[~ok][:5])


def assert_reports_close(got, want, rtol=1e-12):
    """Equal to rtol relative; the mean, which may sit near 0, to rtol times the column's sd."""
    for k in FIELDS:
        g, w = np.asarray(got[k]), np.asarray(want[k])
        assert np.array_equal(np.isnan(g), np.isnan(w)), (k, g, w)
        m = ~np.isnan(w)
        atol = rtol * np.abs(np.asarray(want["sd"])[m]) if k == "mean" else 0
        assert np.allclose(g[m], w[m], rtol=rtol, atol=atol), (k, g, w)
