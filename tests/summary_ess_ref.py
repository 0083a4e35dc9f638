"""Test infrastructure: the numpy stand-in of tests/summary_ref.py with amwg_summary_autocov added (direct sums), and an
independent reference ESS (FFT autocovariances over whole half-chains, then the ArviZ `_ess` loop). Never imported by the product."""
import numpy as np

from summary_ref import NumpyBlockReducer


class NumpyEssReducer(NumpyBlockReducer):
    lag_tile = 16

    def __init__(self, lag_tile=16):
        self.lag_tile = lag_tile

    def autocov(self, block, thresholds, live, lag0, n_lags):
        x = block.numpy()                                    # [rows, entries, chains]
        rows, entries, chains = x.shape
        h = rows // 2
        out = np.zeros((len(live), 3 + n_lags))
        for i, e in enumerate(live):
            y = x[:, e, :]
            if thresholds is not None:
                y = (y <= thresholds[e]).astype(np.float64)
            halves = np.concatenate([y[:h], y[rows - h:]], axis=1)      # [h, 2 * chains]
            m = halves.sum(axis=0) / h
            c = halves - m
            mm = m.mean()
            out[i, :3] = (2 * chains, mm, ((m - mm) ** 2).sum())
            for j in range(n_lags):
                t = lag0 + j
                if t < h:
                    out[i, 3 + j] = np.einsum("nk,nk->", c[:h - t], c[t:])
        return out


def split_chains(y):
    """y [rows, chains] -> [2 * chains, h]: the first and last h rows of every chain."""
    rows = y.shape[0]
    h = rows // 2
    return np.concatenate([y[:h].T, y[rows - h:].T], axis=0)


def _autocov_fft(a):
    """biased autocovariance of every row of a [chains, n] over all lags (ArviZ `_autocov`)."""
    n = a.shape[1]
    c = a - a.mean(axis=1, keepdims=True)
    f = np.fft.rfft(c, n=2 * n, axis=1)
    return np.fft.irfft(f * np.conj(f), n=2 * n, axis=1)[:, :n] / n


def reference_ess(chains_draws):
    """ArviZ `_ess` (stats/diagnostics.py) on chains_draws [M', h]: split chains in, no rank normalisation."""
    ary = np.asarray(chains_draws, dtype=float)
    if not np.all(np.isfinite(ary)):
        return np.nan
    n_chain, n_draw = ary.shape
    if n_draw < 4:
        return np.nan
    acov = _autocov_fft(ary)
    chain_mean = ary.mean(axis=1)
    mean_var = np.mean(acov[:, 0]) * n_draw / (n_draw - 1.0)
    var_plus = mean_var * (n_draw - 1.0) / n_draw + np.var(chain_mean, ddof=1)
    if not var_plus > 0:
        return np.nan
    rho_hat_t = np.zeros(n_draw)
    rho_hat_even = 1.0
    rho_hat_t[0] = rho_hat_even
    rho_hat_odd = 1.0 - (mean_var - np.mean(acov[:, 1])) / var_plus
    rho_hat_t[1] = rho_hat_odd
    t = 1
    while t < (n_draw - 3) and (rho_hat_even + rho_hat_odd) > 0.0:
        rho_hat_even = 1.0 - (mean_var - np.mean(acov[:, t + 1])) / var_plus
        rho_hat_odd = 1.0 - (mean_var - np.mean(acov[:, t + 2])) / var_plus
        if (rho_hat_even + rho_hat_odd) >= 0:
            rho_hat_t[t + 1] = rho_hat_even
            rho_hat_t[t + 2] = rho_hat_odd
        t += 2
    max_t = t - 2
    if rho_hat_even > 0:
        rho_hat_t[max_t + 1] = rho_hat_even
    t = 1
    while t <= max_t - 2:
        if (rho_hat_t[t + 1] + rho_hat_t[t + 2]) > (rho_hat_t[t - 1] + rho_hat_t[t]):
            rho_hat_t[t + 1] = (rho_hat_t[t - 1] + rho_hat_t[t]) / 2.0
            rho_hat_t[t + 2] = rho_hat_t[t + 1]
        t += 2
    ess = n_chain * n_draw
    tau_hat = -1.0 + 2.0 * np.sum(rho_hat_t[: max_t + 1]) + np.sum(rho_hat_t[max_t + 1: max_t + 2])
    tau_hat = max(tau_hat, 1 / np.log10(ess))
    return ess / tau_hat


def reference_ess_block(x):
    """x [rows, entries, chains] -> (ess, ess_tail) per entry, with q05 / q95 from numpy.quantile of the pooled draws."""
    rows, entries, _ = x.shape
    ess, tail = np.empty(entries), np.empty(entries)
    for e in range(entries):
        y = x[:, e, :]
        ess[e] = reference_ess(split_chains(y))
        if not np.all(np.isfinite(y)):
            tail[e] = np.nan
            continue
        q05, q95 = np.quantile(y.ravel(), [0.05, 0.95])
        tail[e] = np.minimum(reference_ess(split_chains((y <= q05).astype(float))), reference_ess(split_chains((y <= q95).astype(float))))
    return ess, tail
