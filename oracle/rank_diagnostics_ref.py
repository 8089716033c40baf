"""Restatement of the rank-normalised convergence diagnostics (pxmcmc_b200.diagnostics.rank_diagnostics, DESIGN.md 7b)
in numpy / scipy: Vehtari, Gelman, Simpson, Carpenter & Buerkner (2021), as ArviZ's rhat(method="rank") and
ess(method="bulk" | "tail").  Written from the definition, not checked against ArviZ.  Ranks come from
scipy.stats.rankdata, z from scipy.special.ndtri and the autocovariance from np.fft -- deliberately another route than
the device's direct lag sums.

For one parameter x[c, i] (m chains, n samples, S = m n, h = n // 2):
  split(x)  the M = 2m series x[c, :h] and x[c, n - h:] (the middle sample of odd n is in none);
  z(y)      Phi^-1((r - 3/8) / (N + 1/4)), r the average rank among all N values of y;
  R(y)      sqrt((B / W + h - 1) / h), B = h var(series means, ddof 1), W = mean series variance (ddof 1);
  rhat      max(R(z(split(x))), R(z(split(|x - median|)))), NaN when either is NaN;
  ESS(y)    Geyer's initial positive / monotone sequence (`ess` below);
  ess_bulk  ESS(z(split(x)));  ess_tail  min(ESS(split(1[x <= q05])), ESS(split(1[x <= q95]))).
All three are NaN when n < 4 or a value is not finite.
"""
import numpy as np
from scipy.special import ndtri
from scipy.stats import rankdata


def split(x):
    """[m, n] -> [2m, n // 2]: the first halves of every chain, then the second halves"""
    x = np.asarray(x, dtype=np.float64)
    h = x.shape[1] // 2
    return np.concatenate([x[:, :h], x[:, x.shape[1] - h:]], axis=0)


def z_scale(y):
    r = rankdata(y, method="average").reshape(y.shape)
    return ndtri((r - 0.375) / (y.size + 0.25))


def R(series):
    h = series.shape[1]
    B = h * np.var(series.mean(axis=1), ddof=1)
    W = np.mean(np.var(series, axis=1, ddof=1))
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.sqrt((B / W + h - 1) / h)


def autocov(series):
    """acov_k(t) = (1/h) sum_{i < h - t} (y_k[i] - mean_k) (y_k[i + t] - mean_k), through a zero-padded FFT"""
    h = series.shape[1]
    c = series - series.mean(axis=1, keepdims=True)
    nfft = 1 << (2 * h - 1).bit_length()
    f = np.fft.rfft(c, n=nfft, axis=1)
    return np.fft.irfft(f * np.conj(f), n=nfft, axis=1)[:, :h] / h


def ess(series):
    M, h = series.shape
    if np.max(series) - np.min(series) < np.finfo(float).resolution:
        return float(M * h)
    acov = autocov(series)
    mean_var = np.mean(acov[:, 0]) * h / (h - 1)
    var_plus = mean_var * (h - 1) / h + np.var(series.mean(axis=1), ddof=1)

    def rho(t):
        return 1.0 - (mean_var - np.mean(acov[:, t])) / var_plus

    r = np.zeros(h)
    r[0] = ev = 1.0
    r[1] = od = rho(1)
    t = 1
    while t < h - 3 and ev + od > 0:
        ev, od = rho(t + 1), rho(t + 2)
        if ev + od >= 0:
            r[t + 1], r[t + 2] = ev, od
        t += 2
    T = t - 2
    if ev > 0:
        r[T + 1] = ev
    t = 1
    while t <= T - 2:
        if r[t + 1] + r[t + 2] > r[t - 1] + r[t]:
            r[t + 1] = r[t + 2] = (r[t - 1] + r[t]) / 2
        t += 2
    tau = max(-1 + 2 * np.sum(r[:T + 1]) + np.sum(r[T + 1:T + 2]), 1 / np.log10(M * h))
    return M * h / tau


def column(x):
    """(rhat, ess_bulk, ess_tail) of one parameter, x: [m, n]"""
    x = np.asarray(x, dtype=np.float64)
    if x.shape[1] < 4 or not np.all(np.isfinite(x)):
        return np.nan, np.nan, np.nan
    zb = z_scale(split(x))
    zf = z_scale(split(np.abs(x - np.median(x))))
    rb, rf = R(zb), R(zf)
    rhat = np.nan if np.isnan(rb) or np.isnan(rf) else max(rb, rf)
    q05, q95 = np.quantile(x, 0.05), np.quantile(x, 0.95)
    tail = min(ess(split((x <= q05).astype(np.float64))), ess(split((x <= q95).astype(np.float64))))
    return rhat, ess(zb), tail


def rank_diagnostics(chains):
    """chains: [m, n, nparams] (or [n, nparams], one chain) -> (rhat, ess_bulk, ess_tail), each [nparams]"""
    x = np.asarray(chains, dtype=np.float64)
    if x.ndim == 2:
        x = x[None]
    out = np.array([column(x[:, :, j]) for j in range(x.shape[2])]).reshape(-1, 3)
    return out[:, 0].copy(), out[:, 1].copy(), out[:, 2].copy()
