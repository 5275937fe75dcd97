"""Pareto-smoothed importance-sampling leave-one-out (PSIS-LOO), one row at a time in plain numpy.

Restates the published algorithm -- Vehtari, Gelman & Gabry (2017) with the generalised Pareto fit of Zhang &
Stephens (2009) and Vehtari's weakly informative prior on k, as ArviZ's _psislw / _gpdfit compute it with r_eff = 1
-- step for step as include/spmf_b200.h states it for spmf_psis_loo.  This is the reference the kernel
(csrc/spmf_loo.cu) and PoissonFactorization.loo are checked against."""
import math

import numpy as np

LOG_DBL_MIN = float(np.log(np.finfo(np.float64).tiny))
DBL_EPS = float(np.finfo(np.float64).eps)


def tail_length(S):
    """M = ceil(min(0.2 S, 3 sqrt(S))), capped at S - 1 (at S = 1 there is no value below the tail)."""
    return min(int(math.ceil(min(0.2 * S, 3.0 * math.sqrt(S)))), S - 1)


def grid_size(n):
    return 30 + int(math.floor(math.sqrt(n)))


def quartile_index(n):
    return int(n / 4.0 + 0.5) - 1


def grid_b(j, m, y_last, y_quart):
    """Grid point b_j (j = 1..m) of the profile fit."""
    return (1.0 - math.sqrt(m / (j - 0.5))) / (3.0 * y_quart) + 1.0 / y_last


def profile(n, b, k):
    """Profile log-likelihood n (log(-b/k) - k - 1) of grid point b, k = mean log1p(-b y)."""
    with np.errstate(divide='ignore', invalid='ignore'):
        return n * (np.log(-(b / k)) - k - 1.0)


def gpd_quantile(p, k, sigma):
    """Generalised Pareto quantile (location 0); the exponential one when |k| < eps."""
    if abs(k) < DBL_EPS:
        return sigma * -np.log1p(-p)
    return np.expm1(-k * np.log1p(-p)) / k * sigma


def gpdfit(y):
    """(k-hat with the prior, sigma) of the generalised Pareto fit to the ascending exceedances y."""
    n = len(y)
    m = grid_size(n)
    b = np.array([grid_b(j, m, y[-1], y[quartile_index(n)]) for j in range(1, m + 1)])
    with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
        k = np.log1p(-b[:, None] * y[None, :]).mean(1)
        L = profile(n, b, k)
        w = 1.0 / np.exp(L[None, :] - L[:, None]).sum(1)        # row j: sum_i exp(L_i - L_j); overflow -> w_j = 0
        keep = w >= 10.0 * DBL_EPS
        w, b = w[keep], b[keep]
        w = w / w.sum()
        bhat = (b * w).sum()
        kk = np.log1p(-bhat * y).mean()
        sigma = -kk / bhat
    return (n * kk + 5.0) / (n + 10.0), sigma


def _logsumexp(x):
    m = np.max(x)
    if m == -np.inf:
        return -np.inf
    return m + np.log(np.sum(np.exp(x - m)))


def psis_loo_row(ll):
    """(elpd, lppd, khat) of one row of per-draw log-likelihoods."""
    ll = np.asarray(ll, np.float64)
    S = ll.size
    if np.isnan(ll).any() or (ll == np.inf).any():
        return np.nan, np.nan, np.nan
    lppd = _logsumexp(ll) - np.log(S)
    if (ll == -np.inf).any():
        return -np.inf, lppd, np.inf
    r = -ll
    r = r - r.max()
    M = tail_length(S)
    srt = np.sort(r)
    cut = max(srt[S - 1 - M], LOG_DBL_MIN)
    tail = np.flatnonzero(r > cut)
    n = tail.size
    khat = np.inf
    if n > 4:
        order = tail[np.argsort(r[tail], kind='stable')]
        y = np.exp(r[order]) - np.exp(cut)
        khat, sigma = gpdfit(y)
        if np.isfinite(khat) and np.isfinite(sigma) and sigma > 0:
            p = (np.arange(n) + 0.5) / n
            r[order] = np.log(np.array([gpd_quantile(pi, khat, sigma) for pi in p]) + np.exp(cut))
            r[r > 0] = 0.0
        else:
            khat = np.inf
    lw = r - _logsumexp(r)
    return _logsumexp(lw + ll), lppd, khat


def psis_loo(ll):
    """Rows of an (N, S) matrix: (elpd, lppd, khat), each of shape (N,)."""
    out = np.array([psis_loo_row(row) for row in np.asarray(ll, np.float64)], np.float64).reshape(-1, 3)
    return out[:, 0], out[:, 1], out[:, 2]
