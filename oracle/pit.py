"""LOO-PIT, one step at a time in numpy / scipy on materialised (S, B, D) rates.

Restates include/spmf_b200.h's contracts of spmf_loo_pit_accum and spmf_loo_pit_hist and the summary of
PoissonFactorization.loo_pit: the PSIS weights of every (row, draw) (oracle/psis.py), the predictive CDFs of every
entry (scipy.stats.poisson.cdf, scipy.special.expit), their weighted sums P- and P+, the non-randomised PIT of
Czado, Gneiting & Held (2009) binned into J bins, and the per-feature and overall summaries.  This is the reference
the kernels (csrc/spmf_pit.cu) and loo_pit are checked against."""
import numpy as np
import scipy.special as sp
import scipy.stats as st

from oracle import psis

MAX_VALUE = 2.0 ** 24


def psis_lw_row(ll):
    """The normalised smoothed log weights lw (S,) of one row, in draw order: steps 1-4 of spmf_psis_loo as
    oracle/psis.py's psis_loo_row takes them (its helpers, the same tail, fit, smoothing and truncation); NaN where
    step 5 applies (the row holds -inf, NaN or +inf)."""
    ll = np.asarray(ll, np.float64)
    S = ll.size
    if not np.isfinite(ll).all():
        return np.full(S, np.nan)
    r = -ll
    r = r - r.max()
    M = psis.tail_length(S)
    cut = max(np.sort(r)[S - 1 - M], psis.LOG_DBL_MIN)
    tail = np.flatnonzero(r > cut)
    n = tail.size
    if n > 4:
        order = tail[np.argsort(r[tail], kind='stable')]
        khat, sigma = psis.gpdfit(np.exp(r[order]) - np.exp(cut))
        if np.isfinite(khat) and np.isfinite(sigma) and sigma > 0:
            p = (np.arange(n) + 0.5) / n
            r[order] = np.log(np.array([psis.gpd_quantile(pi, khat, sigma) for pi in p]) + np.exp(cut))
            r[r > 0] = 0.0
    return r - psis._logsumexp(r)


def loo_weights(ll):
    """(lw (B, S), elpd (B,), khat (B,)) of per-row log-likelihoods ll (B, S)."""
    ll = np.asarray(ll, np.float64)
    elpd, _, khat = psis.psis_loo(ll)
    return np.array([psis_lw_row(row) for row in ll]).reshape(ll.shape), elpd, khat


def entry_cdfs(x, rate, bernoulli):
    """(F(x - 1), F(x), valid) of every (s, b, d): rate (S, B, D) = the Poisson rate or the Bernoulli logit,
    x (B, D) the observed values.  Invalid: a Poisson rate that is negative, not finite or above 2^24, a logit that
    is not finite, or x not an integer of the support; their CDFs are 0."""
    rate = np.asarray(rate, np.float64)
    x = np.broadcast_to(np.asarray(x, np.float64), rate.shape)
    with np.errstate(invalid='ignore'):
        x_ok = (x >= 0) & (x == np.floor(x)) & (x <= (1.0 if bernoulli else MAX_VALUE))
        if bernoulli:
            ok = np.isfinite(rate) & x_ok
            f0 = sp.expit(-np.where(ok, rate, 0.0))
            fm = np.where(x >= 1, f0, 0.0)
            fp = np.where(x >= 1, 1.0, f0)
        else:
            ok = np.isfinite(rate) & (rate >= 0) & (rate <= MAX_VALUE) & x_ok
            lam = np.where(ok, rate, 1.0)
            xs = np.where(ok, x, 0.0)
            fm = st.poisson.cdf(xs - 1, lam)
            fp = st.poisson.cdf(xs, lam)
    return np.where(ok, fm, 0.0), np.where(ok, fp, 0.0), ok


def pit_values(x, rate, lw, bernoulli):
    """(P (B, D, 2), n_invalid (B, D)): P[..., 0] = sum_s exp(lw_bs) F(x_bd - 1 | theta_s), P[..., 1] the same of
    F(x_bd), summed in ascending s over the valid draws; n_invalid = the invalid draws of every entry."""
    fm, fp, ok = entry_cdfs(x, rate, bernoulli)
    w = np.exp(np.asarray(lw, np.float64)).T[:, :, None]        # (S, B, 1)
    P = np.zeros(fm.shape[1:] + (2,))
    for s in range(fm.shape[0]):
        P[..., 0] += w[s] * fm[s]
        P[..., 1] += w[s] * fp[s]
    return P, (~ok).sum(0)


def czado_bins(pm, pp, J):
    """(n, J) bin masses of entries (pm, pp): F((j+1)/J) - F(j/J) of F(u) = clip((u - lo)/(hi - lo), 0, 1), lo, hi
    the values clamped to [0, 1]; unit mass in bin min(J - 1, floor(hi J)) where hi <= lo."""
    lo = np.clip(np.asarray(pm, np.float64).ravel(), 0, 1)[:, None]
    hi = np.clip(np.asarray(pp, np.float64).ravel(), 0, 1)[:, None]
    u = np.arange(J + 1)[None, :] / J
    with np.errstate(divide='ignore', invalid='ignore'):
        F = np.where(u <= lo, 0.0, np.where(u >= hi, 1.0, (u - lo) / (hi - lo)))
    out = np.diff(F, axis=1)
    point = (hi <= lo).ravel()
    if point.any():
        b = np.minimum(J - 1, np.floor(hi[point, 0] * J)).astype(int)
        out[point] = 0.0
        out[np.flatnonzero(point), b] = 1.0
    return out


def histograms(P, valid, J):
    """col_hist (D, J), col_n (D,), col_pit_sum (D,) of the entries where `valid` (B, D)."""
    B, D, _ = P.shape
    masses = czado_bins(P[..., 0], P[..., 1], J).reshape(B, D, J) * valid[..., None]
    mid = 0.5 * (np.clip(P[..., 0], 0, 1) + np.clip(P[..., 1], 0, 1))
    return masses.sum(0), valid.sum(0), np.where(valid, mid, 0.0).sum(0)


def summary(col_hist, col_n):
    """(hist, n, ecdf_dev, col_ecdf_dev) as loo_pit returns them."""
    J = col_hist.shape[1]
    edges = np.arange(1, J + 1) / J
    hist, n = col_hist.sum(0), col_n.sum()
    with np.errstate(divide='ignore', invalid='ignore'):
        col_dev = np.abs(np.cumsum(col_hist, 1) / col_n[:, None] - edges).max(1)
    return hist, n, float(np.abs(np.cumsum(hist) / n - edges).max()), col_dev


def loo_pit(x, rate, ll, J, bernoulli=False):
    """The whole check on one batch: x (B, D), rate (S, B, D), ll (B, S) per-row log-likelihoods.  Returns a dict
    with 'P', 'n_invalid', 'lw', 'col_hist', 'col_n', 'col_pit_sum', 'hist', 'n', 'ecdf_dev', 'col_ecdf_dev'."""
    lw, elpd, khat = loo_weights(ll)
    P, n_inv = pit_values(x, rate, lw, bernoulli)
    valid = (n_inv == 0) & np.isfinite(elpd)[:, None]
    col_hist, col_n, col_pit = histograms(P, valid, J)
    hist, n, dev, col_dev = summary(col_hist, col_n)
    return dict(P=P, n_invalid=n_inv, lw=lw, elpd=elpd, khat=khat, valid=valid, col_hist=col_hist, col_n=col_n,
                col_pit_sum=col_pit, hist=hist, n=n, ecdf_dev=dev, col_ecdf_dev=col_dev)
