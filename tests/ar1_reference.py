"""Reference of the AR(1) error model of the log-likelihood (simplyp_calibrate_ar1_device, csrc/simplyp_ar1.cuh).

For a series with observed days t_1 < ... < t_n, sigma_i = m s_i and Sigma_ij = sigma_i sigma_j phi^|t_i - t_j|,
the log-likelihood is log N(o; s, Sigma).  `loglik_sequential` is its Markov factorisation, the form the kernel sums
(eta_i = (o_i - s_i) / sigma_i, rho_i = phi^(t_i - t_{i-1})), summed with math.fsum; `loglik_dense` evaluates the
dense density with scipy.stats.multivariate_normal.  Conventions of the kernel: |phi| >= 1 (or NaN), s <= 0,
sigma <= 0 or a non-finite sum give -inf; no observed day gives 0.
"""
import math

import numpy as np

LN_SQRT_2PI = 0.91893853320467274178


def loglik_sequential(o, s, m, phi):
    """The AR(1) log-likelihood of observations o [D] (NaN: not observed) given simulated values s [D]."""
    o = np.asarray(o, dtype=np.float64)
    s = np.asarray(s, dtype=np.float64)
    phi = float(phi)
    if not abs(phi) < 1.0:
        return -math.inf
    days = np.flatnonzero(~np.isnan(o))
    if days.size == 0:
        return 0.0
    oo, ss = o[days], s[days]
    sg = m * ss
    if not (np.all(ss > 0) and np.all(sg > 0)):
        return -math.inf
    eta = (oo - ss) / sg
    rho = np.zeros(days.size)
    rho[1:] = np.array([phi ** int(g) for g in np.diff(days)])
    eta_prev = np.concatenate([[0.0], eta[:-1]])
    q = (1.0 - rho) * (1.0 + rho)
    with np.errstate(all="ignore"):
        terms = -LN_SQRT_2PI - np.log(sg) - 0.5 * np.log(q) - (eta - rho * eta_prev) ** 2 / (2.0 * q)
    if not np.all(np.isfinite(terms)):
        return -math.inf
    total = math.fsum(terms.tolist())
    return total if math.isfinite(total) else -math.inf


def covariance(days, sigma, phi):
    """Sigma_ij = sigma_i sigma_j phi^|t_i - t_j| of observed days `days` [n]."""
    lag = np.abs(np.subtract.outer(days, days))
    corr = np.array([[float(phi) ** int(k) for k in row] for row in lag]) if lag.size else np.zeros((0, 0))
    return np.outer(sigma, sigma) * corr


def loglik_dense(o, s, m, phi):
    """log N(o; s, Sigma) on the observed days by scipy.stats.multivariate_normal (for |phi| < 1, s > 0, m > 0)."""
    from scipy.stats import multivariate_normal

    o = np.asarray(o, dtype=np.float64)
    s = np.asarray(s, dtype=np.float64)
    days = np.flatnonzero(~np.isnan(o))
    if days.size == 0:
        return 0.0
    cov = covariance(days, m * s[days], phi)
    return float(multivariate_normal(mean=s[days], cov=cov).logpdf(o[days]))
