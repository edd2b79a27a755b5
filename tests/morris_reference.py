"""NumPy / fsum restatement of the Morris screening (csrc/simplyp_morris.cuh, simplyp_morris_*_device).

- ``levels``: the candidate trajectories in integer levels [n][K + 1][K], drawn from NumPy's Philox4x32-10 with the
  word order of the header (base levels, directions, Fisher-Yates order).
- ``design_values``: min(lo + (hi - lo) (level / (p - 1)), hi), each operation rounded on its own.
- ``distances`` / ``select``: the trajectory distance by brute force (math.sqrt of the integer squared distances,
  i-major running sum), and the greedy spread search.
- ``effects`` / ``bootstrap_conf``: SALib's ``morris.analyze`` estimators, every sum taken by ``math.fsum``.
"""
import math

import numpy as np

from tests import mcmc_reference as mref

BLOCK = 6


def _words(seed, c, n_words, kind):
    """Words [len(c)][n_words] of candidates (or resamples) c: word k from counter (c, k / 4, kind, 6)."""
    c = np.asarray(c, dtype=np.uint64)
    nq = (n_words + 3) // 4
    q = np.arange(nq, dtype=np.uint64)
    ctr = np.stack([np.repeat(c, nq), np.tile(q, c.size), np.full(c.size * nq, kind, dtype=np.uint64),
                    np.full(c.size * nq, BLOCK, dtype=np.uint64)], axis=1)
    w = mref.philox4x32_10(ctr, [seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF])
    return w.reshape(c.size, nq * 4)[:, :n_words]


def pick(w, n):
    return ((np.asarray(w, dtype=np.uint64) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


def levels(seed, K, p, n, c0=0):
    """Levels [n][K + 1][K] of candidates c0 .. c0 + n - 1."""
    h = p // 2
    w = _words(seed, np.arange(c0, c0 + n), 3 * K - 1, 0)
    base = pick(w[:, :K], h)
    neg = pick(w[:, K:2 * K], 2)
    out = np.zeros((n, K + 1, K), dtype=np.int64)
    for c in range(n):
        order = list(range(K))
        for i in range(K - 1, 0, -1):
            j = int(pick(w[c, 2 * K + (K - 1 - i)], i + 1))
            order[i], order[j] = order[j], order[i]
        x = base[c] + h * neg[c]
        out[c, 0] = x
        for s in range(1, K + 1):
            z = order[s - 1]
            x = x.copy()
            x[z] += -h if neg[c, z] else h
            out[c, s] = x
    return out


def design_values(bounds, lev, p):
    """Parameter values [r (K + 1)][K] of trajectories lev [r][K + 1][K]."""
    bounds = np.asarray(bounds, dtype=np.float64)
    lo, hi = bounds[:, 0], bounds[:, 1]
    u = lev.reshape(-1, lev.shape[-1]).astype(np.float64) / float(p - 1)
    v = lo[None, :] + (hi - lo)[None, :] * u                 # numpy never fuses: each operation rounded
    return np.minimum(v, hi[None, :])


def distance(a, b):
    """d(a, b) of two trajectories [K + 1][K] (a the lower candidate index), brute force."""
    total = 0.0
    for i in range(a.shape[0]):
        for j in range(b.shape[0]):
            total += math.sqrt(int(np.sum((a[i] - b[j]) ** 2)))
    return total


def distances(lev):
    """Symmetric matrix [n][n] of d over all candidate pairs (0 on the diagonal), vectorised over the pairs."""
    n, P, _ = lev.shape
    D = np.zeros((n, n))
    for m in range(n - 1):
        a, b = lev[m], lev[m + 1:]
        sq = ((a[None, :, None, :] - b[:, None, :, :]) ** 2).sum(axis=-1)      # [pairs][i][j], exact integers
        s = np.sqrt(sq.astype(np.float64))
        tot = np.zeros(n - 1 - m)
        for i in range(P):
            for j in range(P):
                tot = tot + s[:, i, j]
        D[m, m + 1:] = tot
        D[m + 1:, m] = tot
    return D


def select(lev, r):
    """The greedy spread search: the pair of largest d (lowest (m, l) on ties), then the candidate maximising the sum,
    in selection order, of d(c, s)^2 (lowest c on ties)."""
    n = lev.shape[0]
    D = distances(lev)
    upper = np.where(np.triu(np.ones((n, n), bool), 1), D, -1.0)
    k = int(np.argmax(upper))
    sel = [k // n, k % n]
    score = np.zeros(n)
    for step in range(r - 1):
        score = score + D[:, sel[step]] * D[:, sel[step]]
        if step == 0:
            continue
        masked = score.copy()
        masked[sel] = -np.inf
        sel.append(int(np.argmax(masked)))
    return np.array(sel[:r], dtype=np.int64), D


def spread(D, sel):
    """Campolongo's spread of a set of trajectories: sqrt of the sum over its pairs of d^2."""
    sel = list(sel)
    return math.sqrt(math.fsum(D[a, b] ** 2 for k, a in enumerate(sel) for b in sel[k + 1:]))


def _steps(lev):
    """For trajectories lev [r][K + 1][K]: the parameter moved by each step [r][K] and whether it moved up."""
    d = np.diff(lev, axis=1)
    j = np.argmax(d != 0, axis=2)
    up = np.take_along_axis(d, j[..., None], axis=2)[..., 0] > 0
    return j, up


def elementary_effects_matrix(y, lev, p):
    """EE [r][K] of one output row y [r (K + 1)] and which trajectories are used (all K + 1 values finite)."""
    r, P, K = lev.shape
    Y = np.asarray(y, dtype=np.float64).reshape(r, P)
    used = np.all(np.isfinite(Y), axis=1)
    delta = p / (2.0 * (p - 1))
    j, up = _steps(lev)
    ee = np.full((r, K), np.nan)
    for i in range(r):
        if not used[i]:
            continue
        for s in range(K):
            lo, hi = (Y[i, s], Y[i, s + 1]) if up[i, s] else (Y[i, s + 1], Y[i, s])
            ee[i, j[i, s]] = (hi - lo) / delta
    return ee, used


def effects(y, lev, p):
    """mu, mu_star, sigma [K] and n of one output row y [r (K + 1)] (NaN with n < 2)."""
    ee, used = elementary_effects_matrix(y, lev, p)
    E = ee[used]
    n, K = E.shape[0], lev.shape[2]
    if n < 2:
        return dict(mu=np.full(K, np.nan), mu_star=np.full(K, np.nan), sigma=np.full(K, np.nan), n=n)
    mu = np.array([math.fsum(E[:, k]) / n for k in range(K)])
    mu_star = np.array([math.fsum(np.abs(E[:, k])) / n for k in range(K)])
    sigma = np.array([math.sqrt(math.fsum((E[:, k] - mu[k]) ** 2) / (n - 1)) for k in range(K)])
    return dict(mu=mu, mu_star=mu_star, sigma=sigma, n=n)


def bootstrap_conf(y, lev, p, picks, z):
    """z std (ddof 1) of mu_star over the resamples picks [n_boot][n] (positions 0..n-1 in the used trajectories)."""
    ee, used = elementary_effects_matrix(y, lev, p)
    E = np.abs(ee[used])
    n = E.shape[0]
    ms = np.array([[math.fsum(E[picks[b], k]) / n for k in range(E.shape[1])] for b in range(picks.shape[0])])
    return z * np.std(ms, axis=0, ddof=1)
