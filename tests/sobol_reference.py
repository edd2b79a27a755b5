"""NumPy / fsum restatement of the Sobol' sensitivity analysis (csrc/simplyp_sobol.cuh, simplyp_sobol_*_device).

- ``direction_numbers``: the 32-bit Joe-Kuo direction numbers rebuilt from SciPy's table
  (``scipy/stats/_sobol_direction_numbers.npz``, new-joe-kuo-6.21201).
- ``sobol_points``: unscrambled Sobol' points as 32-bit integers, point n = XOR of V[d][j] over the set bits j of
  gray(n) = n ^ (n >> 1).
- ``design_values``: the Saltelli design in SALib's row order, parameter value lo + (hi - lo) u, each operation
  rounded on its own.
- ``indices``: SALib's ``sobol.analyze`` estimators (Saltelli 2010 first order, Jansen total, Saltelli 2002 second
  order) with every sum taken by ``math.fsum``; ``bootstrap_conf`` the same estimators on given resamples.
"""
import math
import os

import numpy as np


def _npz():
    import scipy.stats
    return np.load(os.path.join(os.path.dirname(scipy.stats.__file__), "_sobol_direction_numbers.npz"))


def direction_numbers(D):
    """V [D][32] uint32: V[d][j] is the direction number of bit j (the most significant bit first)."""
    z = _npz()
    poly, vinit = z["poly"], z["vinit"]
    V = np.zeros((D, 32), dtype=np.uint64)
    V[0] = [1 << (31 - j) for j in range(32)]
    for d in range(1, D):
        p = int(poly[d])
        m = p.bit_length() - 1
        for j in range(m):
            V[d, j] = int(vinit[d, j]) << (31 - j)
        for j in range(m, 32):
            v = int(V[d, j - m])
            v ^= v >> m
            for k in range(1, m):
                if (p >> (m - k)) & 1:
                    v ^= int(V[d, j - k])
            V[d, j] = v
    return V.astype(np.uint32)


def sobol_points(D, n, skip=0):
    """Points skip .. skip + n - 1 of the D-dimensional sequence as uint32 [n][D]."""
    V = direction_numbers(D).astype(np.uint64)
    idx = np.arange(skip, skip + n, dtype=np.uint64)
    g = idx ^ (idx >> np.uint64(1))
    x = np.zeros((n, D), dtype=np.uint64)
    for j in range(32):
        bit = ((g >> np.uint64(j)) & np.uint64(1)).astype(bool)
        x[bit] ^= V[:, j][None, :]
    return x.astype(np.uint32)


def design_slots(K, second_order):
    """P and, per slot, the source (0: A, 1: B) of every column [P][K]."""
    P = 2 * K + 2 if second_order else K + 2
    src = np.zeros((P, K), dtype=np.int64)
    for j in range(K):
        src[1 + j, j] = 1
        if second_order:
            src[K + 1 + j] = 1
            src[K + 1 + j, j] = 0
    src[P - 1] = 1
    return P, src


def design_values(bounds, n_base, skip=0, second_order=False):
    """Parameter values [n_base * P][K] of the Saltelli design, member m = i P + slot."""
    bounds = np.asarray(bounds, dtype=np.float64)
    K = bounds.shape[0]
    P, src = design_slots(K, second_order)
    x = sobol_points(2 * K, n_base, skip)
    u = x.astype(np.float64) * 2.0 ** -32
    lo, hi = bounds[:, 0], bounds[:, 1]
    vals = lo[None, :] + (hi - lo)[None, :] * u[:, :K]          # A; numpy never fuses, each op rounded
    valsB = lo[None, :] + (hi - lo)[None, :] * u[:, K:]
    out = np.where(src[None, :, :] == 1, valsB[:, None, :], vals[:, None, :])
    return out.reshape(n_base * P, K)


def _row_terms(y, K, second_order):
    P = 2 * K + 2 if second_order else K + 2
    Yr = np.asarray(y, dtype=np.float64).reshape(-1, P)
    used = np.all(np.isfinite(Yr), axis=1)
    return Yr, used


def indices(y, K, second_order=False):
    """Point estimates of one row y [N P]: dict S1, ST [K], S2 [K][K] (NaN outside j < k), c, V, n."""
    Yr, used = _row_terms(y, K, second_order)
    U = Yr[used]
    n = U.shape[0]
    nan = dict(S1=np.full(K, np.nan), ST=np.full(K, np.nan), S2=np.full((K, K), np.nan), c=np.nan, V=np.nan, n=n)
    if n < 2:
        return nan
    c = math.fsum(U.ravel()) / U.size
    Uc = U - c
    a, b = Uc[:, 0], Uc[:, -1]
    ab = Uc[:, 1:K + 1]
    ab_ = np.concatenate([a, b])
    mu = math.fsum(ab_) / (2 * n)
    V = math.fsum((ab_ - mu) ** 2) / (2 * n)
    res = dict(S1=np.full(K, np.nan), ST=np.full(K, np.nan), S2=np.full((K, K), np.nan), c=c, V=V, n=n)
    if V == 0:
        return res
    for j in range(K):
        res["S1"][j] = math.fsum(b * (ab[:, j] - a)) / n / V
        res["ST"][j] = 0.5 * (math.fsum((a - ab[:, j]) ** 2) / n) / V
    if second_order:
        ba = Uc[:, K + 1:2 * K + 1]
        for j in range(K):
            for k in range(j + 1, K):
                res["S2"][j, k] = math.fsum(ba[:, j] * ab[:, k] - a * b) / n / V - res["S1"][j] - res["S1"][k]
    return res


def bootstrap_conf(y, K, picks, z, second_order=False):
    """conf = z std (ddof 1) over the resamples picks [n_boot][n] (positions 0..n-1 in the used samples) of S1, ST
    and S2, with c fixed at the full-data value and V recomputed per resample."""
    Yr, used = _row_terms(y, K, second_order)
    U = Yr[used]
    n = U.shape[0]
    c = math.fsum(U.ravel()) / U.size
    Uc = U - c
    nb = picks.shape[0]
    s1 = np.empty((nb, K))
    st = np.empty((nb, K))
    s2 = np.full((nb, K, K), np.nan)
    for t in range(nb):
        X = Uc[picks[t]]
        a, b, ab = X[:, 0], X[:, -1], X[:, 1:K + 1]
        ab_ = np.concatenate([a, b])
        mu = math.fsum(ab_) / (2 * n)
        V = math.fsum((ab_ - mu) ** 2) / (2 * n)
        for j in range(K):
            s1[t, j] = math.fsum(b * (ab[:, j] - a)) / n / V
            st[t, j] = 0.5 * (math.fsum((a - ab[:, j]) ** 2) / n) / V
        if second_order:
            ba = X[:, K + 1:2 * K + 1]
            for j in range(K):
                for k in range(j + 1, K):
                    s2[t, j, k] = math.fsum(ba[:, j] * ab[:, k] - a * b) / n / V - s1[t, j] - s1[t, k]
    return (z * np.std(s1, axis=0, ddof=1), z * np.std(st, axis=0, ddof=1), z * np.std(s2, axis=0, ddof=1))


def philox_picks(words, n):
    """Positions (w n) >> 32 of the bootstrap's words [n_boot][n] (uint32)."""
    return ((words.astype(np.uint64) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


# ---- analytic test functions
def ishigami(x, a=7.0, b=0.1):
    """x [.., 3] in [-pi, pi]^3."""
    return np.sin(x[..., 0]) + a * np.sin(x[..., 1]) ** 2 + b * x[..., 2] ** 4 * np.sin(x[..., 0])


def ishigami_indices(a=7.0, b=0.1):
    V1 = 0.5 * (1 + b * np.pi ** 4 / 5) ** 2
    V2 = a ** 2 / 8
    V13 = b ** 2 * np.pi ** 8 / 18 - b ** 2 * np.pi ** 8 / 50
    V = V1 + V2 + V13
    return np.array([V1, V2, 0.0]) / V, np.array([V1 + V13, V2, V13]) / V


def g_function(x, a):
    """Sobol's G function on x [.., K] in [0, 1]^K."""
    return np.prod((np.abs(4 * x - 2) + a) / (1 + a), axis=-1)


def g_indices(a):
    """First-order and second-order (j < k) indices of the G function."""
    a = np.asarray(a, dtype=np.float64)
    vi = 1.0 / (3.0 * (1 + a) ** 2)
    V = np.prod(1 + vi) - 1
    S2 = np.full((a.size, a.size), np.nan)
    for j in range(a.size):
        for k in range(j + 1, a.size):
            S2[j, k] = vi[j] * vi[k] / V
    return vi / V, S2
