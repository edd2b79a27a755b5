"""Exact reference of the fused fit statistics (the rows stats[M][V][SIMPLYP_NSTAT] of simplyp_calibrate_*).

The simulated counterparts are rebuilt from the kernel's own full-output run (out[M][S][D][25]) in the reference's
order of operations (model.raw_to_frames, model.py:784-793 of the original), and every slot of
include/simplyp_b200.h:141-151 is formed stably: means first, then centred sums, all summed with math.fsum;
Spearman's r on exact (integer) average ranks.  Degenerate series (n = 0, 1, 2, observations <= 0) get the IEEE
results of the NumPy expressions of stats.gof_one without its n > 10 filter.

Every statistic comes with an error bound for the device, derived from the sums it rests on: the device forms
quotients with sp_div and logs with sp_log (last-bit differences from IEEE), forms the simulated value with up to
four roundings, and sums in its own order, so a sum of n terms t_i, each known to within e_i, is bounded by
C * (n * EPS * sum|t_i| + sum e_i); the bounds of derived statistics follow by first-order propagation.
"""
import math
from fractions import Fraction

import numpy as np

from simplyp_b200 import packing as pk

EPS = float(np.finfo(np.float64).eps)       # 2^-52 (twice the unit roundoff: margin for fma-contracted products)
C = 8.0                                     # safety factor on every first-order bound
SIM_ULPS = 4.0                              # roundings in a simulated value: two quotients, a sum (TP) or product (SRP)
LN_SQRT_2PI = 0.91893853320467274178
NSTAT = 10
ST_N, ST_NSE, ST_LOG_NSE, ST_LOGLIK, ST_R2, ST_PBIAS, ST_NRMSD, ST_SSE, ST_SPEARMAN, ST_RESERVED = range(NSTAT)
VAR_KINDS = pk.VAR_KINDS
# Parameter columns by NAME, as the ensemble writes them (packing.MEMBER_INDEX / SC_INDEX), not by the header's
# SIMPLYP_P_* indices the kernel reads: if the two layouts disagree, the reference reads another column than the
# kernel and the comparison fails.
P_F_TDP = pk.MEMBER_INDEX["f_TDP"]
P_ERR_M = [pk.MEMBER_INDEX["err_m:" + v] for v in VAR_KINDS]
SC_A_CATCH = pk.SC_INDEX["A_catch"]


def simulated(out_ms, A_catch, f_TDP, kind):
    """Simulated counterpart [D] of series kind `kind` from one (member, reach) block out[m][s] [D][25]."""
    Qr = out_ms[:, 5]
    with np.errstate(divide="ignore", invalid="ignore"):
        if kind == 0:
            return Qr * A_catch * 1000 / 86400
        ss, tdp, pp = (out_ms[:, 7] / Qr) / A_catch, (out_ms[:, 9] / Qr) / A_catch, (out_ms[:, 11] / Qr) / A_catch
    return {1: ss, 2: tdp, 3: pp, 4: tdp + pp, 5: tdp * f_TDP}[kind]


def _fsum(x):
    """Correctly rounded sum; with a non-finite term, the IEEE sum (inf - inf is NaN, as in NumPy)."""
    x = np.asarray(x, dtype=np.float64)
    return math.fsum(x.tolist()) if np.all(np.isfinite(x)) else float(np.sum(x))


def _div(a, b):
    with np.errstate(divide="ignore", invalid="ignore"):
        return float(np.float64(a) / np.float64(b))


def average_ranks2(x):
    """Twice the average ranks (ties share the mean rank) as exact integers."""
    x = np.asarray(x, dtype=np.float64)
    order = np.argsort(x, kind="mergesort")
    r2 = np.empty(len(x), dtype=object)
    i, n = 0, len(x)
    while i < n:
        j = i
        while j + 1 < n and x[order[j + 1]] == x[order[i]]:
            j += 1
        for k in order[i:j + 1]:
            r2[k] = i + j + 2                      # 2 * (mean of ranks i+1 .. j+1)
        i = j + 1
    return r2


def spearman_exact(o, s):
    """Spearman's r of paired arrays (no NaN): exact integer sums of centred doubled ranks, one rounding in the end."""
    n = len(o)
    if n < 2:
        return float("nan")
    a = [int(v) - (n + 1) for v in average_ranks2(o)]
    b = [int(v) - (n + 1) for v in average_ranks2(s)]
    sxy = sum(p * q for p, q in zip(a, b))
    sxx = sum(q * q for q in b)
    syy = sum(p * p for p in a)
    if sxx == 0 or syy == 0:
        return float("nan")
    return sxy / math.sqrt(sxx * syy)              # sxx * syy is an exact integer


def spearman_tie_bound(o, s, ulps=4):
    """What near-ties of the simulated values (|s_i - s_j| <= ulps ulp) could move Spearman's r by: the device may
    order such a pair either way.  Sum over those pairs of |rank_obs,i - rank_obs,j| / sqrt(Sxx Syy), in rank units."""
    n = len(o)
    if n < 2:
        return 0.0
    ro = [Fraction(int(v), 2) for v in average_ranks2(o)]
    rs = [Fraction(int(v), 2) for v in average_ranks2(s)]
    mean = Fraction(n + 1, 2)
    sxx = sum((r - mean) ** 2 for r in rs)
    syy = sum((r - mean) ** 2 for r in ro)
    if sxx == 0 or syy == 0:
        return 0.0
    order = np.argsort(s, kind="mergesort")
    tot = Fraction(0)
    for p in range(n):
        i = order[p]
        q = p + 1
        while q < n and s[order[q]] - s[i] <= ulps * np.spacing(abs(s[i])):
            if s[order[q]] != s[i]:
                tot += abs(ro[i] - ro[order[q]])
            q += 1
    return float(tot) / math.sqrt(float(sxx) * float(syy))


def fit_stats(o, s, err_m):
    """Every slot of one statistics row for observations `o` [D] (NaN = none) and simulated values `s` [D], error
    scale `err_m`.  Returns (row [NSTAT], bound [NSTAT]); bound[k] is the device's allowed |error| in slot k (0: exact;
    NaN slots compare as NaN)."""
    o = np.asarray(o, dtype=np.float64)
    s = np.asarray(s, dtype=np.float64)
    keep = ~np.isnan(o) & ~np.isnan(s)                # pandas dropna(how='any')
    o, s = o[keep], s[keep]
    n = len(o)
    row = np.full(NSTAT, np.nan)
    bound = np.zeros(NSTAT)
    row[ST_N] = n
    row[ST_RESERVED] = 0.0
    row[ST_SPEARMAN] = spearman_exact(o, s)
    bound[ST_SPEARMAN] = spearman_tie_bound(o, s) + 4 * EPS * (abs(row[ST_SPEARMAN]) if n >= 2 else 0.0)
    with np.errstate(all="ignore"):
        lo, ls = np.log(o), np.where(s > 0, np.log(np.where(s > 0, s, 1.0)), np.nan)
        sg = err_m * s
        d = o - s
        # log-likelihood, MCMC.ipynb:233-240 (a NaN sum is -inf)
        z = d / sg
        lsg = np.where(sg > 0, np.log(np.where(sg > 0, sg, 1.0)), np.nan)
        t_ll = -LN_SQRT_2PI - lsg - 0.5 * z * z
    ll = _fsum(t_ll) if n else 0.0
    row[ST_LOGLIK] = -math.inf if math.isnan(ll) else ll
    if np.all(np.isfinite(t_ll)) and n:
        e_ll = 2 * EPS * (SIM_ULPS + np.abs(lsg)) + np.abs(z) * EPS * (6 * np.abs(z) + SIM_ULPS / abs(err_m))
        bound[ST_LOGLIK] = C * (n * EPS * _fsum(np.abs(t_ll)) + _fsum(e_ll))
    # SSE and NSE
    t_sse = d * d
    sse = _fsum(t_sse)
    e_d = EPS * np.abs(d) + SIM_ULPS * EPS * np.abs(s)          # |error| of o - s on the device
    b_sse = C * (n * EPS * sse + _fsum(2 * np.abs(d) * e_d))
    row[ST_SSE] = sse
    bound[ST_SSE] = b_sse
    mo = _div(_fsum(o), n)
    co = o - mo
    ss_o = _fsum(co * co)
    b_sso = C * n * EPS * ss_o
    row[ST_NSE] = 1.0 - _div(sse, ss_o)
    if ss_o > 0:
        bound[ST_NSE] = b_sse / ss_o + sse * b_sso / ss_o ** 2 + EPS
    # log NSE
    with np.errstate(all="ignore"):
        dl = lo - ls
        t_sl = dl * dl
        if np.all(np.isfinite(lo)) and n:
            mlo = _fsum(lo) / n
            cl = lo - mlo
            ss_lo = _fsum(cl * cl)
        else:                                                    # log of 0 / negative: NumPy's IEEE result
            ss_lo = float(np.sum((lo - np.mean(lo)) ** 2)) if n else 0.0
    ssel = _fsum(t_sl)
    row[ST_LOG_NSE] = 1.0 - _div(ssel, ss_lo)
    if np.isfinite(row[ST_LOG_NSE]) and ss_lo > 0:
        e_dl = 2 * EPS * (np.abs(lo) + np.abs(ls)) + 2 * SIM_ULPS * EPS
        b_ssel = C * (n * EPS * ssel + _fsum(2 * np.abs(dl) * e_dl))
        b_sslo = C * (n * EPS * ss_lo + _fsum(2 * np.abs(cl) * EPS * np.abs(lo)))
        bound[ST_LOG_NSE] = b_ssel / ss_lo + ssel * b_sslo / ss_lo ** 2 + EPS
    # bias, nRMSD
    sum_o = _fsum(o)
    diff = _fsum(np.concatenate([s, -o]))
    row[ST_PBIAS] = _div(100.0 * diff, sum_o)
    if n and sum_o != 0:
        b_diff = C * (n * EPS * (_fsum(np.abs(s)) + _fsum(np.abs(o))))
        bound[ST_PBIAS] = 100.0 * b_diff / abs(sum_o) + 4 * EPS * abs(row[ST_PBIAS])
    sabs = _fsum(np.abs(d))
    std_o = math.sqrt(ss_o / n) if n else float("nan")
    row[ST_NRMSD] = _div(100.0 * _div(sabs, n), std_o) if n else float("nan")
    if n and std_o > 0:
        b_sabs = C * (n * EPS * sabs + _fsum(e_d))
        bound[ST_NRMSD] = abs(row[ST_NRMSD]) * (b_sabs / sabs if sabs else 0.0) + abs(row[ST_NRMSD]) * (
            b_sso / ss_o / 2 + 4 * EPS)
    # r^2: two-pass, centred on the means
    ms = _div(_fsum(s), n)
    cs = s - ms
    sxx = _fsum(cs * cs)
    sxy = _fsum(co * cs)
    with np.errstate(all="ignore"):
        row[ST_R2] = float(np.float64(sxy) * sxy / (np.float64(sxx) * ss_o)) if n else float("nan")
    if n >= 2 and sxx > 0 and ss_o > 0 and sxy != 0:
        # the device sums about c = the simulated value of the first observed day, then S2 - S1^2 / n: the cancellation
        # costs sum (s - c)^2 / Sxx; the per-element error of s - c is that of s, plus its rounding
        c = s[0]
        u = s - c
        e_u = SIM_ULPS * EPS * np.abs(s) + EPS * np.abs(u)
        s1, s2 = _fsum(u), _fsum(u * u)
        b_s1 = n * EPS * _fsum(np.abs(u)) + _fsum(e_u)
        b_sxx = C * (n * EPS * s2 + _fsum(2 * np.abs(u) * e_u) + 2 * abs(s1) * b_s1 / n + EPS * s1 * s1 / n + EPS * s2)
        b_sxy = C * (n * EPS * _fsum(np.abs(co * u)) + _fsum(np.abs(co) * e_u) + EPS * _fsum(np.abs(o)) * abs(s1)
                     + EPS * _fsum(np.abs(o) * np.abs(u)))
        bound[ST_R2] = abs(row[ST_R2]) * (2 * b_sxy / abs(sxy) + b_sxx / sxx + b_sso / ss_o + 4 * EPS)
    return row, bound


def reference_stats(out, member_params, sc_params, obs, obs_desc):
    """Reference rows [M][V][NSTAT] and bounds for the full-output run `out` [M][S][D][25] of the same members,
    sc params [1 or M][S][16], observations [V][D] and obs_desc [V][2] as the calibration run."""
    out = np.asarray(out)
    M, V = out.shape[0], obs.shape[0]
    sc_params = np.asarray(sc_params)
    if sc_params.ndim == 2:
        sc_params = sc_params[None]
    rows = np.zeros((M, V, NSTAT))
    bounds = np.zeros((M, V, NSTAT))
    for m in range(M):
        scp = sc_params[m if sc_params.shape[0] > 1 else 0]
        for v in range(V):
            reach, kind = int(obs_desc[v, 0]), int(obs_desc[v, 1])
            sim = simulated(out[m, reach], scp[reach, SC_A_CATCH], member_params[m, P_F_TDP], kind)
            rows[m, v], bounds[m, v] = fit_stats(obs[v], sim, member_params[m, P_ERR_M[kind]])
    return rows, bounds


def compare(got, want, bound, slots=range(NSTAT)):
    """Indices (m, v, slot) where got and want differ by more than the bound (NaN equals NaN, inf equals inf)."""
    bad = []
    for k in slots:
        g, w, b = got[..., k], want[..., k], bound[..., k]
        with np.errstate(invalid="ignore"):
            same = (g == w) | (np.isnan(g) & np.isnan(w)) | (np.abs(g - w) <= b)
        for idx in zip(*np.nonzero(~same)):
            bad.append(tuple(int(i) for i in idx) + (k,))
    return bad
