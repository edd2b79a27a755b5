"""CPU tier of the fit-statistics reference (tests/fit_stats_reference.py): exact rational arithmetic, the
reference's own goodness-of-fit expressions, SciPy, and invariance under exact scaling of the observations."""
import math
from fractions import Fraction

import numpy as np
import pandas as pd
import pytest
import scipy.stats

from tests import fit_stats_reference as ref


def _exact(o, s):
    """NSE, r^2, bias, nRMSD^2 and SSE of the finite pairs in exact rational arithmetic (None where undefined)."""
    keep = ~np.isnan(o) & ~np.isnan(s)
    fo = [Fraction(float(x)) for x in o[keep]]
    fs = [Fraction(float(x)) for x in s[keep]]
    n = len(fo)
    if n == 0:
        return None
    mo, ms = sum(fo) / n, sum(fs) / n
    sso = sum((x - mo) ** 2 for x in fo)
    sss = sum((x - ms) ** 2 for x in fs)
    sxy = sum((x - mo) * (y - ms) for x, y in zip(fo, fs))
    sse = sum((x - y) ** 2 for x, y in zip(fo, fs))
    sabs = sum(abs(x - y) for x, y in zip(fo, fs))
    return {
        ref.ST_SSE: sse,
        ref.ST_NSE: 1 - sse / sso if sso else None,
        ref.ST_R2: sxy ** 2 / (sso * sss) if sso and sss else None,
        ref.ST_PBIAS: 100 * (sum(fs) - sum(fo)) / sum(fo) if sum(fo) else None,
        "nrmsd2": (100 * sabs / n) ** 2 / (sso / n) if sso else None,
    }


def _inputs(seed):
    """Small series with ties, NaN gaps, zeros and negative values among them."""
    rng = np.random.default_rng(seed)
    cases = []
    for n in (0, 1, 2, 3, 5, 17, 40):
        o = np.round(rng.lognormal(0.0, 1.0, n), 1)                    # rounded: ties
        s = np.round(o * rng.lognormal(0.0, 0.3, n), 2)
        if n > 3:
            o[rng.random(n) < 0.2] = np.nan
            s[rng.integers(0, n)] = s[rng.integers(0, n)]              # a tie on the simulated side
        cases.append((o, s))
    o = np.array([0.0, 1.5, 2.5, -0.5, 3.0, np.nan, 4.0])
    cases.append((o, np.array([0.2, 1.4, 2.6, 0.3, 3.1, 9.0, 3.9])))
    return cases


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_reference_equals_exact_rational_arithmetic(seed):
    for o, s in _inputs(seed):
        row, bound = ref.fit_stats(o, s, 0.3)
        ex = _exact(o, s)
        n = int(np.sum(~np.isnan(o) & ~np.isnan(s)))
        assert row[ref.ST_N] == n
        if ex is None:
            assert row[ref.ST_SSE] == 0.0 and row[ref.ST_LOGLIK] == 0.0
            assert all(np.isnan(row[k]) for k in (ref.ST_NSE, ref.ST_LOG_NSE, ref.ST_R2, ref.ST_PBIAS, ref.ST_NRMSD))
            continue
        w = float(ex[ref.ST_SSE])                                # o - s and its square each rounded once, fsum
        assert abs(row[ref.ST_SSE] - w) <= 4 * ref.EPS * w
        for k in (ref.ST_NSE, ref.ST_R2, ref.ST_PBIAS):
            if ex[k] is None:
                assert not np.isfinite(row[k]) or (k == ref.ST_R2 and np.isnan(row[k])), (k, row[k])
            else:
                w = float(ex[k])
                assert abs(row[k] - w) <= 8 * ref.EPS * max(abs(w), 1e-300) + (8 * ref.EPS if k == ref.ST_NSE else 0), (
                    k, row[k], w)
        if ex["nrmsd2"] is not None:
            w = math.sqrt(float(ex["nrmsd2"]))
            assert abs(row[ref.ST_NRMSD] - w) <= 8 * ref.EPS * w
        else:
            assert not np.isfinite(row[ref.ST_NRMSD])
        assert np.all(bound >= 0)


def test_reference_equals_gof_one():
    from simplyp_b200 import stats
    rng = np.random.default_rng(9)
    idx = pd.date_range("2004-01-01", periods=120)
    for _ in range(5):
        o = rng.lognormal(0.0, 0.8, 120)
        o[rng.random(120) < 0.3] = np.nan
        s = o * rng.lognormal(0.1, 0.4, 120)
        s[np.isnan(s)] = rng.lognormal(0.0, 0.8, int(np.isnan(s).sum()))
        want = stats.gof_one(pd.Series(o, idx), pd.Series(s, idx))
        row, _ = ref.fit_stats(o, s, 0.5)
        got = [row[ref.ST_N], row[ref.ST_NSE], row[ref.ST_LOG_NSE], row[ref.ST_SPEARMAN], row[ref.ST_R2],
               row[ref.ST_PBIAS], row[ref.ST_NRMSD]]
        assert got[0] == want[0]
        assert np.allclose(got[1:], want[1:], rtol=1e-12, atol=1e-13), (got, want)


def test_loglik_and_spearman_equal_scipy():
    rng = np.random.default_rng(4)
    for n, m in ((30, 0.2), (200, 0.7), (7, 1.3)):
        o = np.round(rng.lognormal(0.0, 1.0, n), 1)
        s = np.round(o * rng.lognormal(0.0, 0.3, n), 1)
        o[::9] = np.nan
        row, _ = ref.fit_stats(o, s, m)
        k = ~np.isnan(o)
        want = scipy.stats.norm(s[k], m * s[k]).logpdf(o[k]).sum()
        assert abs(row[ref.ST_LOGLIK] - want) <= 1e-12 * abs(want)
        rho = scipy.stats.spearmanr(o[k], s[k]).statistic
        assert abs(row[ref.ST_SPEARMAN] - rho) <= 4 * ref.EPS
    # err_m = 0: the normal density is undefined, the notebook's NaN -> -inf rule applies
    row, _ = ref.fit_stats(np.array([1.0, 2.0]), np.array([1.1, 2.1]), 0.0)
    assert row[ref.ST_LOGLIK] == -np.inf


def test_scaling_the_observations_leaves_r2_and_spearman_unchanged():
    rng = np.random.default_rng(12)
    o = np.round(rng.lognormal(0.0, 1.0, 300), 2)
    o[rng.random(300) < 0.2] = np.nan
    s = o * rng.lognormal(0.0, 0.3, 300)
    s[np.isnan(s)] = 1.0
    row0, _ = ref.fit_stats(o, s, 0.5)
    for k in (-10, 10, 20):
        row, _ = ref.fit_stats(o * 2.0 ** k, s, 0.5)
        assert row[ref.ST_R2] == row0[ref.ST_R2] and row[ref.ST_SPEARMAN] == row0[ref.ST_SPEARMAN], k


def test_bounds_of_the_reference_series_are_tight(golden_dir):
    """On the reference's own Tarland 2004 series the well-conditioned statistics get bounds below 1e-10 relative."""
    import os
    from simplyp_b200 import tarland
    z = np.load(os.path.join(golden_dir, "ref_tarland2004.npz"))
    cols = [str(c) for c in z["dyny_tight_r_cols"]]
    r = z["dyny_tight_r"]
    obs = tarland.load("2004-01-01", "2004-12-31", dynamic="y")[-1][1]
    idx = pd.date_range("2004-01-01", "2004-12-31")
    for var in ref.VAR_KINDS:
        o = obs[var].reindex(idx).to_numpy(float)
        row, bound = ref.fit_stats(o, r[:, cols.index(var + ("_cumecs" if var == "Q" else "_mgl"))], 0.5)
        for k in (ref.ST_LOGLIK, ref.ST_R2, ref.ST_NRMSD, ref.ST_SSE, ref.ST_LOG_NSE):
            assert 0 < bound[k] <= 1e-10 * abs(row[k]), (var, k, bound[k], row[k])


def test_header_and_packing_agree_on_the_columns_the_statistics_read():
    """The kernel reads the error scale of series kind k at SIMPLYP_P_ERR_M0 + k, f_TDP at SIMPLYP_P_F_TDP and the
    catchment area at SIMPLYP_SC_A_CATCH; the ensemble writes those columns by name through packing.MEMBER_INDEX and
    SC_INDEX.  Both layouts must name the same column, and the kinds must be in the same order."""
    import os
    import re
    from simplyp_b200 import packing as pk
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                               "simplyp_b200.h")).read()
    body = header[header.index("SIMPLYP_P_F_QUICK = 0"):header.index("SIMPLYP_NP_MEMBER = ")]
    member = re.findall(r"SIMPLYP_P_([A-Z0-9_]+)", body)
    kinds = re.findall(r"SIMPLYP_V_([A-Z]+)", header[header.index("SIMPLYP_V_Q = 0"):header.index("SIMPLYP_NVARKIND")])
    assert kinds == pk.VAR_KINDS == ref.VAR_KINDS
    for k, var in enumerate(kinds):
        assert member.index("ERR_M%d" % k) == member.index("ERR_M0") + k == pk.MEMBER_INDEX["err_m:" + var] == \
            ref.P_ERR_M[k], var
    assert member.index("F_TDP") == pk.MEMBER_INDEX["f_TDP"] == ref.P_F_TDP
    assert re.search(r"SIMPLYP_SC_A_CATCH = 0\b", header) and pk.SC_INDEX["A_catch"] == ref.SC_A_CATCH == 0
