"""CPU tier of the period aggregates: the host build of simplyp_periods.cuh (tests/periods_host.cpp) against a NumPy
sequential-loop restatement bitwise and against math.fsum, its daily water-body columns against
model.sum_to_waterbody, the period bounds, PeriodStatistics.exceedance / table, and the input checks of
ensemble.period_statistics."""
import ctypes as C
import math

import numpy as np
import pandas as pd
import pytest

from tests import fit_stats_reference as ref

QR, MSUS, TDP, PP = 5, 7, 9, 11
CONV = 1000.0 / 86400.0


@pytest.fixture(scope="module")
def host():
    from tests import periods_host
    periods_host.load()
    return periods_host


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def _synthetic(M=5, S=3, D=70, seed=1):
    """Full output with positive flows and fluxes, zero-flow and NaN days, per-member A_catch and f_TDP, and one
    failed member."""
    from simplyp_b200 import packing as pk
    rng = np.random.default_rng(seed)
    out = rng.uniform(0.0, 1.0, size=(M, S, D, pk.NOUT))
    out[:, :, :, QR] = rng.lognormal(-3.0, 1.5, size=(M, S, D))
    for c in (MSUS, TDP, PP):
        out[:, :, :, c] = rng.lognormal(0.0, 2.0, size=(M, S, D))
    out[0, 1, 10, QR] = 0.0                        # a zero-flow day of one reach
    out[0, :, 20, QR] = 0.0                        # and of every reach: the water body has Q = 0 that day
    out[0, :, 20, TDP] = 0.0
    out[-1, 0, 33, TDP] = np.nan                   # a NaN flux
    member = np.zeros((M, pk.NP_MEMBER))
    member[:, ref.P_F_TDP] = rng.uniform(0.2, 0.8, size=M)
    sc = np.zeros((M, S, pk.NP_SC))
    sc[:, :, ref.SC_A_CATCH] = rng.uniform(5.0, 60.0, size=(M, S))
    diag = np.zeros((M, S, pk.NDIAG), dtype=np.int64)
    diag[min(3, M - 1), -1, 3] = 1                 # member 3 failed at its last reach
    return out, member, sc, diag


def _daily(out_m, sc_m, f, target, kind, stat, wb):
    """NumPy restatement of period_day over all days: (x [D], q [D])."""
    D = out_m.shape[1]
    with np.errstate(divide="ignore", invalid="ignore"):
        if stat == 0 and target >= 0:
            return ref.simulated(out_m[target], sc_m[target, ref.SC_A_CATCH], f, kind), np.zeros(D)
        q, ms, td, pp = np.zeros(D), np.zeros(D), np.zeros(D), np.zeros(D)
        for s in (wb if target < 0 else [target]):
            q = q + out_m[s, :, QR] * sc_m[s, ref.SC_A_CATCH] * 1000.0 / 86400.0
            ms, td, pp = ms + out_m[s, :, MSUS], td + out_m[s, :, TDP], pp + out_m[s, :, PP]
        conc = {k: (fl / q) * CONV for k, fl in ((1, ms), (2, td), (3, pp))}
        if stat == 0:
            x = {0: q, 1: conc[1], 2: conc[2], 3: conc[3], 4: conc[2] + conc[3], 5: conc[2] * f}[kind]
        else:
            x = {0: q * 86400.0, 1: ms, 2: td, 3: pp, 4: td + pp, 5: td * f}[kind]
    return x, (q if stat == 2 else np.zeros(D))


def _seqsum(x):
    s = np.float64(0.0)
    for v in x:
        s = s + v
    return s


def restate(out, member, sc, diag, desc, bounds, wb):
    """The period aggregates as a sequential loop over the days in NumPy: values [V P][M]."""
    M = out.shape[0]
    sc = sc if sc.ndim == 3 else sc[None]
    values = np.full((len(desc) * len(bounds), M), np.nan)
    for m in range(M):
        if np.any(diag[m, :, 3] != 0):
            continue
        sc_m = sc[m if sc.shape[0] > 1 else 0]
        for v, (target, kind, stat) in enumerate(desc):
            x, q = _daily(out[m], sc_m, member[m, ref.P_F_TDP], target, kind, stat, wb)
            for p, (a, b) in enumerate(bounds):
                sx, sq = _seqsum(x[a:b + 1]), _seqsum(q[a:b + 1])
                with np.errstate(divide="ignore", invalid="ignore"):
                    values[v * len(bounds) + p, m] = {0: sx / np.float64(b - a + 1), 1: sx, 2: (sx / sq) * CONV}[stat]
    return values


def _all_series(S):
    return [(t, k, st) for t in list(range(S)) + [-1] for k in range(6) for st in range(3) if not (st == 2 and k == 0)]


@pytest.mark.parametrize("per_member_sc", [True, False])
def test_host_aggregates_equal_numpy_restatement_bitwise(host, per_member_sc):
    out, member, sc, diag = _synthetic()
    if not per_member_sc:
        sc = sc[:1]
    desc = _all_series(out.shape[1])
    bounds = np.array([(0, 69), (0, 30), (31, 59), (60, 69), (25, 45), (7, 7), (69, 69)], dtype=np.int32)
    wb = [2, 0]
    got = host.aggregate(out, member, sc, diag, desc, bounds, wb)
    want = restate(out, member, sc, diag, np.asarray(desc), bounds, wb)
    assert _same(got, want)
    assert np.all(np.isnan(got[:, 3]))                                        # the failed member
    assert np.isfinite(np.delete(got, 3, axis=1)).mean() > 0.8                # NaN only where a day is NaN or Q = 0


def test_host_sums_are_within_rounding_of_fsum(host):
    out, member, sc, diag = _synthetic(seed=4)
    diag[:] = 0
    out[np.isnan(out)] = 1.0
    out[:, :, :, QR] = np.maximum(out[:, :, :, QR], 1e-3)
    desc = [(t, k, 1) for t in (0, -1) for k in range(6)] + [(1, k, 0) for k in range(6)]
    bounds = np.array([(0, 69), (3, 40)], dtype=np.int32)
    got = host.aggregate(out, member, sc, diag, desc, bounds, [0, 1, 2])
    for v, (t, k, st) in enumerate(desc):
        for m in range(out.shape[0]):
            x, _ = _daily(out[m], sc[m], member[m, ref.P_F_TDP], t, k, st, [0, 1, 2])
            for p, (a, b) in enumerate(bounds):
                seg = x[a:b + 1]
                exact = math.fsum(seg.tolist()) / (b - a + 1 if st == 0 else 1)
                n = b - a + 1
                assert abs(got[v * 2 + p, m] - exact) <= n * ref.EPS * np.abs(seg).sum() / (n if st == 0 else 1) \
                    + ref.EPS * abs(exact)


def test_host_waterbody_columns_equal_model_sum_to_waterbody(host, capsys):
    from simplyp_b200 import model as spm
    out, member, sc, diag = _synthetic(M=1, S=4, D=50, seed=7)
    out[0, :, :, QR] = np.maximum(out[0, :, :, QR], 1e-3)
    out[np.isnan(out)] = 0.5
    ids = [11, 12, 13, 14]
    idx = pd.date_range("2001-01-01", periods=50)
    f = float(member[0, ref.P_F_TDP])
    frames = {}
    for s, sc_id in enumerate(ids):
        _, df_R = spm.raw_to_frames(out[0, s], idx, float(sc[0, s, ref.SC_A_CATCH]), 1.0, f, "None")
        frames[sc_id] = df_R
    p_struc = pd.DataFrame({"Upstream_SCs": [np.nan] * 4, "In_final_flux?": [1.0, np.nan, 1.0, 1.0]},
                           index=pd.Index(ids, name="Reach"))
    want = spm.sum_to_waterbody(p_struc, 4, frames, f)
    got = host.waterbody(out, sc, member, [0, 2, 3])[0]
    from simplyp_b200.engine import Engine
    for j, col in enumerate(Engine.WATERBODY_COLUMNS):
        w = want[col].to_numpy()
        assert np.all(np.abs(got[:, j] - w) <= 1e-12 * np.abs(w)), col


# --------------------------------------------------------------------------- period bounds
def test_year_bounds_keep_partial_years_and_leap_days():
    from simplyp_b200 import ensemble as ens
    idx = pd.date_range("2003-07-01", "2005-02-10")
    b, names = ens.period_bounds(idx, "year")
    assert names == ["2003", "2004", "2005"]
    assert b.tolist() == [[0, 183], [184, 184 + 365], [550, len(idx) - 1]]
    assert (b[:, 1] - b[:, 0] + 1).tolist() == [184, 366, 41]


def test_month_and_all_bounds():
    from simplyp_b200 import ensemble as ens
    idx = pd.date_range("2004-01-15", "2004-03-31")
    b, names = ens.period_bounds(idx, "month")
    assert names == ["2004-01", "2004-02", "2004-03"]
    assert (b[:, 1] - b[:, 0] + 1).tolist() == [17, 29, 31]
    assert b[0, 0] == 0 and b[-1, 1] == len(idx) - 1 and np.all(b[1:, 0] == b[:-1, 1] + 1)
    b, names = ens.period_bounds(idx, "all")
    assert b.tolist() == [[0, len(idx) - 1]] and names == ["2004-01-15/2004-03-31"]


def test_one_day_record_and_overlapping_ranges():
    from simplyp_b200 import ensemble as ens
    one = pd.date_range("2004-02-29", periods=1)
    for kind in ("year", "month", "all"):
        assert ens.period_bounds(one, kind)[0].tolist() == [[0, 0]]
    idx = pd.date_range("2004-01-01", "2005-12-31")
    b, names = ens.period_bounds(idx, [("2004-10-01", "2005-09-30"), ("2005-04-01", "2005-09-30"),
                                       ("2004-01-01", "2004-01-01")])
    assert b.tolist() == [[274, 638], [456, 638], [0, 0]]
    assert names[0] == "2004-10-01/2005-09-30"


@pytest.mark.parametrize("periods, match", [
    ("week", "unknown periods"),
    ([], "no periods"),
    ([("2004-03-01", "2004-02-01")], "reversed"),
    ([("2003-12-31", "2004-02-01")], "not inside the record"),
    ([("2004-02-01", "2005-01-01")], "not inside the record"),
    ([("2004-02-01",)], "pair of dates"),
])
def test_bad_periods_are_refused(periods, match):
    from simplyp_b200 import ensemble as ens
    with pytest.raises(ValueError, match=match):
        ens.period_bounds(pd.date_range("2004-01-01", "2004-12-31"), periods)


# --------------------------------------------------------------------------- result object
def _result():
    from simplyp_b200 import ensemble as ens
    dates = pd.date_range("2004-01-01", "2005-12-31")
    bounds, names = ens.period_bounds(dates, "year")
    values = np.array([[1.0, 2.0, 3.0, np.nan, 5.0], [0.1, 0.2, np.inf, 0.4, np.nan],
                       [np.nan] * 5, [7.0, 7.0, 7.0, 7.0, 7.0]])
    q = np.array([0.5])
    with np.errstate(all="ignore"):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            quant = np.nanquantile(values, q, axis=-1)
            mean = np.nanmean(values, axis=-1)
    return ens.PeriodStatistics(q=q, quantiles=quant, values=values, mean=mean,
                                count=np.sum(~np.isnan(values), axis=-1), n_failed=1,
                                series=[("waterbody", "TP", "load"), (1, "TDP", "fwmc")], periods=names,
                                bounds=bounds, n_days=bounds[:, 1] - bounds[:, 0] + 1, dates=dates)


def test_exceedance_counts_the_finite_entries_of_a_row():
    r = _result()
    assert r.exceedance(0, 2.0) == 2 / 4
    assert r.exceedance(("waterbody", "TP", "load", 2004), 2.0) == 2 / 4
    assert r.exceedance(("waterbody", "TP", "load", "2004"), 0.0) == 1.0
    assert r.exceedance(("waterbody", "TP", "load", 2005), 0.15) == 2 / 3  # +inf is not finite
    assert math.isnan(r.exceedance((1, "TDP", "fwmc", 2004), 0.0))        # no finite entry
    assert r.exceedance((1, "TDP", "fwmc", 2005), 7.0) == 0.0
    with pytest.raises(ValueError, match="no row"):
        r.exceedance((1, "TDP", "fwmc", 2006), 0.0)
    with pytest.raises(ValueError, match="outside"):
        r.exceedance(4, 0.0)


def test_table_has_one_row_per_series_and_period():
    r = _result()
    t = r.table()
    assert list(t[["target", "variable", "statistic", "period"]].itertuples(index=False, name=None)) == r.labels
    assert t["n_days"].tolist() == [366, 365, 366, 365]
    assert t["start"].iloc[1] == pd.Timestamp("2005-01-01") and t["end"].iloc[1] == pd.Timestamp("2005-12-31")
    assert _same(t["q0.5"].to_numpy(), r.quantiles[0])
    assert _same(t["mean"].to_numpy(), r.mean) and t["count"].tolist() == [4, 4, 0, 5]


# --------------------------------------------------------------------------- input checks
def _tarland():
    from simplyp_b200 import tarland
    return tarland.load("2004-01-01", "2004-12-31", dynamic="y")


@pytest.mark.parametrize("series, kw, match", [
    ([(1, "NO3", "load")], {}, "unknown variable"),
    ([(1, "TP", "median")], {}, "unknown statistic"),
    ([(1, "Q", "fwmc")], {}, "undefined"),
    ([(7, "TP", "load")], {}, "not in SC_list"),
    ([("loch", "TP", "load")], {}, "not in SC_list"),
    ([("waterbody", "TP", "load")], {}, "flagged"),
    ([(1, "TP")], {}, r"\(target, variable, statistic\)"),
    ([], {}, "no series"),
    ([(1, "TP", "load")], {"periods": "decade"}, "unknown periods"),
    ([(1, "TP", "load")], {"periods": [("2004-06-01", "2004-05-01")]}, "reversed"),
    ([(1, "TP", "load")], {"periods": [("2004-06-01", "2005-05-01")]}, "not inside"),
    ([(1, "TP", "load")], {"periods": []}, "no periods"),
    ([(1, "TP", "load")], {"quantiles": [0.5, np.nan]}, "finite"),
    ([(1, "TP", "load")], {"quantiles": [1.5]}, r"\[0, 1\]"),
    ([(1, "TP", "load")], {"quantiles": []}, "1..16"),
])
def test_period_statistics_rejects_bad_input_before_device_work(series, kw, match, monkeypatch):
    from simplyp_b200 import engine, ensemble as ens

    def no_device(*a, **k):
        raise AssertionError("device work before the input check")
    monkeypatch.setattr(engine, "Engine", no_device)
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    with pytest.raises(ValueError, match=match):
        ens.period_statistics(met, p_struc, p_SU, p_LU, p_SC, p, dyn, {"fc": np.array([200.0, 300.0])}, series, **kw)


class _SmallDevice:
    """An engine with 1 MB free that refuses any work."""

    def free_bytes(self):
        return 1 << 20

    def __getattr__(self, name):
        raise AssertionError("device work before the memory check: %s" % name)


def test_period_statistics_refuses_values_over_half_the_free_memory():
    from simplyp_b200 import ensemble as ens
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    samples = {"fc": np.linspace(100.0, 400.0, 2000)}                 # 8 * 3 * 12 * 2000 B = 576 kB > 512 kB
    with pytest.raises(ValueError, match="thin"):
        ens.period_statistics(met, p_struc, p_SU, p_LU, p_SC, p, dyn, samples,
                              [(1, "Q", "load"), (1, "TDP", "fwmc"), (1, "TP", "mean")], periods="month",
                              engine=_SmallDevice())


def test_period_entry_point_raises_without_device():
    from simplyp_b200 import _cabi
    lib = _cabi.load()
    if lib.simplyp_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    dims = _cabi.make_dims(4, 2, 10, 1, 0, 0)

    def call(desc, bounds, wb=(), ptr=8, total=4):
        d = (C.c_int32 * len(desc))(*desc)
        b = (C.c_int32 * len(bounds))(*bounds)
        w = (C.c_int32 * max(len(wb), 1))(*wb)
        return lib.simplyp_period_aggregates_device(C.byref(dims), ptr, 8, 8, 8, d, len(desc) // 3, b,
                                                    len(bounds) // 2, w if wb else None, len(wb), 8, total, 0, None)
    # bad arguments first (SIMPLYP_EINVAL), then the missing device (SIMPLYP_ENODEVICE)
    assert call([0, 1, 1], [0, 9], ptr=None) == -1
    assert call([2, 1, 1], [0, 9]) == -1                     # reach outside 0..S-1
    assert call([-1, 1, 1], [0, 9]) == -1                    # water body without reaches
    assert call([-1, 1, 1], [0, 9], wb=[2]) == -1            # water-body reach outside 0..S-1
    assert call([0, 6, 1], [0, 9]) == -1                     # variable kind
    assert call([0, 1, 3], [0, 9]) == -1                     # statistic
    assert call([0, 0, 2], [0, 9]) == -1                     # fwmc of Q
    assert call([0, 1, 1], [0, 10]) == -1                    # day outside the record
    assert call([0, 1, 1], [5, 4]) == -1                     # reversed
    assert call([0, 1, 1], [0, 9], total=3) == -1            # members outside n_members_total
    assert call([0, 1, 1], [0, 9]) == -2
    assert call([-1, 5, 2, 1, 0, 0], [0, 9, 3, 3], wb=[1, 0]) == -2
