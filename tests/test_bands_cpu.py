"""CPU tier of the posterior predictive bands: the host build of simplyp_bands.cuh (tests/bands_host.cpp) against
NumPy — the Philox words and Box-Muller deviates of the error draws, and the index / interpolation arithmetic of the
selection against np.nanquantile, bitwise — and the input checks of ensemble.predictive_bands."""
import warnings

import numpy as np
import pytest
from scipy import stats

from tests import mcmc_reference as ref

SEED = 0x5eed_0000_b0d5


@pytest.fixture(scope="module")
def host():
    from tests import bands_host
    bands_host.load()
    return bands_host


def eps_reference(seed, member, day, series):
    """Box-Muller of the NumPy Philox words in extended precision (x86 long double: 64-bit significand)."""
    member = np.asarray(member, dtype=np.uint64)
    n = member.size
    ctr = np.stack([member, np.broadcast_to(np.asarray(day, dtype=np.uint64), (n,)),
                    np.broadcast_to(np.asarray(series, dtype=np.uint64), (n,)), np.full(n, 2, dtype=np.uint64)], axis=1)
    r = ref.philox4x32_10(ctr, [seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF]).astype(np.uint64)
    u1 = 1.0 - ref.u53(r[:, 0], r[:, 1])
    u2 = ref.u53(r[:, 2], r[:, 3])
    return np.sqrt(np.longdouble(-2.0) * np.log(u1.astype(np.longdouble))) * cospi_reference(2.0 * u2), u1, u2


def cospi_reference(x):
    """cos(pi x) in extended precision: x - n/2 (|.| <= 1/4) is exact in float64, so the cosine keeps its relative
    accuracy next to its zeros."""
    pi = np.longdouble("3.14159265358979323846264338327950288")
    n = np.rint(2.0 * x)
    t = pi * (x - 0.5 * n).astype(np.longdouble)
    k = n.astype(np.int64) & 3
    return np.select([k == 0, k == 1, k == 2], [np.cos(t), -np.sin(t), -np.cos(t)], np.sin(t))


# The host eps has three roundings of its own (log, sqrt, product) and a cosine of pi r formed from cos / sin of a
# rounded pi r (|r| <= 1/4): within 8 ulp of the extended-precision value.  The device's cospi is within 2 ulp, so a
# device eps lies within EPS_ULPS + 4 ulp of the host one.
EPS_ULPS = 8


def test_band_words_equal_numpy_philox(host):
    rng = np.random.default_rng(2)
    m = rng.integers(0, 2 ** 31 - 1, 5000)
    d = rng.integers(0, 11000, 5000)
    v = rng.integers(0, 40, 5000)
    ctr = np.stack([m, d, v, np.full(5000, 2)], axis=1).astype(np.uint64)
    want = ref.philox4x32_10(ctr, [SEED & 0xFFFFFFFF, SEED >> 32])
    assert np.array_equal(host.words(SEED, m, d, v), want)
    # the sampler's blocks 0 and 1 of the same first three words give other words
    for block in (0, 1):
        other = ref.philox4x32_10(np.stack([m, d, v, np.full(5000, block)], axis=1).astype(np.uint64),
                                  [SEED & 0xFFFFFFFF, SEED >> 32])
        assert not np.any(np.all(other == want, axis=1))


def test_host_epsilon_equals_numpy_box_muller(host):
    rng = np.random.default_rng(3)
    m = rng.integers(0, 2 ** 31 - 1, 200000)
    d = rng.integers(0, 11000, 200000)
    v = rng.integers(0, 40, 200000)
    got = host.epsilon(SEED, m, d, v)
    want, u1, u2 = eps_reference(SEED, m, d, v)
    err = np.abs(got.astype(np.longdouble) - want)
    assert np.all(err <= EPS_ULPS * np.spacing(np.abs(want.astype(np.float64)))), float(np.max(err))
    # also the quadrant boundaries of the cosine: u2 on multiples of 1/8
    assert np.all(np.isfinite(got)) and np.all(u1 > 0.0) and np.all(u1 <= 1.0)


def test_host_epsilon_is_standard_normal(host):
    n = 1_000_000
    m = np.arange(n) % 5000
    d = np.arange(n) // 5000
    eps = host.epsilon(SEED, m, d, 3)
    assert stats.kstest(eps, "norm").pvalue > 1e-3
    assert abs(eps.mean()) < 5.0 / np.sqrt(n) and abs(eps.std() - 1.0) < 5.0 / np.sqrt(2 * n)


def _np_nanquantile(x, q):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return np.nanquantile(x, q, axis=-1)


def _same(a, b):
    """Bitwise equal, NaN equal to NaN, +0 equal to -0."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


Q_GRID = [0.0, 0.025, 0.1, 0.25, 1 / 3, 0.5, 0.75, 0.9, 0.975, 1.0, 0.999999, 1e-9]


def test_host_quantiles_equal_numpy_on_random_rows(host):
    rng = np.random.default_rng(4)
    for N in (3, 7, 64, 501):
        x = rng.normal(size=(200, N))
        x[:50] = np.round(x[:50], 1)                                  # ties
        x[rng.random(x.shape) < 0.15] = np.nan
        x[50:60, 0] = np.inf
        x[60:70, -1] = -np.inf
        x[70:75] = np.nan                                              # all-NaN rows
        x[75:80, 1:] = np.nan                                          # n <= 1
        x[80:85] = 0.0
        x[80:85, ::2] = -0.0
        assert _same(host.nanquantile(x, Q_GRID), _np_nanquantile(x, Q_GRID))


@pytest.mark.parametrize("row", [[], [np.nan], [2.5], [-1.0, 3.0], [np.nan, 3.0, np.nan, -1.0], [np.inf],
                                 [1.0, np.inf], [-np.inf, 1.0], [-np.inf, np.inf], [0.0, -0.0]])
def test_host_quantiles_equal_numpy_on_short_rows(host, row):
    x = np.asarray([row], dtype=np.float64).reshape(1, len(row)) if row else np.zeros((1, 0))
    q = [0.0, 0.25, 0.5, 0.75, 1.0]
    want = _np_nanquantile(x, q) if row else np.full((5, 1), np.nan)
    assert _same(host.nanquantile(x, q), want)


def test_host_quantiles_where_g_is_exactly_one_half(host):
    rng = np.random.default_rng(5)
    x = rng.normal(size=(64, 9))                                       # (n - 1) q = 8 q: g = 0.5 at q = k/8 + 1/16
    q = [1 / 16, 3 / 16, 0.5 + 1 / 16, 15 / 16]
    assert _same(host.nanquantile(x, q), _np_nanquantile(x, q))
    x = rng.normal(size=(64, 3))                                       # 2 q = 0.5, 1.5
    assert _same(host.nanquantile(x, [0.25, 0.75]), _np_nanquantile(x, [0.25, 0.75]))


def test_keys_order_values_and_put_nan_last(host):
    x = np.array([np.nan, -np.inf, -1e308, -1.0, -5e-324, -0.0, 0.0, 5e-324, 1.0, 1e308, np.inf, -np.nan])
    k, back = host.keys(x)
    order = np.argsort(k, kind="stable")
    assert list(order[:-2]) == list(range(1, 11)) and set(order[-2:]) == {0, 11}
    assert _same(back[1:11], x[1:11]) and np.all(np.isnan(back[[0, 11]]))
    assert np.signbit(back[5]) and not np.signbit(back[6])


# ---- input checks of ensemble.predictive_bands, before any device work
def _tarland():
    from simplyp_b200 import tarland
    return tarland.load("2004-01-01", "2004-12-31", dynamic="y")


@pytest.mark.parametrize("series, kw, match", [
    ([(1, "NO3")], {}, "unknown variable"),
    ([(7, "Q")], {}, "not in SC_list"),
    ([], {}, "no series"),
    ([(1, "Q")], {"quantiles": [0.5, np.nan]}, "finite"),
    ([(1, "Q")], {"quantiles": [0.5, np.inf]}, "finite"),
    ([(1, "Q")], {"quantiles": [-0.1, 0.5]}, r"\[0, 1\]"),
    ([(1, "Q")], {"quantiles": [0.5, 1.5]}, r"\[0, 1\]"),
    ([(1, "Q")], {"quantiles": np.linspace(0, 1, 17)}, "1..16"),
    ([(1, "Q")], {"quantiles": []}, "1..16"),
])
def test_predictive_bands_rejects_bad_input_before_device_work(series, kw, match, monkeypatch):
    from simplyp_b200 import engine, ensemble as ens

    def no_device(*a, **k):
        raise AssertionError("device work before the input check")
    monkeypatch.setattr(engine, "Engine", no_device)
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    with pytest.raises(ValueError, match=match):
        ens.predictive_bands(met, p_struc, p_SU, p_LU, p_SC, p, dyn, {"fc": np.array([200.0, 300.0])}, series, **kw)


class _SmallDevice:
    """An engine with 1 MB free that refuses any work."""

    def free_bytes(self):
        return 1 << 20

    def __getattr__(self, name):
        raise AssertionError("device work before the memory check: %s" % name)


def test_predictive_bands_refuses_draws_over_half_the_free_memory():
    from simplyp_b200 import ensemble as ens
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    samples = {"fc": np.linspace(100.0, 400.0, 400)}                  # 8 * 2 * 366 * 400 B = 2.3 MB > 0.5 MB
    with pytest.raises(ValueError, match="thin"):
        ens.predictive_bands(met, p_struc, p_SU, p_LU, p_SC, p, dyn, samples, [(1, "Q"), (1, "TDP")],
                             engine=_SmallDevice())


def test_coverage_needs_computed_bounds_and_counts_like_numpy():
    import pandas as pd
    from simplyp_b200 import ensemble as ens
    dates = pd.date_range("2004-01-01", periods=6)
    q = np.array([0.1, 0.5, 0.9])
    lo, mid, hi = np.zeros((1, 6)), np.ones((1, 6)), np.full((1, 6), 2.0)
    b = ens.PredictiveBands(q=q, quantiles=np.stack([lo, mid, hi]), mean=mid, count=np.full((1, 6), 10),
                            n_failed=0, labels=[(1, "Q")], dates=dates)
    obs = {1: pd.DataFrame({"Q": [0.0, 2.0, 2.5, np.nan, -1.0, 1.0]}, index=dates)}
    assert b.coverage(obs, 0.1, 0.9) == {(1, "Q"): (5, 3 / 5)}
    with pytest.raises(ValueError, match="not one of"):
        b.coverage(obs, 0.05, 0.9)
    with pytest.raises(ValueError, match="not one of"):
        b.coverage(obs, 0.1, 0.95)


def test_band_entry_points_raise_without_device():
    import ctypes as C
    from simplyp_b200 import _cabi
    lib = _cabi.load()
    if lib.simplyp_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    dims = _cabi.make_dims(4, 1, 10, 1, 0, 0)
    q = (C.c_double * 1)(0.5)
    # bad arguments first (SIMPLYP_EINVAL), then the missing device (SIMPLYP_ENODEVICE)
    assert lib.simplyp_predictive_draws_device(C.byref(dims), None, 8, 8, 8, 8, 1, 8, 4, 0, 0, 0, None) == -1
    assert lib.simplyp_predictive_draws_device(C.byref(dims), 8, 8, 8, 8, 8, 1, 8, 3, 0, 0, 0, None) == -1
    assert lib.simplyp_predictive_draws_device(C.byref(dims), 8, 8, 8, 8, 8, 0, 8, 4, 0, 0, 0, None) == -1
    assert lib.simplyp_predictive_draws_device(C.byref(dims), 8, 8, 8, 8, 8, 1, 8, 4, 0, 0, 0, None) == -2
    assert lib.simplyp_nanquantile_device(8, 4, 0, q, 1, 8, 8, 8, None, 0, None) == -1
    assert lib.simplyp_nanquantile_device(8, 4, 10, q, 17, 8, 8, 8, None, 0, None) == -1
    assert lib.simplyp_nanquantile_device(8, 4, 10, (C.c_double * 1)(1.5), 1, 8, 8, 8, None, 0, None) == -1
    assert lib.simplyp_nanquantile_device(None, 4, 10, q, 1, 8, 8, 8, None, 0, None) == -1
    assert lib.simplyp_nanquantile_device(8, 4, 10, q, 1, 8, 8, 8, None, 0, None) == -2
