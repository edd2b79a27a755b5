"""CPU tier of the Sobol' sensitivity analysis: the host build of simplyp_sobol.cuh (tests/sobol_host.cpp) against
SciPy and NumPy — the embedded direction numbers, the points, the design values and the bootstrap picks, bitwise —
the fsum reference estimators on analytic functions, and the input checks of sensitivity.sobol_indices."""
import numpy as np
import pytest
from scipy.stats import qmc

from tests import mcmc_reference as mref
from tests import sobol_reference as ref

SEED = 0x5eed_0000_50b0


@pytest.fixture(scope="module")
def host():
    from tests import sobol_host
    sobol_host.load()
    return sobol_host


def test_embedded_direction_numbers_equal_scipy_table(host):
    assert np.array_equal(host.table(), ref.direction_numbers(128))


@pytest.mark.parametrize("K", [1, 2, 18, 64])
@pytest.mark.parametrize("skip", [0, 12345])
def test_points_equal_scipy_sobol_bitwise(host, K, skip):
    n = 1 << 16 if K <= 18 else 1 << 12
    eng = qmc.Sobol(2 * K, scramble=False, bits=32)
    if skip:
        eng.fast_forward(skip)
    x = host.points(2 * K, n, skip)
    assert np.array_equal(x.astype(np.float64) * 2.0 ** -32, eng.random(n))
    assert np.array_equal(x, ref.sobol_points(2 * K, n, skip))


def _sobol(bounds, n_base, skip=0, second_order=False, targets=None, n_sc=1):
    from simplyp_b200 import _cabi
    K = len(bounds)
    targets = targets or [(_cabi.MCMC_MEMBER, k, 0) for k in range(K)]
    b = np.asarray(bounds, dtype=np.float64)
    return _cabi.make_sobol(targets, b[:, 0], b[:, 1], n_sc, n_base, skip, False, second_order)


@pytest.mark.parametrize("second_order", [False, True])
@pytest.mark.parametrize("skip", [0, 1000])
def test_design_values_equal_numpy_bitwise(host, second_order, skip):
    from simplyp_b200 import ensemble as ens
    bounds = np.array(list(ens.TARLAND_RANGES.values()))
    sb = _sobol(bounds, 256, skip, second_order)
    want = ref.design_values(bounds, 256, skip, second_order)
    got = np.concatenate([host.design(sb, 0, 1000), host.design(sb, 1000, want.shape[0] - 1000)])
    assert np.array_equal(got, want)
    # Saltelli layout: AB_j differs from A in column j only, B is the last slot
    K = bounds.shape[0]
    P = want.shape[0] // 256
    X = want.reshape(256, P, K)
    for j in range(K):
        assert np.array_equal(np.delete(X[:, 1 + j], j, axis=1), np.delete(X[:, 0], j, axis=1))
        assert np.array_equal(X[:, 1 + j, j], X[:, P - 1, j])
    if second_order:
        for j in range(K):
            assert np.array_equal(X[:, K + 1 + j, j], X[:, 0, j])


@pytest.mark.parametrize("n", [1, 2, 5, 4096, 100003])
def test_bootstrap_picks_are_the_philox_words_mapped(host, n):
    n_boot = 3
    got = host.picks(SEED, n_boot, n)
    for t in range(n_boot):
        q = np.arange((n + 3) // 4, dtype=np.uint64)
        ctr = np.stack([np.full(q.size, t, dtype=np.uint64), q, np.zeros(q.size, dtype=np.uint64),
                        np.full(q.size, 3, dtype=np.uint64)], axis=1)
        words = mref.philox4x32_10(ctr, [SEED & 0xFFFFFFFF, SEED >> 32]).reshape(-1)[:n]
        assert np.array_equal(got[t], ref.philox_picks(words, n))
    assert got.min() >= 0 and got.max() < n


def test_reference_estimators_recover_ishigami():
    bounds = np.array([[-np.pi, np.pi]] * 3)
    X = ref.design_values(bounds, 1 << 14)
    y = ref.ishigami(X)
    r = ref.indices(y, 3)
    s1, st = ref.ishigami_indices()
    assert np.allclose(r["S1"], s1, atol=0.02) and np.allclose(r["ST"], st, atol=0.02)


def test_reference_drops_non_finite_samples():
    y = np.random.default_rng(1).normal(size=(64, 5))
    y[3, 2], y[10, 0], y[11, 4] = np.nan, np.inf, -np.inf
    assert ref.indices(y.ravel(), 3)["n"] == 61
    assert np.all(np.isnan(ref.indices(np.full(10, np.nan), 3)["S1"]))


# ---- input checks of sensitivity.sobol_indices, before any device work
def _tarland():
    from simplyp_b200 import tarland
    return tarland.load("2004-01-01", "2004-12-31", dynamic="y")


_RANGES = {"fc": (100.0, 400.0), "alpha": (0.5, 1.2)}


@pytest.mark.parametrize("ranges, kw, match", [
    ({}, {}, "no free parameters"),
    ({"nope": (0.0, 1.0)}, {}, "unknown parameter"),
    ({"fc": (2.0, 1.0)}, {}, "lo < hi"),
    ({"fc": (0.0, np.inf)}, {}, "lo < hi"),
    ({"d_maxE_spr": (1.0, 100.0)}, {}, "integer"),
    ({"sc:f_Ar": (0.0, 1.0)}, {}, "land-use"),
    ({"D_snow_0": (0.0, 1.0)}, {}, "snow_on_device"),
    ({"sc:TDPeff@3": (0.0, 1.0)}, {}, "run-order position"),
    (_RANGES, {"n_base": 100}, "power of two"),
    (_RANGES, {"n_base": 1}, "power of two"),
    (_RANGES, {"n_base": 1 << 20, "skip": (1 << 32) - 10}, "2\\^32"),
    (_RANGES, {"skip": -1}, "skip"),
    (_RANGES, {"objectives": None}, "exactly one"),
    (_RANGES, {"series": [(1, "Q")]}, "exactly one"),
    (_RANGES, {"obs_dict": None}, "obs_dict"),
    (_RANGES, {"objectives": ["NSE", "KGE"]}, "unknown statistic"),
    (_RANGES, {"objectives": None, "series": [(1, "NO3")]}, "unknown variable"),
    (_RANGES, {"objectives": None, "series": [(7, "Q")]}, "not in SC_list"),
    (_RANGES, {"objectives": None, "series": []}, "no series"),
    (_RANGES, {"n_boot": -1}, "n_boot"),
    (_RANGES, {"n_boot": 10001}, "n_boot"),
    (_RANGES, {"n_boot": 2.5}, "n_boot"),
    (_RANGES, {"conf_level": 0.0}, "conf_level"),
    (_RANGES, {"conf_level": 1.0}, "conf_level"),
])
def test_sobol_indices_rejects_bad_input_before_device_work(ranges, kw, match, monkeypatch):
    from simplyp_b200 import engine, sensitivity

    def no_device(*a, **k):
        raise AssertionError("device work before the input check")
    monkeypatch.setattr(engine, "Engine", no_device)
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    args = dict(n_base=64, obs_dict=obs, objectives=["NSE"])
    args.update(kw)
    n_base = args.pop("n_base")
    with pytest.raises(ValueError, match=match):
        sensitivity.sobol_indices(met, p_struc, p_SU, p_LU, p_SC, p, dyn, ranges, n_base, **args)


class _SmallDevice:
    """An engine with 1 MB free that refuses any work."""

    def free_bytes(self):
        return 1 << 20

    def __getattr__(self, name):
        raise AssertionError("device work before the memory check: %s" % name)


@pytest.mark.parametrize("kw", [{"objectives": ["NSE", "lp"]}, {"series": [(1, "Q")]}])
def test_sobol_indices_refuses_more_than_half_the_free_memory(kw):
    from simplyp_b200 import sensitivity
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    with pytest.raises(ValueError, match="free device memory"):
        sensitivity.sobol_indices(met, p_struc, p_SU, p_LU, p_SC, p, dyn, _RANGES, 1 << 12, obs_dict=obs,
                                  engine=_SmallDevice(), **kw)


def test_sobol_entry_points_raise_without_device():
    from simplyp_b200 import _cabi
    lib = _cabi.load()
    if lib.simplyp_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    import ctypes as C
    sb = _sobol([(0.0, 1.0), (0.0, 2.0)], 64)
    bad = _sobol([(0.0, 1.0), (0.0, 2.0)], 48)
    assert lib.simplyp_sobol_design_device(C.byref(bad), 0, 4, 8, 8, None) == -1
    assert lib.simplyp_sobol_design_device(C.byref(sb), 0, 64 * 4 + 1, 8, 8, None) == -1
    assert lib.simplyp_sobol_design_device(C.byref(sb), 0, 4, 8, 8, None) == -2
    assert lib.simplyp_sobol_outputs_device(8, 8, 4, 1, 1, 8, 0, 8, None) == -1
    assert lib.simplyp_sobol_outputs_device(8, 8, 4, 1, 1, 8, 1, 8, None) == -2
    assert _cabi.sobol_workspace_bytes(sb, 10) > 0
    ws = _cabi.sobol_workspace_bytes(sb, 3)
    assert lib.simplyp_sobol_indices_device(C.byref(sb), 8, 3, 10, 1.96, 0, 8, 8, 8, 8, None, None, 8, 8, 8, 8,
                                            ws - 1, None) == -1
    assert lib.simplyp_sobol_indices_device(C.byref(sb), 8, 3, 10001, 1.96, 0, 8, 8, 8, 8, None, None, 8, 8, 8, 8,
                                            ws, None) == -1
    assert lib.simplyp_sobol_indices_device(C.byref(sb), 8, 3, 10, 1.96, 0, 8, 8, 8, 8, None, None, 8, 8, 8, 8, ws,
                                            None) == -2
