"""CPU tier of the Morris screening: the host build of simplyp_morris.cuh (tests/morris_host.cpp) against NumPy — the
trajectories' structure and distribution, the Philox words, the design values and the greedy selection, bitwise —
the fsum reference estimators on analytic functions, MorrisResult.screen, and the input checks of
sensitivity.elementary_effects."""
import numpy as np
import pytest
from scipy import stats

from tests import morris_reference as ref

SEED = 0x5eed_0000_3022


@pytest.fixture(scope="module")
def host():
    from tests import morris_host
    morris_host.load()
    return morris_host


def _morris(bounds, r, p=4, n_candidates=0, seed=SEED, targets=None, n_sc=1):
    from simplyp_b200 import _cabi
    b = np.asarray(bounds, dtype=np.float64)
    targets = targets or [(_cabi.MCMC_MEMBER, k, 0) for k in range(b.shape[0])]
    return _cabi.make_morris(targets, b[:, 0], b[:, 1], n_sc, r, p, n_candidates, False, seed)


@pytest.mark.parametrize("K, p", [(1, 2), (3, 4), (18, 4), (7, 10), (64, 16)])
def test_trajectories_move_every_coordinate_once_by_half_the_levels(host, K, p):
    lev = host.levels(SEED, K, p, 200)
    assert lev.min() >= 0 and lev.max() <= p - 1
    d = np.diff(lev, axis=1)                                   # [n][K][K]
    assert np.all((d != 0).sum(axis=2) == 1)
    assert np.all(np.abs(d[d != 0]) == p // 2)
    assert np.all((d != 0).sum(axis=1) == 1)                   # each coordinate moves at exactly one step


def test_trajectory_draws_pass_chi_square(host):
    K, p, n = 6, 8, 10_000
    lev = host.levels(SEED, K, p, n)
    h = p // 2
    d = np.diff(lev, axis=1)
    neg = (d.sum(axis=1) < 0).astype(int)                      # [n][K] direction of each coordinate
    base = lev[:, 0, :] - h * neg                               # base levels 0..h-1
    pos = np.argmax(d != 0, axis=1)                             # [n][K] step that moves each coordinate
    for z in range(K):
        assert stats.chisquare(np.bincount(base[:, z], minlength=h)).pvalue > 1e-4
        assert stats.chisquare(np.bincount(neg[:, z], minlength=2)).pvalue > 1e-4
        assert stats.chisquare(np.bincount(pos[:, z], minlength=K)).pvalue > 1e-4


@pytest.mark.parametrize("K, p, c0", [(1, 2, 0), (5, 4, 0), (18, 6, 4000), (64, 16, 7)])
def test_trajectories_equal_the_numpy_philox_words(host, K, p, c0):
    assert np.array_equal(host.levels(SEED, K, p, 64, c0), ref.levels(SEED, K, p, 64, c0))


@pytest.mark.parametrize("selected", [None, [5, 0, 17, 3]])
def test_design_values_equal_numpy_bitwise(host, selected):
    from simplyp_b200 import ensemble as ens
    bounds = np.array(list(ens.TARLAND_RANGES.values()))
    K, p = bounds.shape[0], 6
    r = 4 if selected else 9
    mo = _morris(bounds, r, p, 20 if selected else 0)
    cand = np.asarray(selected) if selected else np.arange(r)
    lev = ref.levels(SEED, K, p, 20)[cand]
    want = ref.design_values(bounds, lev, p)
    M = r * (K + 1)
    got = np.concatenate([host.design(mo, 0, 7, selected), host.design(mo, 7, M - 7, selected)])
    assert np.array_equal(got, want)
    assert np.all(got >= bounds[:, 0]) and np.all(got <= bounds[:, 1])


@pytest.mark.parametrize("nc, r, K, p", [(12, 3, 2, 4), (40, 6, 5, 4), (60, 10, 18, 4), (30, 4, 7, 10),
                                          (16, 5, 64, 16), (25, 2, 3, 2)])
def test_greedy_selection_equals_numpy(host, nc, r, K, p):
    mo = _morris([(0.0, 1.0)] * K, r, p, nc)
    lev = ref.levels(SEED, K, p, nc)
    want, D = ref.select(lev, r)
    got = host.select(mo)
    assert np.array_equal(got, want)
    assert len(set(got.tolist())) == r
    assert ref.spread(D, got) > ref.spread(D, range(r))
    m, l = got[0], got[1]
    assert D[m, l] == ref.distance(lev[m], lev[l])


def test_bootstrap_picks_are_the_philox_words_mapped(host):
    for n in (1, 3, 100, 1001):
        got = host.picks(SEED, 3, n)
        for b in range(3):
            assert np.array_equal(got[b], ref.pick(ref._words(SEED, [b], n, 1)[0], n))
        assert got.min() >= 0 and got.max() < n


# ---- the fsum reference estimators on analytic functions
def _analytic(f, bounds, r=50, p=4, seed=SEED):
    bounds = np.asarray(bounds, dtype=np.float64)
    lev = ref.levels(seed, bounds.shape[0], p, r)
    X = ref.design_values(bounds, lev, p)
    return f(X), lev


def test_linear_function_gives_its_slopes_times_the_box():
    bounds = np.array([[0.0, 2.0], [-1.0, 1.0], [10.0, 40.0], [0.0, 1.0]])
    c = np.array([3.0, -2.0, 0.5, 0.0])
    y, lev = _analytic(lambda X: X @ c, bounds)
    res = ref.effects(y, lev, 4)
    want = c * (bounds[:, 1] - bounds[:, 0])
    assert np.allclose(res["mu"], want, rtol=1e-12, atol=1e-12)
    assert np.allclose(res["mu_star"], np.abs(want), rtol=1e-12, atol=1e-12)
    assert np.all(res["sigma"] <= 1e-10)
    assert res["mu_star"][3] == 0.0 and res["mu"][3] == 0.0 and res["sigma"][3] == 0.0


def test_product_term_spreads_both_factors():
    bounds = np.array([[0.0, 1.0]] * 3)
    y, lev = _analytic(lambda X: X[:, 0] * X[:, 1] + X[:, 2], bounds)
    res = ref.effects(y, lev, 4)
    assert res["sigma"][0] > 0.1 and res["sigma"][1] > 0.1 and res["sigma"][2] <= 1e-12


def test_reference_drops_non_finite_trajectories():
    bounds = np.array([[0.0, 1.0]] * 3)
    y, lev = _analytic(lambda X: X.sum(axis=1), bounds, r=10)
    y[4 * 2 + 1] = np.nan
    y[4 * 7 + 3] = np.inf
    assert ref.effects(y, lev, 4)["n"] == 8
    assert np.all(np.isnan(ref.effects(np.full(40, np.nan), lev, 4)["mu_star"]))


# ---- MorrisResult.screen
def _result(mu_star):
    from simplyp_b200.sensitivity import MorrisResult
    mu_star = np.asarray(mu_star, dtype=np.float64)
    R, K = mu_star.shape
    names = ["fc", "alpha", "T_g", "err_m:Q"][:K]
    return MorrisResult(names=names, bounds=np.zeros((K, 2)), labels=[(1, "Q", "NSE"), (1, "TDP", "NSE")][:R],
                        mu=mu_star, mu_star=mu_star, sigma=mu_star, mu_star_conf=mu_star, n_used=np.full(R, 10),
                        n_failed=0, selected=np.arange(10), num_levels=4, conf_level=0.95,
                        ranges={n: (float(k), float(k) + 1.0) for k, n in enumerate(names)})


def test_screen_keeps_parameters_that_matter_in_some_row_in_their_order():
    res = _result([[1.0, 0.05, 0.2, 0.0], [0.0, 0.3, 0.001, 0.0]])
    assert list(res.screen(0.1)) == ["fc", "alpha", "T_g"]
    assert res.screen(0.1) == {"fc": (0.0, 1.0), "alpha": (1.0, 2.0), "T_g": (2.0, 3.0)}
    assert list(res.screen(0.1, rows=[0])) == ["fc", "T_g"]
    assert list(res.screen(0.5, rows=[(1, "TDP", "NSE")])) == ["alpha"]
    assert list(_result([[np.nan] * 4, [0.0] * 4]).screen(0.1)) == []
    with pytest.raises(ValueError, match="fraction"):
        res.screen(1.5)


# ---- input checks of sensitivity.elementary_effects, before any device work
def _tarland():
    from simplyp_b200 import tarland
    return tarland.load("2004-01-01", "2004-12-31", dynamic="y")


_RANGES = {"fc": (100.0, 400.0), "alpha": (0.5, 1.2)}


@pytest.mark.parametrize("ranges, kw, match", [
    ({}, {}, "no free parameters"),
    ({"nope": (0.0, 1.0)}, {}, "unknown parameter"),
    ({"fc": (2.0, 1.0)}, {}, "lo < hi"),
    ({"d_maxE_spr": (1.0, 100.0)}, {}, "integer"),
    ({"D_snow_0": (0.0, 1.0)}, {}, "snow_on_device"),
    ({"sc:TDPeff@3": (0.0, 1.0)}, {}, "run-order position"),
    ({"fc": (100.0, 400.0), "err_phi:Q": (0.0, 0.9)}, {}, "AR\\(1\\)"),
    (_RANGES, {"n_trajectories": 1}, "n_trajectories"),
    (_RANGES, {"n_trajectories": 2.5}, "n_trajectories"),
    (_RANGES, {"num_levels": 5}, "num_levels"),
    (_RANGES, {"num_levels": 18}, "num_levels"),
    (_RANGES, {"num_levels": 0}, "num_levels"),
    (_RANGES, {"n_candidates": 10}, "n_candidates"),
    (_RANGES, {"n_candidates": 8193}, "n_candidates"),
    (_RANGES, {"objectives": None}, "exactly one"),
    (_RANGES, {"obs_dict": None}, "obs_dict"),
    (_RANGES, {"objectives": ["NSE", "KGE"]}, "unknown statistic"),
    (_RANGES, {"objectives": None, "series": [(7, "Q")]}, "not in SC_list"),
    (_RANGES, {"n_boot": 10001}, "n_boot"),
    (_RANGES, {"conf_level": 1.0}, "conf_level"),
])
def test_elementary_effects_rejects_bad_input_before_device_work(ranges, kw, match, monkeypatch):
    from simplyp_b200 import engine, sensitivity

    def no_device(*a, **k):
        raise AssertionError("device work before the input check")
    monkeypatch.setattr(engine, "Engine", no_device)
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    args = dict(n_trajectories=10, obs_dict=obs, objectives=["NSE"])
    args.update(kw)
    r = args.pop("n_trajectories")
    with pytest.raises(ValueError, match=match):
        sensitivity.elementary_effects(met, p_struc, p_SU, p_LU, p_SC, p, dyn, ranges, r, **args)


class _SmallDevice:
    """An engine with 1 MB free that refuses any work."""

    def free_bytes(self):
        return 1 << 20

    def __getattr__(self, name):
        raise AssertionError("device work before the memory check: %s" % name)


@pytest.mark.parametrize("kw", [{"objectives": ["NSE", "lp"]}, {"series": [(1, "Q")]}])
def test_elementary_effects_refuses_more_than_half_the_free_memory(kw):
    from simplyp_b200 import sensitivity
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    with pytest.raises(ValueError, match="free device memory"):
        sensitivity.elementary_effects(met, p_struc, p_SU, p_LU, p_SC, p, dyn, _RANGES, 5000, obs_dict=obs,
                                       engine=_SmallDevice(), **kw)


def test_morris_entry_points_check_arguments_without_device():
    import ctypes as C
    from simplyp_b200 import _cabi
    lib = _cabi.load()
    if lib.simplyp_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    mo = _morris([(0.0, 1.0), (0.0, 2.0)], 4, 4, 20)
    plain = _morris([(0.0, 1.0), (0.0, 2.0)], 4)
    for bad in (_morris([(0.0, 1.0)], 4, 5), _morris([(0.0, 1.0)], 1), _morris([(0.0, 1.0)], 4, 4, 4),
                _morris([(0.0, 1.0)], 4, 4, 8193), _morris([(1.0, 0.0)], 4)):
        assert lib.simplyp_morris_workspace_bytes(C.byref(bad), 0) == -1
    ws = _cabi.morris_workspace_bytes(mo, 0)
    assert ws > 0 and _cabi.morris_workspace_bytes(mo, 100) >= ws
    assert _cabi.morris_workspace_bytes(plain, 0) == 0
    assert lib.simplyp_morris_select_device(C.byref(plain), 8, 8, 1 << 20, None) == -1
    assert lib.simplyp_morris_select_device(C.byref(mo), 8, 8, ws - 1, None) == -1
    assert lib.simplyp_morris_select_device(C.byref(mo), 8, 8, ws, None) == -2
    assert lib.simplyp_morris_design_device(C.byref(mo), None, 0, 4, 8, 8, None) == -1
    assert lib.simplyp_morris_design_device(C.byref(plain), None, 0, 13, 8, 8, None) == -1
    assert lib.simplyp_morris_design_device(C.byref(plain), None, 0, 12, 8, 8, None) == -2
    need = _cabi.morris_workspace_bytes(plain, 3)
    assert lib.simplyp_morris_effects_device(C.byref(plain), None, 8, 3, 10, 1.96, 8, 8, 8, 8, 8, 8, need - 1,
                                             None) == -1
    assert lib.simplyp_morris_effects_device(C.byref(plain), None, 8, 3, 10001, 1.96, 8, 8, 8, 8, 8, 8, need,
                                             None) == -1
    assert lib.simplyp_morris_effects_device(C.byref(plain), None, 8, 3, 10, 1.96, 8, 8, 8, 8, 8, 8, need,
                                             None) == -2
