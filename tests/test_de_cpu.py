"""CPU tier of differential evolution: the host build of simplyp_de.cuh (tests/de_host.cpp) against the NumPy
restatement (tests/de_reference.py) — picks, trials, scaling, energies and selection, bitwise — the restatement
against scipy.optimize.differential_evolution on Rosenbrock and the sphere, and the input checks of
optimize.differential_evolution."""
import numpy as np
import pytest
from scipy.optimize import differential_evolution as scipy_de

from tests import de_reference as ref

SEED = 0x5eed_0000_0de0


@pytest.fixture(scope="module")
def host():
    from tests import de_host
    de_host.load()
    return de_host


def _de(N, K, strategy="best1bin", mutation=(0.5, 1.0), recombination=0.7, bounds=None, seed=SEED):
    from simplyp_b200 import _cabi
    b = np.asarray(bounds if bounds is not None else [(-1.0 - k, 2.0 + 3 * k) for k in range(K)], dtype=np.float64)
    return _cabi.make_de(N, [(_cabi.MCMC_MEMBER, k, 0) for k in range(K)], b[:, 0], b[:, 1], 1, 1,
                         strategy=strategy, mutation=mutation, recombination=recombination, seed=seed)


@pytest.mark.parametrize("strategy", ["best1bin", "rand1bin"])
@pytest.mark.parametrize("K", [1, 2, 18, 64])
@pytest.mark.parametrize("case", ["min_population", "interior", "faces_and_large_F"])
def test_trials_equal_numpy_bitwise(host, strategy, K, case):
    rng = np.random.default_rng(K)
    N = {"best1bin": 3, "rand1bin": 4}[strategy] if case == "min_population" else 97
    mutation = (1.9, 1.999) if case == "faces_and_large_F" else (0.5, 1.0)
    pop = rng.uniform(size=(N, K))
    if case == "faces_and_large_F":
        pop[rng.uniform(size=pop.shape) < 0.5] = 0.0
        pop[rng.uniform(size=pop.shape) < 0.3] = 1.0
    de = _de(N, K, strategy, mutation)
    best = N // 2
    outside = 0
    for g in (0, 1, 12345, (1 << 32) + 7):
        F = ref.dither(SEED, g, mutation)
        assert host.dither(de, g) == F and mutation[0] <= F <= mutation[1]
        got = host.trials(de, pop, best, g)
        assert np.array_equal(got, ref.trials(pop, best, g, SEED, strategy, F, 0.7))
        assert np.all((got >= 0.0) & (got <= 1.0))
        outside += ref.bprime_outside(pop, best, g, SEED, strategy, F)
    if case == "faces_and_large_F":
        assert outside > 0          # redraws happened and still matched


@pytest.mark.parametrize("strategy", ["best1bin", "rand1bin"])
def test_picks_are_distinct_and_never_the_target(host, strategy):
    N, K = 10007, 3
    de = _de(N, K, strategy)
    n = 3 if strategy == "rand1bin" else 2
    for g in (0, 5):
        got = host.picks(de, g)
        r, fill = ref.picks(N, K, g, SEED, strategy)
        assert np.array_equal(got[:, :3], r) and np.array_equal(got[:, 3], fill)
        p = got[:, :n].astype(np.int64)
        i = np.arange(N)
        assert np.all((p >= 0) & (p < N))
        assert np.all(p != i[:, None])
        for a in range(n):
            for b in range(a + 1, n):
                assert np.all(p[:, a] != p[:, b])
        if n == 2:
            assert np.all(got[:, 2] == -1)
    # over 40 generations of 1,000 members each member is picked about 40 n times
    small = _de(1000, K, strategy)
    seen = np.zeros(1000, dtype=np.int64)
    for g in range(40):
        np.add.at(seen, host.picks(small, g)[:, :n].ravel(), 1)
    assert seen.min() > 0 and abs(seen.mean() - 40 * n) < 1e-9 and seen.std() < 2 * np.sqrt(40 * n)


def test_minimum_population_picks_every_other_member(host):
    for strategy, N in (("best1bin", 3), ("rand1bin", 4)):
        de = _de(N, 2, strategy)
        for g in range(20):
            p = host.picks(de, g)[:, :N - 1 if strategy == "rand1bin" else 2]
            for i in range(N):
                assert i not in p[i] and len(set(p[i])) == p.shape[1]


def test_selection_follows_le_and_nan_or_failed_become_inf(host):
    N, K, R = 8, 3, 2
    rng = np.random.default_rng(3)
    y = rng.normal(size=(R, N))
    w = np.array([1.0, -0.5])
    y[0, 2] = np.nan
    y[1, 5] = np.inf                  # -0.5 * inf -> E = +inf
    diag = np.zeros((N, 2, 4), dtype=np.int64)
    diag[4, 1, 3] = 7                 # a failed integration, whatever its statistics
    e = host.energy(y, w, diag)
    assert np.array_equal(e, ref.energies(y, w, np.any(diag[..., 3] != 0, axis=1)))
    assert e[2] == e[4] == e[5] == np.inf and np.all(np.isfinite(np.delete(e, [2, 4, 5])))
    pop = rng.uniform(size=(N, K))
    trial = rng.uniform(size=(N, K))
    energy = e.copy()
    energy[0] = e[0]                  # equal: the trial replaces
    energy[1] = e[1] - 1.0            # better target: kept
    energy[3] = e[3] + 1.0            # worse target: replaced
    energy[2] = np.inf                # inf <= inf: replaced, as scipy's _accept_trial
    energy[4] = 0.0                   # a failed trial never replaces a finite target
    before_pop, before_e = pop.copy(), energy.copy()
    ok = host.select(e, trial, pop, energy)
    want = e <= before_e
    assert np.array_equal(ok, want)
    assert ok[0] and not ok[1] and ok[2] and ok[3] and not ok[4]
    assert np.array_equal(pop, np.where(want[:, None], trial, before_pop))
    assert np.array_equal(energy, np.where(want, e, before_e))


def test_scaled_values_stay_inside_the_box(host):
    from simplyp_b200 import optimize
    K = 6
    bounds = np.array([(0.1, 0.3), (-1e-300, 1e-300), (100.0, 400.0), (0.05, 1.0), (1.0 - 2e-16, 1.0),
                       (-7.3, 1e6)])
    de = _de(5, K, bounds=bounds)
    rng = np.random.default_rng(11)
    u = np.concatenate([rng.uniform(size=(20000, K)), np.zeros((1, K)), np.ones((1, K)),
                        np.full((1, K), np.nextafter(1.0, 0.0)), np.full((1, K), 0.5)])
    got = host.scale(de, u)
    assert np.array_equal(got, ref.scale(u, bounds))
    assert np.array_equal(got, optimize.scale(u, bounds))
    assert np.all((got >= bounds[:, 0]) & (got <= bounds[:, 1]))
    v = 0.5 * (bounds[:, 0] + bounds[:, 1]) + (u - 0.5) * np.fabs(bounds[:, 0] - bounds[:, 1])
    moved = got != v
    assert np.all(moved <= ((v < bounds[:, 0]) | (v > bounds[:, 1])))   # the clamp is the only change
    assert np.array_equal(optimize.unscale(got[:2], bounds).shape, (2, K))


@pytest.mark.parametrize("fn, box, f_tol, x_opt", [(ref.rosenbrock, (-2.0, 2.0), 1e-10, 1.0),
                                                   (ref.sphere, (-5.0, 5.0), 1e-12, 0.0)])
@pytest.mark.parametrize("strategy", ["best1bin", "rand1bin"])
def test_restatement_and_scipy_reach_the_known_minimum(fn, box, f_tol, x_opt, strategy):
    """The NumPy restatement and scipy's deferred-updating solver, from the same population, both converge to the
    known minimum in a similar number of generations: the restatement is scipy's algorithm."""
    from simplyp_b200 import optimize
    K, N = 5, 75
    bounds = np.array([box] * K)
    u0 = optimize.latin_hypercube_unit(N, K, 2)
    r = ref.run(lambda x: (-fn(x)[None], np.zeros(x.shape[0], bool)), np.array([1.0]), u0, bounds, 5000, SEED,
                strategy=strategy, tol=1e-8)
    s = scipy_de(lambda x: fn(x[None])[0], bounds, strategy=strategy, updating="deferred", polish=False,
                 init=ref.scale(u0, bounds), rng=1, maxiter=5000, tol=1e-8)
    x = ref.scale(r["population"][r["best"]], bounds)
    assert r["converged"] and s.success
    assert r["energy"][r["best"]] <= f_tol and s.fun <= f_tol
    assert np.allclose(x, x_opt, atol=1e-4) and np.allclose(s.x, x_opt, atol=1e-4)
    assert 0.5 < r["generation"] / s.nit < 2.0
    h = r["history"]
    assert np.all(np.diff(h[:, 0]) >= 0)        # the best objective never decreases


# ---- input checks of optimize.differential_evolution, before any device work
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
    (_RANGES, {"strategy": "best2bin"}, "unknown strategy"),
    (_RANGES, {"n_population": 2}, "n_population >= 3"),
    (_RANGES, {"n_population": 3, "strategy": "rand1bin"}, "n_population >= 4"),
    (_RANGES, {"max_generations": 0}, "max_generations"),
    (_RANGES, {"check_every": 0}, "check_every"),
    (_RANGES, {"start_generation": -1}, "start_generation"),
    (_RANGES, {"mutation": (1.0, 0.5)}, "mutation"),
    (_RANGES, {"mutation": (-0.1, 0.5)}, "mutation"),
    (_RANGES, {"mutation": 2.0}, "mutation"),
    (_RANGES, {"mutation": (0.5, np.nan)}, "mutation"),
    (_RANGES, {"recombination": 1.5}, "recombination"),
    (_RANGES, {"recombination": -0.1}, "recombination"),
    (_RANGES, {"tol": -1.0}, "tol"),
    (_RANGES, {"tol": np.inf}, "tol"),
    (_RANGES, {"tol_abs": np.nan}, "tol_abs"),
    (_RANGES, {"objective": "pbias"}, "unknown statistic"),
    (_RANGES, {"objective": "KGE"}, "unknown statistic"),
    (_RANGES, {"objective": {}}, "non-empty"),
    (_RANGES, {"objective": {(7, "Q", "NSE"): 1.0}}, "unknown series"),
    (_RANGES, {"objective": {"NSE": 0.0}}, "zero"),
    (_RANGES, {"objective": {"NSE": np.inf}}, "finite"),
    (_RANGES, {"objective": {"SSE": np.nan, "NSE": 1.0}}, "finite"),
    (_RANGES, {"initial": np.full((8, 3), 200.0)}, "shape"),
    (_RANGES, {"initial": np.full((8, 2), 0.7)}, "inside the box"),
    (_RANGES, {"initial": {"fc": np.full(8, 200.0), "alpha": np.full(8, np.nan)}}, "inside the box"),
])
def test_differential_evolution_rejects_bad_input_before_device_work(ranges, kw, match, monkeypatch):
    from simplyp_b200 import engine, optimize

    def no_device(*a, **k):
        raise AssertionError("device work before the input check")
    monkeypatch.setattr(engine, "Engine", no_device)
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    args = dict(n_population=8, max_generations=5)
    args.update(kw)
    n, g = args.pop("n_population"), args.pop("max_generations")
    with pytest.raises(ValueError, match=match):
        optimize.differential_evolution(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, ranges, n, g, **args)


class _SmallDevice:
    """An engine with 1 MB free that refuses any work."""

    def free_bytes(self):
        return 1 << 20

    def __getattr__(self, name):
        raise AssertionError("device work before the memory check: %s" % name)


def test_differential_evolution_refuses_more_than_half_the_free_memory():
    from simplyp_b200 import optimize
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    with pytest.raises(ValueError, match="free device memory"):
        optimize.differential_evolution(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, _RANGES, 1 << 14, 10,
                                        engine=_SmallDevice())


def test_objective_weights_build_the_sensitivity_rows():
    from simplyp_b200 import optimize, sensitivity
    labels = [(1, "Q"), (1, "TDP")]
    rows, lab, w = optimize._objective_weights("lp", labels)
    assert rows.tolist() == [[0, -1]] and lab == [(None, None, "lp")] and w.tolist() == [1.0]
    rows, lab, w = optimize._objective_weights({"NSE": 1.0, (1, "TDP", "SSE"): -2.0, "lp": 0.5}, labels)
    want_rows, _ = sensitivity.objective_rows(labels, ["NSE", "SSE", "lp"])
    # rows NSE(Q), SSE(Q), NSE(TDP), SSE(TDP), lp; SSE(Q) has weight 0 and is dropped
    assert lab == [(1, "Q", "NSE"), (1, "TDP", "NSE"), (1, "TDP", "SSE"), (None, None, "lp")]
    assert w.tolist() == [1.0, 1.0, -2.0, 0.5]
    assert rows.tolist() == [want_rows[i].tolist() for i in (0, 2, 3, 4)]


def test_de_entry_points_raise_without_device():
    from simplyp_b200 import _cabi
    lib = _cabi.load()
    if lib.simplyp_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    import ctypes as C
    good = _de(8, 2)
    st = _cabi.make_de_state(8, 8, 8, 8, 8, 8, 8, 8, 8, 8, 8, 3)
    bad = [_de(2, 2), _de(3, 2, strategy="rand1bin"), _de(8, 2, mutation=(1.0, 2.0)),
           _de(8, 2, recombination=1.5), _de(8, 2, bounds=[(1.0, 0.0), (0.0, 1.0)])]
    for de in bad:
        assert lib.simplyp_de_trial_device(C.byref(de), C.byref(st), 8, 8, None) == -1
    nan_tol = _de(8, 2)
    nan_tol.tol = float("nan")
    assert lib.simplyp_de_select_device(C.byref(nan_tol), C.byref(st), 8, 8, None) == -1
    null_state = _cabi.make_de_state(8, 8, 8, 8, None, 8, 8, 8, 8, 8, 8, 3)
    assert lib.simplyp_de_init_device(C.byref(good), C.byref(null_state), 8, 8, None) == -1
    assert lib.simplyp_de_select_device(C.byref(good), C.byref(st), None, 8, None) == -1
    assert lib.simplyp_de_trial_device(C.byref(good), C.byref(st), 8, 8, None) == -2
    assert lib.simplyp_de_select_device(C.byref(good), C.byref(st), 8, 8, None) == -2
    assert lib.simplyp_de_init_device(C.byref(good), C.byref(st), 8, 8, None) == -2
