"""CPU tier of NSGA-II: the NumPy restatement (tests/nsga2_reference.py) against brute-force front peeling and a
textbook crowding distance, the survival and selection orders, the host build of simplyp_nsga2.cuh
(tests/nsga2_host.cpp) against the restatement, the restatement's run on ZDT1, ZDT2 and DTLZ2, and the input checks of
optimize.nsga2."""
import numpy as np
import pytest

from tests import nsga2_reference as ref

SEED = 0x5eed_0000_5a2a


@pytest.fixture(scope="module")
def host():
    from tests import nsga2_host
    nsga2_host.load()
    return nsga2_host


def _ns(N, K, M=2, crossover=0.9, mutation=None, eta_c=15.0, eta_m=20.0, seed=SEED):
    from simplyp_b200 import _cabi
    return _cabi.make_nsga2(N, [(_cabi.MCMC_MEMBER, k, 0) for k in range(K)], np.zeros(K), np.ones(K), 1,
                            [1.0] * M, crossover=crossover, mutation=mutation, eta_c=eta_c, eta_m=eta_m, seed=seed)


def _points(n, M, seed):
    """Oriented objectives with ties, duplicates and NaN rows (infeasible points)."""
    rng = np.random.default_rng(seed)
    f = np.round(rng.normal(size=(n, M)), 1)          # coarse values: many ties
    f[rng.integers(0, n, n // 8)] = f[rng.integers(0, n, n // 8)]   # duplicates
    f[rng.uniform(size=n) < 0.1] = np.nan
    return f


def _brute_force_ranks(f):
    """Textbook peeling: a front is the feasible unranked points no other feasible unranked point dominates."""
    n = f.shape[0]
    ok = ~np.isnan(f[:, 0])
    rank = np.full(n, -1)
    r = 0
    while (ok & (rank < 0)).any():
        left = np.flatnonzero(ok & (rank < 0))
        for i in left:
            if not any(np.all(f[j] >= f[i]) and np.any(f[j] > f[i]) for j in left if j != i):
                rank[i] = r
        r += 1
    rank[~ok] = r
    return rank


@pytest.mark.parametrize("M", [2, 3, 8])
@pytest.mark.parametrize("seed", [1, 2])
def test_ranks_equal_brute_force_peeling(M, seed):
    f = _points(150, M, seed)
    rank, n_fronts, last, before = ref.ranks(f, f.shape[0])
    want = _brute_force_ranks(f)
    assert np.array_equal(rank, want)
    assert n_fronts == want.max() + 1 and last == want.max() and before == np.sum(want < last)
    # stopping once >= N are ranked: the ranked points keep their ranks, the others are not reached
    N = 40
    part, n_fronts, last, before = ref.ranks(f, N)
    reached = part != ref.UNRANKED
    assert np.array_equal(part[reached], want[reached]) and reached.sum() >= N and before < N
    assert np.all(want[~reached] >= last)


def test_a_fully_ordered_set_has_one_point_per_front():
    n = 64
    f = np.stack([np.arange(n, dtype=float)] * 2, axis=1)[::-1].copy()
    rank, n_fronts, last, before = ref.ranks(f, n)
    assert np.array_equal(rank, np.arange(n)) and n_fronts == n and before == n - 1


def _textbook_crowding(f, rank):
    """Deb's crowding distance with a stable argsort per objective (ties in index order)."""
    out = np.zeros(f.shape[0])
    ok = ~np.isnan(f[:, 0]) & (rank != ref.UNRANKED)
    for r in np.unique(rank[ok]):
        F = np.flatnonzero(ok & (rank == r))
        acc = np.zeros(F.size)
        for m in range(f.shape[1]):
            v = f[F, m]
            o = np.argsort(v, kind="stable")
            term = np.zeros(F.size)
            span = v[o[-1]] - v[o[0]]
            for pos in range(1, F.size - 1):
                term[o[pos]] = 0.0 if span == 0 else (v[o[pos + 1]] - v[o[pos - 1]]) / span
            term[o[0]] = term[o[-1]] = np.inf
            acc = acc + term
        out[F] = acc
    return out


@pytest.mark.parametrize("M", [2, 3, 8])
def test_crowding_equals_the_textbook_distance_bitwise(M):
    f = _points(200, M, 7)
    f[:, M - 1] = np.where(np.isnan(f[:, 0]), np.nan, 0.5)            # a constant objective
    rank = ref.ranks(f, f.shape[0])[0]
    got = ref.crowding(f, rank)
    assert np.array_equal(got, _textbook_crowding(f, rank))
    sizes = np.bincount(rank[~np.isnan(f[:, 0])])
    assert {1, 2} & set(sizes.tolist()) or sizes.min() > 2
    for F in (np.array([[0.3, 0.1]]), np.array([[0.3, 0.1], [0.1, 0.3]])):    # fronts of one and two points
        assert np.all(ref.crowding(F, np.zeros(len(F), dtype=np.int64)) == np.inf)


def test_survivors_and_selection_follow_the_stated_orders():
    rng = np.random.default_rng(5)
    f = _points(120, 3, 11)
    rank, _, last, before = ref.ranks(f, 60)
    crowd = ref.crowding(f, rank)
    keep = ref.survivors(rank, crowd, 60)
    key = sorted(range(120), key=lambda i: (rank[i], -crowd[i], i))
    assert keep.tolist() == sorted(key[:60])
    assert np.all(rank[keep] <= last) and np.sum(rank[keep] < last) == before
    # tournaments: lower rank, then larger crowding, then lower index
    a, b = rng.integers(0, 120, 500), rng.integers(0, 120, 500)
    got = ref.better(rank, crowd, a, b)
    want = [min((x, y), key=lambda i: (rank[i], -crowd[i], i)) for x, y in zip(a, b)]
    assert got.tolist() == want


def _zdt_fn(which):
    return lambda x: (ref.zdt(x, which), np.zeros(x.shape[0], bool))


def test_the_ideal_point_over_the_survivors_never_gets_worse():
    from simplyp_b200 import optimize
    u0 = optimize.latin_hypercube_unit(40, 6, 3)

    def fn(x):
        y = ref.zdt(x, 1)
        y[:, x[:, 1] > 0.9] = np.nan                  # a NaN region
        return y, x[:, 2] < 0.05                      # and failed members
    r = ref.run(fn, u0, 30, SEED, [-1.0, -1.0])
    best = r["history"][:, 2:]                        # minimised: the best value never increases
    assert np.all(np.diff(best, axis=0) <= 0) and r["n_failed"] > 0
    assert np.all(r["history"][:, 0] >= 1)


@pytest.mark.parametrize("K", [1, 2, 18, 64])
@pytest.mark.parametrize("case", ["interior", "faces"])
def test_host_offspring_equal_numpy(host, K, case):
    rng = np.random.default_rng(K)
    N = 98
    pop = rng.uniform(size=(N, K))
    if case == "faces":
        pop[rng.uniform(size=pop.shape) < 0.4] = 0.0
        pop[rng.uniform(size=pop.shape) < 0.3] = 1.0
    rank = rng.integers(0, 4, N).astype(np.int32)
    crowd = np.where(rng.uniform(size=N) < 0.1, np.inf, rng.uniform(size=N))
    crowd[:10] = crowd[10:20]                        # ties in crowding as well
    for mutation, eta in ((None, (15.0, 20.0)), (0.5, (0.0, 0.0)), (1.0, (2.0, 100.0))):
        ns = _ns(N, K, mutation=mutation, eta_c=eta[0], eta_m=eta[1])
        for g in (0, 1, 777, (1 << 32) + 5):
            got, dec = host.offspring(ns, pop, rank, crowd, g)
            want, wdec = ref.offspring(pop, rank, crowd, g, SEED, 0.9, ns.mutation, eta[0], eta[1])
            assert np.array_equal(dec, wdec)
            assert np.max(np.abs(got - want)) <= ref.OFFSPRING_ULP * 2.0 ** -52
            assert np.all((got >= 0.0) & (got <= 1.0))
            pk = host.picks(ns, g)
            assert np.array_equal(pk, ref.picks(N, g, SEED))
            assert np.all(pk[:, 0] != pk[:, 1]) and np.all(pk[:, 2] != pk[:, 3])
            assert np.all((pk >= 0) & (pk < N))
        bits = wdec[:, 3:]
        assert (bits & 1).any() and (bits & 4).any() and (bits & 8).any()


def test_tournament_picks_are_uniform(host):
    N = 1000
    ns = _ns(N, 2)
    seen = np.zeros(N, dtype=np.int64)
    for g in range(40):
        np.add.at(seen, host.picks(ns, g).ravel(), 1)
    assert seen.min() > 0 and seen.sum() == 40 * 2 * N and seen.std() < 2 * np.sqrt(80)


def test_host_orientation_and_dominance_equal_numpy(host):
    rng = np.random.default_rng(2)
    M, n = 3, 64
    ns = _ns(n, 2, M=M)
    for m, s in enumerate((1.0, -1.0, 1.0)):
        ns.sense[m] = s
    y = np.round(rng.normal(size=(M, n)), 1)
    y[1, 3], y[0, 4], y[2, 5] = np.nan, np.inf, -np.inf
    status = (rng.uniform(size=n) < 0.1).astype(np.int32)
    f = host.orient(ns, y, status)
    want = ref.orient(y, status, [1.0, -1.0, 1.0])
    assert np.array_equal(f, want, equal_nan=True) and np.isnan(f[[3, 4, 5]]).all()
    assert np.array_equal(host.dominance(f).T, ref.dominance(f).T)


@pytest.mark.parametrize("which, generations, threshold", [(1, 150, 0.02), (2, 200, 0.02)])
def test_reference_driver_reaches_the_zdt_fronts(which, generations, threshold):
    """ZDT1 / ZDT2 with K = 30 and N = 100: the inverted generational distance to 500 points of the analytic front
    falls below the threshold.  (The restatement measured 0.0079 (ZDT1, 150 generations) and 0.0087 (ZDT2, 200).)"""
    from simplyp_b200 import optimize
    u0 = optimize.latin_hypercube_unit(100, 30, which)
    r = ref.run(_zdt_fn(which), u0, generations, SEED + which, [-1.0, -1.0])
    f1 = np.linspace(0.0, 1.0, 500)
    front = np.stack([f1, 1.0 - (np.sqrt(f1) if which == 1 else f1 ** 2)], axis=1)
    d = ref.igd(r["objectives"][r["rank"] == 0], front)
    print("ZDT%d: IGD %.4f after %d generations" % (which, d, generations))
    assert d < threshold


def test_reference_driver_reaches_the_dtlz2_sphere():
    """DTLZ2 with M = 3, K = 12, N = 100, 250 generations: the first-front members lie near the unit sphere (sum of
    squares 1): the median within 0.02, every one within 0.2.  (The restatement measured a median of 0.0125 and a
    largest distance of 0.101.)"""
    from simplyp_b200 import optimize
    u0 = optimize.latin_hypercube_unit(100, 12, 4)
    r = ref.run(lambda x: (ref.dtlz2(x), np.zeros(x.shape[0], bool)), u0, 250, SEED, [-1.0] * 3)
    y = r["objectives"][r["rank"] == 0]
    err = np.abs((y ** 2).sum(axis=1) - 1.0)
    print("DTLZ2: %d front members, |sum f^2 - 1| median %.4f, max %.4f" % (y.shape[0], np.median(err), err.max()))
    assert y.shape[0] >= 50 and np.median(err) < 0.02 and err.max() < 0.2


# ---- input checks of optimize.nsga2, before any device work
def _tarland():
    from simplyp_b200 import tarland
    return tarland.load("2004-01-01", "2004-12-31", dynamic="y")


_RANGES = {"fc": (100.0, 400.0), "alpha": (0.5, 1.2)}


@pytest.mark.parametrize("ranges, kw, match", [
    ({}, {}, "no free parameters"),
    ({"nope": (0.0, 1.0)}, {}, "unknown parameter"),
    ({"fc": (2.0, 1.0)}, {}, "lo < hi"),
    ({"d_maxE_spr": (1.0, 100.0)}, {}, "integer"),
    ({"sc:f_Ar": (0.0, 1.0)}, {}, "land-use"),
    ({"D_snow_0": (0.0, 1.0)}, {}, "snow_on_device"),
    ({"sc:TDPeff@3": (0.0, 1.0)}, {}, "run-order position"),
    ({"err_phi:TDP": (0.0, 0.9)}, {}, "err_phi"),
    (_RANGES, {"n_population": 7}, "even"),
    (_RANGES, {"n_population": 2}, "even and >= 4"),
    (_RANGES, {"max_generations": 0}, "max_generations"),
    (_RANGES, {"start_generation": -1}, "start_generation"),
    (_RANGES, {"objectives": ["NSE"], "variables": ("Q",)}, "2..16"),
    (_RANGES, {"objectives": [(1, "Q", "NSE")]}, "2..16"),
    (_RANGES, {"objectives": ["NSE", "log_NSE", "r2", "SSE", "nRMSD", "loglik"]}, "2..16"),
    (_RANGES, {"objectives": "NSE"}, "list"),
    (_RANGES, {"objectives": [(1, "Q", "pbias"), (1, "Q", "NSE")]}, "unknown statistic"),
    (_RANGES, {"objectives": [(1, "Q", "KGE"), (1, "Q", "NSE")]}, "unknown statistic"),
    (_RANGES, {"objectives": [(7, "Q", "NSE"), (1, "Q", "SSE")]}, "unknown series"),
    (_RANGES, {"objectives": [(1, "Q", "NSE"), (1, "Q", "NSE")]}, "repeated"),
    (_RANGES, {"objectives": ["NSE", (1, "TP", "NSE")]}, "repeated"),
    (_RANGES, {"crossover": 1.5}, "crossover"),
    (_RANGES, {"crossover": -0.1}, "crossover"),
    (_RANGES, {"mutation": 1.01}, "mutation"),
    (_RANGES, {"mutation": np.nan}, "mutation"),
    (_RANGES, {"eta_c": -1.0}, "eta_c"),
    (_RANGES, {"eta_c": np.inf}, "eta_c"),
    (_RANGES, {"eta_m": np.nan}, "eta_m"),
    (_RANGES, {"initial": np.full((8, 3), 200.0)}, "shape"),
    (_RANGES, {"initial": np.full((8, 2), 0.7)}, "inside the box"),
    (_RANGES, {"initial": {"fc": np.full(8, 200.0), "alpha": np.full(8, np.nan)}}, "inside the box"),
])
def test_nsga2_rejects_bad_input_before_device_work(ranges, kw, match, monkeypatch):
    from simplyp_b200 import engine, optimize

    def no_device(*a, **k):
        raise AssertionError("device work before the input check")
    monkeypatch.setattr(engine, "Engine", no_device)
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    args = dict(n_population=8, max_generations=5)
    args.update(kw)
    n, g = args.pop("n_population"), args.pop("max_generations")
    with pytest.raises(ValueError, match=match):
        optimize.nsga2(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, ranges, n, g, **args)


def test_nsga2_refuses_more_than_half_the_free_memory():
    from simplyp_b200 import optimize

    class SmallDevice:
        def free_bytes(self):
            return 1 << 20

        def __getattr__(self, name):
            raise AssertionError("device work before the memory check: %s" % name)
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    with pytest.raises(ValueError, match="free device memory"):
        optimize.nsga2(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, _RANGES, 1 << 14, 10, engine=SmallDevice())


def test_objective_rows_and_senses():
    from simplyp_b200 import optimize, packing as pk
    labels = [(1, "Q"), (1, "SS"), (1, "TP")]
    rows, lab, sense = optimize._pareto_objectives(["NSE", (1, "SS", "SSE"), "lp"], labels)
    assert lab == [(1, "Q", "NSE"), (1, "SS", "NSE"), (1, "TP", "NSE"), (1, "SS", "SSE"), (None, None, "lp")]
    assert rows.tolist() == [[0, 1], [1, 1], [2, 1], [1, pk.STAT_NAMES.index("SSE")], [0, -1]]
    assert sense.tolist() == [1.0, 1.0, 1.0, -1.0, 1.0]
    assert all(optimize.NSGA2_SENSE[s] == (-1.0 if s in ("SSE", "nRMSD") else 1.0) for s in optimize.DE_OBJECTIVES)


def test_nsga2_entry_points_raise_without_device():
    from simplyp_b200 import _cabi
    lib = _cabi.load()
    if lib.simplyp_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    import ctypes as C
    good = _ns(8, 2)
    ws = _cabi.nsga2_workspace_bytes(good)
    st = _cabi.make_nsga2_state(8, 8, 8, 8, 8, 8, 8, 8, 3, 8, ws)
    bad = [_ns(6 + 1, 2), _ns(2, 2), _ns(8, 2, M=1), _ns(8, 2, crossover=1.5), _ns(8, 2, eta_m=-1.0)]
    bad_sense = _ns(8, 2)
    bad_sense.sense[0] = 0.5
    for ns in bad + [bad_sense]:
        assert lib.simplyp_nsga2_offspring_device(C.byref(ns), C.byref(st), 8, 8, None) == -1
    small = _cabi.make_nsga2_state(8, 8, 8, 8, 8, 8, 8, 8, 3, 8, ws - 1)
    assert lib.simplyp_nsga2_survive_device(C.byref(good), C.byref(small), 8, 8, None) == -1
    assert lib.simplyp_nsga2_survive_device(C.byref(good), C.byref(st), None, 8, None) == -1
    assert lib.simplyp_nsga2_offspring_device(C.byref(good), C.byref(st), 8, 8, None) == -2
    assert lib.simplyp_nsga2_survive_device(C.byref(good), C.byref(st), 8, 8, None) == -2
    assert lib.simplyp_nsga2_init_device(C.byref(good), C.byref(st), 8, 8, None) == -2


@pytest.mark.parametrize("change, match", [("labels", "objectives"), ("bounds", "boxes"), ("names", "optimises")])
def test_nsga2_refuses_to_continue_a_result_of_another_problem(change, match, monkeypatch):
    """A continued run keeps the result's objectives, ranks and crowding without evaluating them again, so a result of
    other objective rows or boxes is refused before any device work."""
    from simplyp_b200 import engine, optimize

    def no_device(*a, **k):
        raise AssertionError("device work before the input check")
    monkeypatch.setattr(engine, "Engine", no_device)
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    N, M = 8, len(optimize.DEFAULT_NSGA2_OBJECTIVES)
    bounds = np.array([_RANGES[k] for k in _RANGES])
    unit = np.full((N, 2), 0.5)
    prev = optimize.ParetoResult(
        names=list(_RANGES), bounds=bounds, labels=list(optimize.DEFAULT_NSGA2_OBJECTIVES),
        population=optimize.scale(unit, bounds), unit=unit, objectives=np.zeros((N, M)), rank=np.zeros(N, np.int32),
        crowding=np.zeros(N), history=np.zeros((1, 2 + M)), generations=5, n_evaluations=N, n_failed=0)
    if change == "labels":
        prev.labels = [(1, "Q", "NSE"), (1, "TP", "NSE"), (1, "SS", "NSE")]
    elif change == "bounds":
        prev.bounds = bounds * 1.5
    else:
        prev.names = ["alpha", "fc"]
    with pytest.raises(ValueError, match=match):
        optimize.nsga2(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, _RANGES, N, 5, initial=prev, start_generation=5)
