"""GPU tier of NSGA-II (simplyp_nsga2_*_device, simplyp_b200.optimize.nsga2): the kernels in lock-step with the NumPy
restatement, a set with one point per front, graph replay against a hand-driven loop, continuation, the box, Tarland
end to end, a twin experiment and the AR(1) error model."""
import numpy as np
import pandas as pd
import pytest

from tests import nsga2_reference as ref

pytestmark = pytest.mark.gpu

FREE = {"fc": (100.0, 400.0), "T_g": (20.0, 150.0), "alpha": (0.5, 1.2)}
Q2 = [(1, "Q", "NSE"), (1, "Q", "log_NSE")]


@pytest.fixture(scope="module")
def cabi():
    from simplyp_b200 import _cabi
    _cabi.require_device()
    return _cabi


def _tarland():
    from simplyp_b200 import tarland
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(dynamic="y")
    return met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs


class _Kernels:
    """The three entry points on hand-made buffers, for analytic objectives injected as y [M][N] and diag."""

    def __init__(self, cabi, N, K, M, sense, u0, seed):
        import torch
        from simplyp_b200.engine import Engine
        self.eng = eng = Engine()
        dev = eng.device
        self.t = t = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)
        self.N, self.K, self.M, self.sense = N, K, M, np.asarray(sense, dtype=np.float64)
        self.pop, self.obj = t(u0), t(np.full((N, M), np.nan))
        self.rank, self.crowd = t(np.zeros(N), torch.int32), t(np.zeros(N))
        self.kids, self.counters = t(np.zeros((N, K))), t([0, 0], torch.int64)
        self.history = t(np.full((200, 2 + M), np.nan))
        self.mem, self.sc = t(np.zeros((N, 40))), t(np.zeros((1, 1, 16)))
        self.diag = torch.zeros((N, 1, 4), dtype=torch.int64, device=dev)
        self.ns = cabi.make_nsga2(N, [(cabi.MCMC_MEMBER, k, 0) for k in range(K)], np.zeros(K), np.ones(K), 1, sense,
                                  seed=seed)
        ws = cabi.nsga2_workspace_bytes(self.ns)
        self.ws = torch.empty(ws, dtype=torch.uint8, device=dev)
        c = self.counters
        self.st = cabi.make_nsga2_state(self.pop.data_ptr(), self.obj.data_ptr(), self.rank.data_ptr(),
                                        self.crowd.data_ptr(), self.kids.data_ptr(), c[0].data_ptr(), c[1].data_ptr(),
                                        self.history.data_ptr(), 200, self.ws.data_ptr(), ws)

    def inject(self, y, status):
        import torch
        self.diag.zero_()
        self.diag[:, 0, 3] = self.t(np.asarray(status, dtype=np.int64) * 4, torch.int64)
        return self.t(y)

    def state(self):
        return (self.pop.cpu().numpy(), self.obj.cpu().numpy(), self.rank.cpu().numpy().astype(np.int64),
                self.crowd.cpu().numpy())


def _zdt_rows(x):
    """ZDT1 (minimised), NaN where x1 > 0.85, a status bit where x2 < 0.03."""
    y = ref.zdt(x, 1)
    y[1, x[:, 1] > 0.85] = np.nan
    return y, x[:, 2] < 0.03


@pytest.mark.parametrize("N, n", [(96, 100), (1000, 25)])
def test_kernels_in_lock_step_with_the_reference(cabi, N, n):
    """N = 96: the 2N points fit one block.  N = 1,000: 2N = 2,000 points run the survival over eight blocks, with a
    partial last tile, two 1,024-point chunks of the survivors' scan, and several fronts peeled across the grid."""
    from simplyp_b200 import optimize
    K, M, seed = 6, 2, 0xfeed_0000_5a2a
    sense = [-1.0, -1.0]
    u0 = optimize.latin_hypercube_unit(N, K, 5)
    k = _Kernels(cabi, N, K, M, sense, u0, seed)
    y, st = _zdt_rows(u0)
    k.eng.nsga2_init(k.ns, k.st, k.inject(y, st), k.diag)
    pop, obj, rank, crowd, h = ref.survive(ref.orient(y, st, sense), u0, sense, N)
    got = k.state()
    for a, b in zip(got, (pop, obj, rank, crowd)):
        assert np.array_equal(a, b, equal_nan=True)
    n_failed = int(np.isnan(ref.orient(y, st, sense)[:, 0]).sum())
    worst = 0.0
    for g in range(n):
        k.eng.nsga2_offspring(k.ns, k.st, k.mem, k.sc)
        kids = k.kids.cpu().numpy()
        assert np.array_equal(k.mem[:, :K].cpu().numpy(), optimize.scale(kids, np.array([(0.0, 1.0)] * K)))
        want, _ = ref.offspring(pop, rank, crowd, g, seed, 0.9, 1.0 / K, 15.0, 20.0)
        worst = max(worst, float(np.max(np.abs(kids - want))))
        assert np.max(np.abs(kids - want)) <= ref.OFFSPRING_ULP * 2.0 ** -52, g
        y, st = _zdt_rows(kids)
        k.eng.nsga2_survive(k.ns, k.st, k.inject(y, st), k.diag)
        fk = ref.orient(y, st, sense)
        n_failed += int(np.isnan(fk[:, 0]).sum())
        f = np.concatenate([np.asarray(sense)[None, :] * obj, fk])
        pop, obj, rank, crowd, h = ref.survive(f, np.concatenate([pop, kids]), sense, N)
        got = k.state()
        for name, a, b in zip(("population", "objectives", "rank", "crowding"), got, (pop, obj, rank, crowd)):
            assert np.array_equal(a, b, equal_nan=True), (g, name)
        assert np.array_equal(k.history[g + 1].cpu().numpy(), h, equal_nan=True), g
        pop, obj, rank, crowd = got          # the next generation starts from the device's own state
    gen, nf = k.counters.cpu().numpy().tolist()
    fronts = k.history[:n + 1, 1].cpu().numpy()
    print("lock-step N = %d: largest offspring difference %.3g (bound %.3g), n_failed %d, fronts ranked %d..%d"
          % (N, worst, ref.OFFSPRING_ULP * 2.0 ** -52, nf, fronts.min(), fronts.max()))
    assert gen == n and nf == n_failed > 0 and fronts.max() > 1


@pytest.mark.parametrize("N", [256, 1000])
def test_identical_objectives_give_one_point_per_front(cabi, N):
    """M = 2 with both objectives equal and all values distinct: N fronts of one point each (N = 1,000: four blocks
    meeting at 1,000 grid barriers)."""
    K = 2
    rng = np.random.default_rng(9)
    u0 = rng.uniform(size=(N, K))
    k = _Kernels(cabi, N, K, 2, [1.0, 1.0], u0, 3)
    v = rng.permutation(N).astype(np.float64)
    y = np.stack([v, v])
    k.eng.nsga2_init(k.ns, k.st, k.inject(y, np.zeros(N, bool)), k.diag)
    _, obj, rank, crowd = k.state()
    assert np.array_equal(rank, (N - 1 - v).astype(np.int64))
    assert np.all(crowd == np.inf) and k.history[0, 1].item() == N
    want = ref.survive(ref.orient(y, np.zeros(N, bool), [1.0, 1.0]), u0, [1.0, 1.0], N)
    assert np.array_equal(rank, want[2]) and np.array_equal(obj, want[1])


def _run(**kw):
    from simplyp_b200 import optimize
    return optimize.nsga2(*_tarland(), FREE, kw.pop("N", 32), kw.pop("G", 12), objectives=kw.pop("objectives", Q2),
                          variables=("Q",), **kw)


def _equal(a, b):
    for f in ("unit", "population", "objectives", "rank", "crowding", "history"):
        assert np.array_equal(getattr(a, f), getattr(b, f), equal_nan=True), f
    for f in ("generations", "n_evaluations", "n_failed"):
        assert getattr(a, f) == getattr(b, f), f


def test_graph_replay_equals_hand_driven_loop(cabi):
    from simplyp_b200 import optimize
    o = optimize._Nsga2(*_tarland(), FREE, 32, 12, objectives=Q2, variables=("Q",), seed=3)
    o.evaluate_initial()
    for _ in range(12):
        o.generation_step()
    _equal(o.result(), _run(seed=3))


def test_continuation_equals_one_run(cabi):
    one = _run(G=60, seed=9)
    a = _run(G=30, seed=9)
    b = _run(G=30, seed=9, initial=a, start_generation=a.generations)
    assert b.generations == 60 and b.n_evaluations == 30 * 32
    for f in ("unit", "population", "objectives", "rank", "crowding"):
        assert np.array_equal(getattr(b, f), getattr(one, f), equal_nan=True), f
    assert np.array_equal(np.concatenate([a.history, b.history[1:]]), one.history, equal_nan=True)
    assert a.n_failed + b.n_failed == one.n_failed


@pytest.mark.parametrize("kind", ["tarland", "network5"])
def test_rows_handed_to_the_integrator_lie_inside_the_box(cabi, kind):
    from simplyp_b200 import optimize, packing as pk
    met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs = _tarland()
    ranges = {"fc": (280.0, 300.0), "T_g": (60.0, 70.0), "sc:TDPeff": (0.1, 0.2)}
    objectives = [(1, "Q", "NSE"), (1, "TDP", "NSE")]
    if kind == "network5":
        from tests.golden.networks import network5_inputs
        p, p_LU, p_SC, p_struc = network5_inputs(p, p_LU, p_SC, p_struc)
        pk.validate_land_use(p_SC, p["SC_list"])
        obs = {5: obs[1]}
        ranges = {"fc": (280.0, 300.0), "T_g": (60.0, 70.0), "sc:TDPeff@2": (0.0, 0.5)}
        objectives = [(5, "Q", "NSE"), (5, "TDP", "NSE")]
    names = list(ranges)
    b = np.array([ranges[k] for k in names])
    o = optimize._Nsga2(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, ranges, 16, 10, seed=4, objectives=objectives,
                        variables=("Q", "TDP"), mutation=1.0, eta_m=0.0, eta_c=0.0)
    o.evaluate_initial()
    S = o.S
    for _ in range(10):
        o.offspring_step()
        mem, sc = o.d_mem.cpu().numpy(), o.d_sc.cpu().numpy()
        kids = o.offspring.cpu().numpy()
        assert np.all((kids >= 0.0) & (kids <= 1.0))
        want = optimize.scale(kids, b)
        for k, n in enumerate(names):
            if n.startswith("sc:"):
                row, _, at = n[3:].partition("@")
                cols = sc[:, int(at), pk.SC_INDEX[row]][:, None] if at else sc[:, :, pk.SC_INDEX[row]]
            else:
                cols = mem[:, pk.MEMBER_INDEX[n]][:, None]
            assert cols.shape[1] in (1, S)
            assert np.all(cols == want[:, k:k + 1]), n
            assert np.all((cols >= b[k, 0]) & (cols <= b[k, 1])), n
        o.evaluate()
        o.survive()
    r = o.result()
    assert np.all((r.population >= b[:, 0]) & (r.population <= b[:, 1]))


def _dominates(a, b):
    return np.all(a >= b) and np.any(a > b)


def test_tarland_end_to_end(cabi):
    """K = 18 on Tarland 2004, objectives NSE(Q), NSE(TDP), log_NSE(Q): the objectives equal a fresh evaluation
    through calibrate_ensemble bitwise, the first front is mutually non-dominated, the ideal point never gets worse,
    two runs are bitwise equal, and the first front feeds predictive_bands."""
    from simplyp_b200 import ensemble as ens, optimize, packing as pk
    args = _tarland()
    objectives = [(1, "Q", "NSE"), (1, "TDP", "NSE"), (1, "Q", "log_NSE")]
    kw = dict(objectives=objectives, variables=("Q", "TDP"), seed=12)
    r = optimize.nsga2(*args, ens.TARLAND_RANGES, 64, 20, **kw)
    _equal(r, optimize.nsga2(*args, ens.TARLAND_RANGES, 64, 20, **kw))
    assert len(r.names) == 18 and r.history.shape == (21, 5) and r.n_evaluations == 64 * 21
    assert np.all(np.diff(r.history[:, 2:], axis=0) >= 0)
    samples = {k: r.population[:, j] for j, k in enumerate(r.names)}
    stats, labels, diag = ens.calibrate_ensemble(*args, samples, variables=("Q", "TDP"))
    s, failed = stats.cpu().numpy(), diag.cpu().numpy()[..., 3].any(axis=1)
    for m, (sc, var, stat) in enumerate(r.labels):
        want = np.where(failed, np.nan, s[:, labels.index((sc, var)), pk.STAT_NAMES.index(stat)])
        bad = ~np.all(np.isfinite(np.stack([s[:, labels.index((c, v)), pk.STAT_NAMES.index(t)]
                                            for c, v, t in r.labels])), axis=0)
        want[bad] = np.nan
        assert np.array_equal(r.objectives[:, m], want, equal_nan=True), r.labels[m]
    front = r.objectives[r.rank == 0]
    assert front.shape[0] >= 2
    for i in range(front.shape[0]):
        for j in range(front.shape[0]):
            assert not _dominates(front[j], front[i])
    df = r.front()
    assert list(df.columns) == r.names + ["NSE(Q@1)", "NSE(TDP@1)", "log_NSE(Q@1)"] and len(df) == front.shape[0]
    fs = r.front_samples()
    met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs = args
    bands = ens.predictive_bands(met, p_struc, p_SU, p_LU, p_SC, p, dyn, fs, [(1, "TP")])
    assert bands is not None


def test_twin_experiment_finds_the_truth(cabi):
    """Noise-free Q of a known member: NSE(Q) and log_NSE(Q) over fc, T_g and alpha both get close to 1."""
    from simplyp_b200 import ensemble as ens, model as spm, optimize, packing as pk, tarland
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, _ = tarland.load(dynamic="y")
    topo = pk.build_topology(p_struc, p["SC_list"])
    opt = spm.make_options(p_SU, p, dyn, topo)
    out, diag = cabi.run_host(pk.forcing_matrix(met), pk.member_vector(p, p_LU)[None], pk.sc_matrix(p_SC, topo.sc_ids),
                              topo.parent_offsets, topo.parent_ids, opt)
    q = out[0, 0, :, pk.RAW_COLS.index("Qr")] * float(p_SC.loc["A_catch", 1]) * 1000 / 86400
    obs = {1: pd.DataFrame({"Q": q}, index=met.index)}
    ranges = {k: ens.TARLAND_RANGES[k] for k in ("fc", "T_g", "alpha")}
    r = optimize.nsga2(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, ranges, 64, 80, objectives=Q2,
                       variables=("Q",), seed=77)
    best = r.history[-1, 2:]
    print("twin: best NSE %.9f, best log_NSE %.9f, first front %d" % (best[0], best[1], r.history[-1, 0]))
    assert np.all(best >= 0.999)


def test_ar1_error_model_range(cabi):
    """An err_phi:Q range is optimised with the model parameters, as differential evolution does: the objectives
    equal a fresh calibrate_ensemble of the population bitwise."""
    from simplyp_b200 import ensemble as ens, optimize, packing as pk
    args = _tarland()
    ranges = dict(FREE, **{"err_phi:Q": (0.0, 0.95)})
    r = optimize.nsga2(*args, ranges, 32, 8, objectives=[(1, "Q", "loglik"), (1, "Q", "NSE")], variables=("Q",),
                       seed=5)
    assert np.all((r.population[:, 3] >= 0.0) & (r.population[:, 3] <= 0.95))
    samples = {k: r.population[:, j] for j, k in enumerate(r.names)}
    stats, labels, diag = ens.calibrate_ensemble(*args, samples, variables=("Q",))
    s = stats.cpu().numpy()
    for m, (sc, var, stat) in enumerate(r.labels):
        want = s[:, labels.index((sc, var)), pk.STAT_NAMES.index(stat)]
        ok = np.isfinite(r.objectives[:, m])
        assert ok.sum() > 0 and np.array_equal(r.objectives[ok, m], want[ok])
