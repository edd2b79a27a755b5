"""GPU tier of the Morris screening (simplyp_morris_*_device, sensitivity.elementary_effects): the design rows and the
selection against the host build and NumPy bitwise, the estimators against the fsum reference, Tarland end to end on
the fit statistics and on the simulated series, the 5-reach network, failed members and graph capture."""
import statistics

import numpy as np
import pytest

from tests import morris_reference as ref

pytestmark = pytest.mark.gpu

SEED = 0x5eed_0000_3022
Z95 = statistics.NormalDist().inv_cdf(0.5 + 0.95 / 2)


@pytest.fixture(scope="module")
def eng():
    from simplyp_b200.engine import Engine
    return Engine()


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def _morris(bounds, r, p=4, n_candidates=0, targets=None, n_sc=1, sc_per_member=False, seed=SEED):
    from simplyp_b200 import _cabi
    b = np.asarray(bounds, dtype=np.float64)
    targets = targets or [(_cabi.MCMC_MEMBER, k, 0) for k in range(b.shape[0])]
    return _cabi.make_morris(targets, b[:, 0], b[:, 1], n_sc, r, p, n_candidates, sc_per_member, seed)


# --------------------------------------------------------------------------- 1. design rows
@pytest.mark.parametrize("n_candidates", [0, 40])
def test_design_rows_equal_host_build(eng, n_candidates):
    import torch
    from simplyp_b200 import _cabi, packing as pk
    from tests import morris_host
    bounds = np.array([[100.0, 400.0], [0.0, 0.5], [20.0, 50.0], [20.0, 150.0]])
    targets = [(_cabi.MCMC_MEMBER, pk.MEMBER_INDEX["fc"], 0), (_cabi.MCMC_SC_ALL, pk.SC_INDEX["TDPeff"], 0),
               (_cabi.MCMC_SC_AT, pk.SC_INDEX["A_catch"], 1), (_cabi.MCMC_MEMBER, pk.MEMBER_INDEX["T_g"], 0)]
    r, S, K = 12, 3, 4
    mo = _morris(bounds, r, 6, n_candidates, targets, S, True)
    M = r * (K + 1)
    sel = eng.morris_select(mo) if n_candidates else None
    mem = torch.full((M, pk.NP_MEMBER), -1.0, dtype=torch.float64, device=eng.device)
    sc = torch.full((M, S, pk.NP_SC), -2.0, dtype=torch.float64, device=eng.device)
    for m0, n in ((0, 5), (5, 31), (36, M - 36)):
        eng.morris_design(mo, mem, sc, sel, m0, n)
    selh = sel.cpu().numpy() if sel is not None else None
    want = morris_host.design(mo, 0, M, selh)
    if sel is not None:
        assert np.array_equal(selh, morris_host.select(mo))
    mh, sh = mem.cpu().numpy(), sc.cpu().numpy()
    assert np.array_equal(mh[:, pk.MEMBER_INDEX["fc"]], want[:, 0])
    assert np.array_equal(mh[:, pk.MEMBER_INDEX["T_g"]], want[:, 3])
    for s in range(S):
        assert np.array_equal(sh[:, s, pk.SC_INDEX["TDPeff"]], want[:, 1])
    assert np.array_equal(sh[:, 1, pk.SC_INDEX["A_catch"]], want[:, 2])
    assert np.all(sh[:, [0, 2], pk.SC_INDEX["A_catch"]] == -2.0)
    other = np.ones(pk.NP_MEMBER, bool)
    other[[pk.MEMBER_INDEX["fc"], pk.MEMBER_INDEX["T_g"]]] = False
    assert np.all(mh[:, other] == -1.0)


# --------------------------------------------------------------------------- 2. selection
@pytest.mark.parametrize("nc, r, K, p", [(1000, 20, 5, 4), (1000, 10, 18, 4), (4096, 50, 4, 4), (300, 8, 64, 16)])
def test_selection_equals_host_and_numpy(eng, nc, r, K, p):
    from simplyp_b200 import _cabi
    from tests import morris_host
    # the selection reads no target; error-model targets fit any K
    mo = _morris([(0.0, 1.0)] * K, r, p, nc, targets=[(_cabi.MCMC_ERROR_MODEL, k % 6, 0) for k in range(K)])
    got = eng.morris_select(mo).cpu().numpy()
    assert np.array_equal(got, morris_host.select(mo))
    if nc * nc * (K + 1) ** 2 * K <= 4096 * 4096 * 25 * 4:           # the NumPy all-pairs pass at this size
        want, D = ref.select(ref.levels(SEED, K, p, nc), r)
        assert np.array_equal(got, want)
        assert ref.spread(D, got) > ref.spread(D, range(r))


# --------------------------------------------------------------------------- 3. estimators
def _rows(lev, bounds, p, seed=5):
    X = ref.design_values(bounds, lev, p)
    rng = np.random.default_rng(seed)
    K = X.shape[1]
    # no parameter enters linearly: a constant |EE| has a bootstrap spread of rounding noise, which no relative
    # tolerance compares; an unread parameter has EE = 0 exactly
    return np.stack([(X ** 2) @ rng.normal(size=K) + X[:, 0] * X[:, 2], X[:, 0] * X[:, 1] + np.sin(3 * X[:, 2]),
                     1e3 + np.exp(X[:, -1]) * X[:, 1]])


def test_estimators_equal_fsum_reference(eng):
    from tests import morris_host
    K, r, p, n_boot = 5, 300, 6, 60
    bounds = np.array([[0.0, 1.0], [-2.0, 2.0], [0.0, 3.0], [1.0, 5.0], [0.0, 0.1]])
    mo = _morris(bounds, r, p, 1000)
    sel = eng.morris_select(mo)
    lev = ref.levels(SEED, K, p, 1000)[sel.cpu().numpy()]
    y = _rows(lev, bounds, p)
    y[1, 7 * (K + 1) + 2] = np.nan                             # drops trajectory 7 of row 1
    y[2, 11 * (K + 1)] = np.inf
    y[2, 12 * (K + 1) + K] = -np.inf
    got = {k: v.cpu().numpy() for k, v in eng.morris_effects(mo, eng.to_device(y), n_boot, Z95, sel).items()}
    assert list(got["n_used"]) == [r, r - 1, r - 2]
    for i in range(3):
        want = ref.effects(y[i], lev, p)
        for k in ("mu", "mu_star", "sigma"):
            assert np.allclose(got[k][i], want[k], rtol=0, atol=1e-12), k
        picks = morris_host.picks(SEED, n_boot, want["n"])
        assert np.allclose(got["mu_star_conf"][i], ref.bootstrap_conf(y[i], lev, p, picks, Z95), rtol=1e-10, atol=0)
    # too few used trajectories, no bootstrap
    y[0, :] = np.nan
    y[0, :K + 1] = 1.0
    got = {k: v.cpu().numpy() for k, v in eng.morris_effects(mo, eng.to_device(y), 0, Z95, sel).items()}
    assert got["n_used"][0] == 1 and np.all(np.isnan(got["mu_star"][0])) and np.all(np.isnan(got["mu_star_conf"]))
    assert np.all(np.isfinite(got["mu_star"][1:]))


# --------------------------------------------------------------------------- 4. Tarland end to end, objectives
def _tarland(years=("2004-01-01", "2004-12-31")):
    from simplyp_b200 import tarland
    return tarland.load(years[0], years[1], dynamic="y")


OBJ = ["NSE", "log_NSE", "loglik", "r2", "pbias", "nRMSD", "SSE", "lp"]


@pytest.fixture(scope="module")
def tarland_obj(eng):
    from simplyp_b200 import ensemble as ens, sensitivity
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    runs = [sensitivity.elementary_effects(met, p_struc, p_SU, p_LU, p_SC, p, dyn, ens.TARLAND_RANGES, 40,
                                           obs_dict=obs, objectives=OBJ, n_candidates=200, n_boot=200, engine=eng)
            for _ in range(2)]
    return runs, (p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs)


def test_tarland_statistics_equal_calibrate_ensemble(eng, tarland_obj):
    import torch
    from simplyp_b200 import _cabi, ensemble as ens, mcmc, packing as pk, sensitivity
    (r, _), (p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs) = tarland_obj
    names, targets, bounds = mcmc._check_priors(ens.TARLAND_RANGES, 1, False)
    K = len(names)
    mo = _cabi.make_morris(targets, bounds[:, 0], bounds[:, 1], 1, 40, 4, 200, True, sensitivity.DEFAULT_MORRIS_SEED)
    X = ref.design_values(bounds, ref.levels(sensitivity.DEFAULT_MORRIS_SEED, K, 4, 200)[r.selected], 4)
    samples = {n: X[:, k] for k, n in enumerate(names)}
    stats, labels, diag = ens.calibrate_ensemble(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, samples, engine=eng)
    assert np.all(diag.cpu().numpy()[:, :, 3] == 0)
    rows = [(v, pk.STAT_NAMES.index(o)) for v in range(len(labels)) for o in OBJ if o != "lp"] + [(0, -1)]
    y = torch.empty((len(rows), X.shape[0]), dtype=torch.float64, device=eng.device)
    eng.sobol_outputs(stats, diag, eng.to_device(np.asarray(rows, dtype=np.int32)), y)
    sel = eng.to_device(r.selected.astype(np.int32))
    res = eng.morris_effects(mo, y, 200, Z95, sel)
    for k in ("mu", "mu_star", "sigma", "mu_star_conf", "n_used"):
        assert _same(res[k].cpu().numpy(), getattr(r, k)), k
    assert [lab[2] for lab in r.labels] == [o for _ in labels for o in OBJ if o != "lp"] + ["lp"]


def test_tarland_runs_repeat_bitwise_and_ignore_unread_error_scales(tarland_obj):
    (r, r2), _ = tarland_obj
    for k in ("mu", "mu_star", "sigma", "mu_star_conf", "n_used", "selected"):
        assert _same(getattr(r, k), getattr(r2, k)), k
    col = {n: k for k, n in enumerate(r.names)}
    for i, (sc, var, stat) in enumerate(r.labels):
        zero = []
        if stat in ("NSE", "log_NSE", "r2", "pbias", "nRMSD", "SSE"):
            zero = ["err_m:Q", "err_m:TDP"]
        elif stat == "loglik":
            zero = ["err_m:TDP"] if var == "Q" else ["err_m:Q"]
        for n in zero:
            assert r.mu_star[i, col[n]] == 0.0 and r.mu[i, col[n]] == 0.0, (r.labels[i], n)
    # no member fails, but a statistic can be non-finite at a face of the box (the levels include 0 and 1)
    assert r.n_failed == 0 and np.all(r.n_used <= 40) and np.all(r.n_used >= 30) and r.n_used[0] == 40
    kept = r.screen(0.1)
    assert kept and list(kept) == [n for n in r.names if n in kept]
    assert list(r.table(0).columns) == ["mu", "mu_star", "sigma", "mu_star_conf"]


# --------------------------------------------------------------------------- 5. series mode
def test_series_mode_chunking_does_not_change_the_result(eng):
    from simplyp_b200 import ensemble as ens, sensitivity
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    kw = dict(series=[(1, "Q"), (1, "TDP")], n_boot=50, engine=eng)
    a = sensitivity.elementary_effects(met, p_struc, p_SU, p_LU, p_SC, p, dyn, ens.TARLAND_RANGES, 30, **kw)
    b = sensitivity.elementary_effects(met, p_struc, p_SU, p_LU, p_SC, p, dyn, ens.TARLAND_RANGES, 30,
                                       members_per_chunk=77, **kw)
    for k in ("mu", "mu_star", "sigma", "mu_star_conf", "n_used"):
        assert _same(getattr(a, k), getattr(b, k)), k
    D = len(met)
    assert len(a.labels) == 2 * D and a.labels[D] == (1, "TDP", met.index[0])
    col = {n: k for k, n in enumerate(a.names)}
    for n in ("err_m:Q", "err_m:TDP"):
        assert np.all(a.mu_star[:, col[n]] == 0.0), n


def test_series_mode_failed_members_drop_their_trajectories(eng, monkeypatch):
    from simplyp_b200 import ensemble as ens, model, packing as pk, sensitivity
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland(("2004-01-01", "2004-03-31"))
    ranges = {"T_s:A": (1.0, 8.0), "E_M": (300.0, 3000.0), "fc": (100.0, 400.0)}
    make = model.make_options

    def few_steps(*a, **k):
        o = make(*a, **k)
        o.max_steps_per_day = 4
        return o
    monkeypatch.setattr(model, "make_options", few_steps)
    r_traj, K = 64, 3
    r = sensitivity.elementary_effects(met, p_struc, p_SU, p_LU, p_SC, p, dyn, ranges, r_traj, series=[(1, "Q")],
                                       n_boot=10, engine=eng)
    names = list(ranges)
    X = ref.design_values(np.array([ranges[n] for n in names]),
                          ref.levels(sensitivity.DEFAULT_MORRIS_SEED, K, 4, r_traj), 4)
    topo = pk.build_topology(p_struc, p["SC_list"])
    member, sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids),
                                  {n: X[:, k] for k, n in enumerate(names)})
    opt = few_steps(p_SU, p, dyn, topo)
    _, diag = eng.run(eng.to_device(pk.forcing_matrix(met)), eng.to_device(member), eng.to_device(sc),
                      topo.parent_offsets, topo.parent_ids, opt)
    failed = np.any(diag.cpu().numpy()[:, :, 3] != 0, axis=1)
    assert r.n_failed == failed.sum() > 0
    n_ok = r_traj - np.any(failed.reshape(r_traj, K + 1), axis=1).sum()
    assert np.all(r.n_used == n_ok)


# --------------------------------------------------------------------------- 6. the 5-reach network
def test_network5_with_per_member_sc_targets(eng):
    from simplyp_b200 import packing as pk, sensitivity
    from tests.golden.networks import network5_inputs
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland(("2004-01-01", "2004-06-30"))
    p, p_LU, p_SC, p_struc = network5_inputs(p, p_LU, p_SC, p_struc)
    pk.validate_land_use(p_SC, p["SC_list"])
    ranges = {"fc": (100.0, 400.0), "sc:A_catch@2": (20.0, 50.0), "sc:TDPeff": (0.0, 0.5), "err_m:Q": (0.05, 1.0)}
    topo = pk.build_topology(p_struc, p["SC_list"])
    reach = topo.sc_ids[2]
    r = sensitivity.elementary_effects(met, p_struc, p_SU, p_LU, p_SC, p, dyn, ranges, 16,
                                       series=[(reach, "Q"), (topo.sc_ids[0], "Q")], n_candidates=64, n_boot=20,
                                       engine=eng)
    D = len(met)
    col = {n: k for k, n in enumerate(r.names)}
    assert np.all(r.mu_star[:, col["err_m:Q"]] == 0.0)
    assert np.nanmax(r.mu_star[:D, col["sc:A_catch@2"]]) > 0.0
    if 2 not in [int(x) for x in np.asarray(topo.parent_ids)]:
        assert np.all(r.mu_star[D:, col["sc:A_catch@2"]] == 0.0)
    assert "sc:A_catch@2" in r.screen(0.01, rows=list(range(D)))


# --------------------------------------------------------------------------- 7. graph capture
def test_design_calibrate_outputs_and_effects_capture_into_a_graph(eng):
    import torch
    from simplyp_b200 import _cabi, ensemble as ens, mcmc, model as spm, packing as pk
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland(("2004-01-01", "2004-03-31"))
    names, targets, bounds = mcmc._check_priors(ens.TARLAND_RANGES, 1, False)
    K, r = len(names), 16
    mo = _cabi.make_morris(targets, bounds[:, 0], bounds[:, 1], 1, r, 4, 100, True, SEED)
    topo = pk.build_topology(p_struc, p["SC_list"])
    opt = spm.make_options(p_SU, p, dyn, topo)
    M = r * (K + 1)
    base_m, base_sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), {})
    mem = eng.to_device(base_m).expand(M, pk.NP_MEMBER).contiguous()
    sc = eng.to_device(base_sc).expand(M, 1, pk.NP_SC).contiguous()
    forc = eng.to_device(pk.forcing_matrix(met))
    o, odesc, labels = pk.obs_arrays(obs, topo, met.index, ("Q", "TDP"))
    d_obs, d_odesc = eng.to_device(o), eng.to_device(odesc)
    rows = eng.to_device(np.array([[0, 1], [1, 1], [0, -1]], dtype=np.int32))
    stats = torch.empty((M, len(labels), pk.NSTAT), dtype=torch.float64, device=eng.device)
    diag = torch.zeros((M, 1, pk.NDIAG), dtype=torch.int64, device=eng.device)
    y = torch.empty((3, M), dtype=torch.float64, device=eng.device)
    sel = eng.morris_select(mo)

    def step(out=None):
        diag.zero_()
        eng.morris_design(mo, mem, sc, sel)
        eng.calibrate(forc, mem, sc, topo.parent_offsets, topo.parent_ids, d_obs, d_odesc, opt, stats=stats,
                      diag=diag)
        eng.sobol_outputs(stats, diag, rows, y)
        return eng.morris_effects(mo, y, 40, Z95, sel, out=out)
    direct = {k: v.clone() for k, v in step().items()}
    torch.cuda.synchronize()
    out = {k: torch.full_like(v, -5) for k, v in direct.items()}
    g = eng.capture(lambda: step(out))
    for v in out.values():
        v.fill_(-5)
    y.zero_()
    g.replay()
    torch.cuda.synchronize()
    for k in direct:
        assert _same(out[k].cpu().numpy(), direct[k].cpu().numpy()), k
    assert np.all(np.isfinite(direct["mu_star"].cpu().numpy()))
