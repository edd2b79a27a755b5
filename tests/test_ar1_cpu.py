"""CPU tier of the AR(1) error model of the log-likelihood: the sequential factorisation (tests/ar1_reference.py)
against the dense multivariate normal and the iid reference, the host build of simplyp_ar1.cuh (tests/ar1_host.cpp)
against the factorisation on every edge, the sampler's row writes of an error-model target, and the input checks of
every public entry point that takes ``err_phi:<kind>``."""
import ctypes as C
import math

import numpy as np
import pytest

from tests import ar1_reference as ref
from tests import fit_stats_reference as fsr

PHIS = [-0.4, 0.0, 0.5, 0.95, 0.999]


def _series(rng, D, frac, m=0.3):
    """Simulated values s [D] > 0 and observations o [D] (NaN on unobserved days, irregular gaps)."""
    s = rng.uniform(0.2, 3.0, D)
    o = s * (1.0 + m * rng.standard_normal(D))
    o[rng.random(D) >= frac] = np.nan
    return o, s


def _rel(a, b):
    return abs(a - b) / abs(b)


@pytest.mark.parametrize("phi", PHIS)
@pytest.mark.parametrize("seed", range(4))
def test_sequential_factorisation_equals_dense_density(phi, seed):
    rng = np.random.default_rng(1000 + seed)
    D = int(rng.integers(20, 1200))
    o, s = _series(rng, D, rng.uniform(0.05, 0.9))
    while np.count_nonzero(~np.isnan(o)) > 500:
        o[rng.integers(0, D)] = np.nan
    m = rng.uniform(0.05, 1.0)
    seq, dense = ref.loglik_sequential(o, s, m, phi), ref.loglik_dense(o, s, m, phi)
    assert math.isfinite(seq)
    assert _rel(seq, dense) <= 1e-10, (seq, dense)


@pytest.mark.parametrize("seed", range(4))
def test_phi_zero_is_the_iid_gaussian(seed):
    rng = np.random.default_rng(2000 + seed)
    o, s = _series(rng, 366, 0.6)
    m = 0.25
    row, _bound = fsr.fit_stats(o, s, m)
    assert _rel(ref.loglik_sequential(o, s, m, 0.0), row[fsr.ST_LOGLIK]) <= 1e-13


@pytest.mark.parametrize("phi", PHIS + [-0.95])
@pytest.mark.parametrize("seed", range(6))
def test_host_build_matches_the_reference_per_row(phi, seed):
    from tests import ar1_host
    rng = np.random.default_rng(3000 + seed)
    D = [1, 31, 32, 33, 366, 1000][seed]
    o, s = _series(rng, D, [1.0, 0.3, 0.9, 0.05, 0.5, 0.2][seed])
    if np.all(np.isnan(o)):
        o[D // 2] = s[D // 2] * 1.1
    got, want = ar1_host.row(o, s, 0.4, phi), ref.loglik_sequential(o, s, 0.4, phi)
    assert _rel(got, want) <= 1e-12, (got, want)


def test_host_build_first_observation_and_long_gaps():
    from tests import ar1_host
    D = 700
    s = np.linspace(0.5, 2.0, D)
    o = np.full(D, np.nan)
    for d in (0, 200, 201, 365, 366, 367, 699):          # the first day, gaps across many chunks, runs of days
        o[d] = s[d] * 1.2
    for phi in PHIS:
        got, want = ar1_host.row(o, s, 0.3, phi), ref.loglik_sequential(o, s, 0.3, phi)
        assert _rel(got, want) <= 1e-12
    # one observation: the first term alone, whatever phi
    one = np.full(D, np.nan)
    one[450] = 1.0
    assert _rel(ar1_host.row(one, s, 0.3, 0.9), ar1_host.row(one, s, 0.3, 0.0)) <= 1e-15


@pytest.mark.parametrize("case", ["s_zero", "s_negative", "s_nan", "m_zero", "phi_one", "phi_minus_one", "phi_big",
                                  "phi_nan"])
def test_host_build_gives_minus_inf_where_the_density_is_undefined(case):
    from tests import ar1_host
    rng = np.random.default_rng(4000)
    o, s = _series(rng, 100, 0.5)
    days = np.flatnonzero(~np.isnan(o))
    m, phi = 0.3, 0.5
    if case == "s_zero":
        s[days[3]] = 0.0
    elif case == "s_negative":
        s[days[-1]] = -1.0
    elif case == "s_nan":
        s[days[0]] = np.nan
    elif case == "m_zero":
        m = 0.0
    else:
        phi = {"phi_one": 1.0, "phi_minus_one": -1.0, "phi_big": 1.5, "phi_nan": np.nan}[case]
    assert ar1_host.row(o, s, m, phi) == -math.inf
    assert ref.loglik_sequential(o, s, m, phi) == -math.inf


def test_host_build_gives_zero_without_observed_days():
    from tests import ar1_host
    s = np.ones(100)
    assert ar1_host.row(np.full(100, np.nan), s, 0.3, 0.7) == 0.0
    assert ar1_host.row(np.zeros(0), np.zeros(0), 0.3, 0.7) == 0.0
    assert ref.loglik_sequential(np.full(100, np.nan), s, 0.3, 0.7) == 0.0


def test_an_unobserved_day_is_ignored_whatever_its_simulated_value():
    from tests import ar1_host
    rng = np.random.default_rng(5000)
    o, s = _series(rng, 200, 0.5)
    s2 = s.copy()
    s2[np.isnan(o)] = -1.0                               # sim_obs holds NaN there; any value must be unused
    assert ar1_host.row(o, s, 0.3, 0.8) == ar1_host.row(o, s2, 0.3, 0.8)


# ---------------------------------------------------------------------------------------------- sampler row writes
def _mcmc(kinds, W=8):
    from simplyp_b200 import _cabi
    targets = [(k, i, 0) for k, i in kinds]
    lo = np.array([0.0, 1.0, -0.5, 10.0])[:len(kinds)]
    hi = lo + np.array([1.0, 2.0, 1.0, 5.0])[:len(kinds)]
    return _cabi.make_mcmc(W, targets, lo, hi, n_sc=2, n_obs_series=2, sc_per_member=True, seed=77)


def test_error_model_target_leaves_the_parameter_rows_and_the_other_proposals_unchanged():
    from simplyp_b200 import _cabi
    from simplyp_b200 import packing as pk
    from tests import ar1_host, mcmc_host
    plain = [(_cabi.MCMC_MEMBER, pk.MEMBER_INDEX["fc"]), (_cabi.MCMC_SC_ALL, pk.SC_INDEX["TDPeff"]),
             (_cabi.MCMC_MEMBER, pk.MEMBER_INDEX["T_g"]), (_cabi.MCMC_SC_AT, pk.SC_INDEX["S_reach"])]
    with_phi = list(plain)
    with_phi[2] = (_cabi.MCMC_ERROR_MODEL, pk.VAR_INDEX["TDP"])
    mc_a, mc_b = _mcmc(plain), _mcmc(with_phi)
    rng = np.random.default_rng(6000)
    walkers = np.stack([rng.uniform(mc_a.param[k].lo, mc_a.param[k].hi, 8) for k in range(4)], axis=1)
    for t, half in ((0, 0), (3, 1), (1 << 33, 0)):
        pa, za, oa = mcmc_host.propose(mc_a, walkers, t, half)
        pb, zb, ob = mcmc_host.propose(mc_b, walkers, t, half)
        assert np.array_equal(pa, pb) and np.array_equal(za, zb) and np.array_equal(oa, ob)
        for k in range(4):
            mrow_a = np.arange(pk.NP_MEMBER, dtype=np.float64)
            srow_a = np.arange(2 * pk.NP_SC, dtype=np.float64).reshape(2, pk.NP_SC)
            mrow_b, srow_b = mrow_a.copy(), srow_a.copy()
            ar1_host.write_targets(mc_a.param, 2, pa[k], mrow_a, srow_a)
            ar1_host.write_targets(mc_b.param, 2, pb[k], mrow_b, srow_b)
            # the error-model target is in no row; every other column is written as before
            assert mrow_b[pk.MEMBER_INDEX["T_g"]] == pk.MEMBER_INDEX["T_g"]
            mrow_b[pk.MEMBER_INDEX["T_g"]] = mrow_a[pk.MEMBER_INDEX["T_g"]]
            assert np.array_equal(mrow_a, mrow_b) and np.array_equal(srow_a, srow_b)
            assert mrow_a[pk.MEMBER_INDEX["fc"]] == pa[k, 0]
            assert np.all(srow_a[:, pk.SC_INDEX["TDPeff"]] == pa[k, 1])
            assert srow_a[0, pk.SC_INDEX["S_reach"]] == pa[k, 3]


def test_entry_points_refuse_bad_ar1_arguments_without_device():
    from simplyp_b200 import _cabi
    from simplyp_b200 import packing as pk
    lib = _cabi.load()
    if lib.simplyp_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    opt = _cabi.default_options()
    po = (C.c_int32 * 2)(0, 0)
    pid = (C.c_int32 * 1)(0)

    def call(ar, V=2):
        dims = _cabi.make_dims(4, 1, 10, 1, V, 0)
        return lib.simplyp_calibrate_ar1_device(C.byref(dims), C.byref(opt), 8, 8, 8, po, pid, 8, 8,
                                                C.byref(ar) if ar is not None else None, 8, 8, 8, None)
    assert call(None) == -1
    assert call(_cabi.make_ar1(8, 2, [0, -1]), V=_cabi.AR1_MAX_SERIES + 1) == -1
    assert call(_cabi.make_ar1(8, -1, [0, -1])) == -1
    assert call(_cabi.make_ar1(None, 2, [0, -1])) == -1
    assert call(_cabi.make_ar1(None, 2, [-1, -1])) == -2          # no phi read: a null pointer is fine
    assert call(_cabi.make_ar1(8, 2, [0, 1])) == -2
    with pytest.raises(ValueError, match="at most"):
        _cabi.make_ar1(8, 1, [0] * (_cabi.AR1_MAX_SERIES + 1))
    # the error-model target kind: its index is a series kind
    de = _cabi.make_de(8, [(_cabi.MCMC_ERROR_MODEL, len(pk.VAR_KINDS), 0)],
                       [0.0], [0.9], 1, 1)
    assert lib.simplyp_de_scale_device(C.byref(de), 8, 8, 8, None) == -1
    de = _cabi.make_de(8, [(_cabi.MCMC_ERROR_MODEL, pk.VAR_INDEX["TDP"], 0)], [0.0], [0.9], 1, 1)
    assert lib.simplyp_de_scale_device(C.byref(de), None, 8, 8, None) == -1
    assert lib.simplyp_de_scale_device(C.byref(de), 8, 8, 8, None) == -2


# ---------------------------------------------------------------------------------------------- public interface
def _tarland():
    from simplyp_b200 import tarland
    return tarland.load("2004-01-01", "2004-12-31", dynamic="y")


@pytest.fixture
def no_device(monkeypatch):
    from simplyp_b200 import engine

    def refuse(*a, **k):
        raise AssertionError("device work before the input check")
    monkeypatch.setattr(engine, "Engine", refuse)


def test_ar1_columns():
    from simplyp_b200 import packing as pk
    labels = [(1, "Q"), (1, "TDP"), (2, "Q")]
    assert pk.ar1_columns(["fc", "err_phi:Q", "err_m:Q"], labels, ("Q", "TDP")) == [1, -1, 1]
    assert pk.ar1_columns(["err_phi:TDP", "err_phi:Q"], labels, None) == [1, 0, 1]
    assert pk.ar1_columns(["fc"], labels, ("Q",)) == [-1, -1, -1]
    with pytest.raises(ValueError, match="unknown series kind"):
        pk.ar1_columns(["err_phi:NO3"], labels, ("Q", "TDP"))
    with pytest.raises(ValueError, match="not among the calibrated variables"):
        pk.ar1_columns(["err_phi:SS"], labels, ("Q", "TDP"))


@pytest.mark.parametrize("name, match", [("err_phi:NO3", "unknown series kind"),
                                         ("err_phi:SS", "not among the calibrated variables"),
                                         ("err_phi:", "unknown series kind")])
def test_calibrate_ensemble_refuses_bad_phi_before_device_work(name, match, no_device):
    from simplyp_b200 import ensemble as ens
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    samples = {"fc": np.full(4, 200.0), name: np.full(4, 0.5)}
    with pytest.raises(ValueError, match=match):
        ens.calibrate_ensemble(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, samples, variables=("Q", "TDP"))


@pytest.mark.parametrize("name, match", [("err_phi:NO3", "unknown series kind"),
                                         ("err_phi:SS", "not among the calibrated variables")])
def test_sampler_and_optimizer_refuse_bad_phi_before_device_work(name, match, no_device):
    from simplyp_b200 import mcmc, optimize
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    priors = {"fc": (100.0, 400.0), name: (0.0, 0.9)}
    with pytest.raises(ValueError, match=match):
        mcmc.sample(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, priors, 8, 2)
    with pytest.raises(ValueError, match=match):
        optimize.differential_evolution(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, priors, 8, 2)


def test_sobol_refuses_phi_before_device_work(no_device):
    from simplyp_b200 import sensitivity
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    with pytest.raises(ValueError, match="AR\\(1\\)"):
        sensitivity.sobol_indices(met, p_struc, p_SU, p_LU, p_SC, p, dyn, {"fc": (100.0, 400.0),
                                  "err_phi:Q": (0.0, 0.9)}, 8, obs_dict=obs, objectives=["NSE"])


def test_phi_is_in_no_parameter_row():
    from simplyp_b200 import ensemble as ens
    from simplyp_b200 import packing as pk
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    base_m, base_sc = pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, [1])
    s = {"fc": np.linspace(150.0, 250.0, 5), "err_m:Q": np.full(5, 0.2)}
    with_phi = dict(s, **{"err_phi:Q": np.linspace(0.0, 0.9, 5), "err_phi:TDP": np.full(5, 0.3)})
    m0, sc0 = ens.pack_members(base_m, base_sc, s)
    m1, sc1 = ens.pack_members(base_m, base_sc, with_phi)
    m2, sc2, phi = ens.pack_members(base_m, base_sc, with_phi, return_phi=True)
    assert np.array_equal(m0, m1) and np.array_equal(sc0, sc1) and np.array_equal(m0, m2) and np.array_equal(sc0, sc2)
    assert list(phi) == ["err_phi:Q", "err_phi:TDP"] and np.array_equal(phi["err_phi:Q"], with_phi["err_phi:Q"])
    assert ens.pack_members(base_m, base_sc, s, return_phi=True)[2] == {}
    pa, pLUa, pSCa = ens.apply_member_to_pandas(with_phi, 3, p, p_LU, p_SC)
    pb, pLUb, pSCb = ens.apply_member_to_pandas(s, 3, p, p_LU, p_SC)
    assert pa.equals(pb) and pLUa.equals(pLUb) and pSCa.equals(pSCb)
