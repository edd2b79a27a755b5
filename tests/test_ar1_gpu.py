"""GPU tier of the AR(1) error model of the log-likelihood (simplyp_calibrate_ar1_device, csrc/simplyp_ar1.cuh) on
Tarland 2004: LOGLIK against the NumPy factorisation and the host build, rebuilt from a full-output run of the same
members; every other statistic bitwise unchanged; invariance to the batch; the sampler with phi among its priors;
recovery of a known phi by differential evolution."""
import math

import numpy as np
import pandas as pd
import pytest

from tests import ar1_reference as ref
from tests import fit_stats_reference as fsr

pytestmark = pytest.mark.gpu

PHI_RANGES = {"err_phi:Q": (0.0, 0.95), "err_phi:TDP": (0.0, 0.95)}
M = 256


@pytest.fixture(scope="module")
def cabi():
    from simplyp_b200 import _cabi
    _cabi.require_device()
    return _cabi


@pytest.fixture(scope="module")
def tarland():
    from simplyp_b200 import tarland as t
    return t.load("2004-01-01", "2004-12-31", dynamic="y")


def _args(tarland):
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland
    return met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs


@pytest.fixture(scope="module")
def ensemble(cabi, tarland):
    """256 Latin-hypercube members with phi of Q and TDP in [0, 0.95] (every eighth member phi = 0), their statistics
    with and without the AR(1) model, rank statistics off and on, and the full-output run of the same members."""
    from simplyp_b200 import ensemble as ens, model as spm, packing as pk
    samples = ens.latin_hypercube(M, dict(ens.TARLAND_RANGES, **PHI_RANGES), seed=11)
    for k in PHI_RANGES:
        samples[k][::8] = 0.0
    iid = {k: v for k, v in samples.items() if k not in PHI_RANGES}
    a = _args(tarland)
    got = {}
    for rank in (False, True):
        for name, s in (("ar1", samples), ("iid", iid)):
            stats, labels, diag = ens.calibrate_ensemble(*a, s, rank_stats=rank)
            got[name, rank] = (stats.cpu().numpy(), diag.cpu().numpy())
    met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs_dict = a
    topo = pk.build_topology(p_struc, p["SC_list"])
    opt = spm.make_options(p_SU, p, dyn, topo)
    member, sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), samples)
    out, diag = cabi.run_host(pk.forcing_matrix(met), member, sc, topo.parent_offsets, topo.parent_ids, opt)
    obs, desc, labels2 = pk.obs_arrays(obs_dict, topo, met.index, ("Q", "TDP"))
    assert labels2 == labels and [v for _s, v in labels] == ["Q", "TDP"]
    return dict(samples=samples, got=got, out=out, diag=diag, member=member, sc=sc, obs=obs, desc=desc, labels=labels)


def _sim(e, m, v):
    reach, kind = int(e["desc"][v, 0]), int(e["desc"][v, 1])
    scp = e["sc"][m if e["sc"].shape[0] > 1 else 0]
    return fsr.simulated(e["out"][m, reach], scp[reach, fsr.SC_A_CATCH], e["member"][m, fsr.P_F_TDP], kind), kind


def test_loglik_matches_the_reference_and_the_host_build(ensemble):
    from tests import ar1_host
    e = ensemble
    stats, diag = e["got"]["ar1", False]
    assert not diag[..., 3].any() and not e["diag"][..., 3].any()
    worst_ref = worst_host = 0.0
    for m in range(M):
        for v, (_sc, var) in enumerate(e["labels"]):
            s, kind = _sim(e, m, v)
            phi, em = e["samples"]["err_phi:" + var][m], e["member"][m, fsr.P_ERR_M[kind]]
            want = ref.loglik_sequential(e["obs"][v], s, em, phi)
            host = ar1_host.row(e["obs"][v], s, em, phi)
            g = stats[m, v, fsr.ST_LOGLIK]
            assert math.isfinite(want) and math.isfinite(g), (m, v, g, want)
            worst_ref = max(worst_ref, abs(g - want) / abs(want))
            worst_host = max(worst_host, abs(g - host) / abs(host))
    print("AR(1) LOGLIK: max relative difference %.3g to NumPy, %.3g to the host build" % (worst_ref, worst_host))
    assert worst_ref <= 1e-10 and worst_host <= 1e-10


@pytest.mark.parametrize("rank", [False, True])
def test_other_statistics_are_bitwise_those_of_the_iid_run(ensemble, rank):
    e = ensemble
    a, da = e["got"]["ar1", rank]
    b, db = e["got"]["iid", rank]
    assert np.array_equal(da, db)
    others = [k for k in range(fsr.NSTAT) if k != fsr.ST_LOGLIK]
    assert np.array_equal(a[..., others], b[..., others], equal_nan=True)
    if rank:
        assert np.isfinite(a[..., fsr.ST_SPEARMAN]).all()
    # phi = 0 is the iid likelihood
    zero = np.arange(0, M, 8)
    x, y = a[zero, :, fsr.ST_LOGLIK], b[zero, :, fsr.ST_LOGLIK]
    assert np.all(np.abs(x - y) <= 1e-12 * np.abs(y))
    # and the AR(1) model changes it elsewhere
    assert np.all(a[1:8, :, fsr.ST_LOGLIK] != b[1:8, :, fsr.ST_LOGLIK])


def test_a_member_alone_and_in_the_batch_give_the_same_bits(ensemble, tarland):
    from simplyp_b200 import ensemble as ens
    e = ensemble
    batch = e["got"]["ar1", False][0]
    a = _args(tarland)
    for i in (0, 37, M - 1):
        one = {k: v[i:i + 1] for k, v in e["samples"].items()}
        stats, _l, _d = ens.calibrate_ensemble(*a, one)
        assert np.array_equal(stats.cpu().numpy()[0], batch[i], equal_nan=True)        # (Spearman's r is NaN)
    rev = {k: np.ascontiguousarray(v[::-1]) for k, v in e["samples"].items()}
    stats, _l, _d = ens.calibrate_ensemble(*a, rev)
    assert np.array_equal(stats.cpu().numpy()[::-1], batch, equal_nan=True)


def test_sampler_with_phi_under_graph_replay(cabi, tarland):
    from simplyp_b200 import ensemble as ens, mcmc
    a = _args(tarland)
    priors = {"fc": (100.0, 400.0), "T_g": (20.0, 150.0), "err_m:Q": (0.05, 1.0), "err_phi:Q": (0.0, 0.95)}
    r = mcmc.sample(*a, priors, 64, 50, seed=5)
    k = r.names.index("err_phi:Q")
    assert np.all((r.chain[..., k] >= 0.0) & (r.chain[..., k] <= 0.95))
    assert r.acceptance_fraction.mean() > 0
    last = {n: np.ascontiguousarray(r.last[:, j]) for j, n in enumerate(r.names)}
    stats, labels, diag = ens.calibrate_ensemble(*a, last)
    st, dg = stats.cpu().numpy(), diag.cpu().numpy()
    lp = np.zeros(64)
    for v in range(st.shape[1]):
        lp = lp + st[:, v, fsr.ST_LOGLIK]
    lp[np.any(dg[..., 3] != 0, axis=1) | np.isnan(lp)] = -np.inf
    assert np.isfinite(r.last_log_prob).all()
    assert np.array_equal(lp, r.last_log_prob)


def test_differential_evolution_recovers_phi(cabi, tarland):
    """Q of a known member times (1 + m eta), eta a stationary AR(1) with phi = 0.8 on the real 2004 Q days; DE over
    phi and m with the model parameters at the truth.  The standard error of phi-hat is about 0.03 at n ~ 360."""
    from simplyp_b200 import model as spm, optimize, packing as pk
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland
    topo = pk.build_topology(p_struc, p["SC_list"])
    opt = spm.make_options(p_SU, p, dyn, topo)
    out, diag = cabi.run_host(pk.forcing_matrix(met), pk.member_vector(p, p_LU)[None], pk.sc_matrix(p_SC, topo.sc_ids),
                              topo.parent_offsets, topo.parent_ids, opt)
    assert not diag[..., 3].any()
    q = out[0, 0, :, pk.RAW_COLS.index("Qr")] * float(p_SC.loc["A_catch", 1]) * 1000 / 86400
    ser = obs[1]["Q"]
    seen = ser[~ser.index.duplicated()].reindex(met.index).notna().to_numpy()
    phi, m = 0.8, 0.1
    rng = np.random.default_rng(20261021)
    eta = np.empty(len(q))
    eta[0] = rng.standard_normal()
    for t in range(1, len(q)):
        eta[t] = phi * eta[t - 1] + math.sqrt(1.0 - phi * phi) * rng.standard_normal()
    q_obs = np.where(seen, q * (1.0 + m * eta), np.nan)
    data = {1: pd.DataFrame({"Q": q_obs}, index=met.index)}
    ranges = {"err_phi:Q": (0.0, 0.99), "err_m:Q": (0.02, 0.5)}
    r = optimize.differential_evolution(met, p_struc, p_SU, p_LU, p_SC, p, dyn, data, ranges, 32, 200,
                                        objective="lp", variables=("Q",), seed=3, tol=1e-8)
    print("AR(1) recovery: phi-hat %.4f, m-hat %.4f, n = %d, generations %d"
          % (r.best["err_phi:Q"], r.best["err_m:Q"], int(seen.sum()), r.generations))
    assert abs(r.best["err_phi:Q"] - phi) <= 0.1
    # the optimum is the maximum of the AR(1) likelihood: the NumPy factorisation agrees at the best member
    want = ref.loglik_sequential(q_obs, q, r.best["err_m:Q"], r.best["err_phi:Q"])
    assert abs(r.best_objective - want) <= 1e-9 * abs(want)
