"""GPU tier of the posterior predictive bands (simplyp_predictive_draws_device, simplyp_nanquantile_device,
ensemble.predictive_bands): the selection against np.nanquantile and torch.nanquantile bitwise on both of its paths,
the draws against the fit-statistics reference on the kernel's own full output, the error draws against the host
build, chunking, failed members, an end-to-end run after the sampler, graph capture and the memory check."""
import math
import warnings

import numpy as np
import pytest

from tests import fit_stats_reference as ref

pytestmark = pytest.mark.gpu

SEED = 0x5eed_0000_b0d5
Q = [0.0, 0.025, 0.25, 0.5, 0.75, 0.975, 1.0, 1 / 3]


@pytest.fixture(scope="module")
def eng():
    from simplyp_b200.engine import Engine
    return Engine()


def _np_nanquantile(x, q):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return np.nanquantile(x, q, axis=-1)


def _same(a, b):
    """Bitwise equal, NaN equal to NaN, +0 equal to -0."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def _matrix(R, N, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(size=(R, N))
    x[: R // 4] = np.round(x[: R // 4], 2)                      # ties
    x[rng.random(x.shape) < 0.1] = np.nan
    x[1] = np.nan                                               # all NaN
    x[2] = np.nan
    x[2, N // 2] = 1.25                                         # a single value
    x[3, :: 7] = np.inf
    x[4, :: 5] = -np.inf
    x[5] = 0.0
    x[5, ::2] = -0.0
    return x


# --------------------------------------------------------------------------- 1. selection
@pytest.mark.parametrize("N", [1, 2, 1000, 20000, 40000, 100003])
def test_nanquantile_equals_numpy_and_torch(eng, N):
    import torch
    from simplyp_b200 import _cabi
    shared = _cabi.nanquantile_workspace_bytes(8, N) == 0
    assert shared == (N <= 20000)                               # both paths are exercised
    x = _matrix(12, N, N)
    quant, mean, count = eng.nanquantile(eng.to_device(x), Q)
    quant, mean, count = quant.cpu().numpy(), mean.cpu().numpy(), count.cpu().numpy()
    assert _same(quant, _np_nanquantile(x, Q))
    # torch as a second reference, on the rows without infinities and the q whose (n - 1) q is exact: elsewhere
    # torch's own weight can differ from NumPy's by an ulp (q = 1/3 at n = 2), and NumPy is the specification
    finite = np.array([np.all(np.isfinite(r[~np.isnan(r)])) and np.any(~np.isnan(r)) for r in x])
    dyadic = [k for k, q in enumerate(Q) if q in (0.0, 0.25, 0.5, 0.75, 1.0)]
    qt = torch.tensor([Q[k] for k in dyadic], dtype=torch.float64)
    want_t = torch.nanquantile(torch.from_numpy(x[finite]), qt, dim=-1).numpy()
    assert _same(quant[dyadic][:, finite], want_t)
    assert np.array_equal(count, np.sum(~np.isnan(x), axis=-1))
    for r in range(x.shape[0]):
        v = x[r][~np.isnan(x[r])]
        if v.size == 0:
            assert np.isnan(mean[r])
        elif np.all(np.isfinite(v)):
            want = math.fsum(v.tolist()) / v.size
            assert abs(mean[r] - want) <= v.size * ref.EPS * np.abs(v).sum() / v.size + ref.EPS * abs(want)


# --------------------------------------------------------------------------- 2.-4. draws
def _ensemble(kind, M, seed=3, extra=None, years=("2004-01-01", "2004-12-31")):
    from simplyp_b200 import ensemble as ens, model as spm, packing as pk, tarland
    from tests.golden.networks import network5_inputs
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(years[0], years[1], dynamic="y")
    ranges = {"fc": (100.0, 400.0), "T_g": (20.0, 150.0), "a_Q": (0.2, 0.9), "f_TDP": (0.2, 0.8),
              "err_m:Q": (0.05, 0.3), "err_m:SS": (0.2, 0.4), "err_m:TDP": (0.3, 0.6), "err_m:PP": (0.4, 0.7),
              "err_m:TP": (0.5, 0.9), "err_m:SRP": (0.6, 1.0)}
    if kind == "network5":
        p, p_LU, p_SC, p_struc = network5_inputs(p, p_LU, p_SC, p_struc)
        pk.validate_land_use(p_SC, p["SC_list"])
        ranges["sc:A_catch@2"] = (20.0, 50.0)
        ranges["sc:TDPeff"] = (0.0, 0.5)
    ranges.update(extra or {})
    samples = ens.latin_hypercube(M, ranges, seed=seed)
    topo = pk.build_topology(p_struc, p["SC_list"])
    member, sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), samples)
    return dict(inputs=(met, p_struc, p_SU, p_LU, p_SC, p, dyn), obs=obs, samples=samples, topo=topo,
                opt=spm.make_options(p_SU, p, dyn, topo), member=member, sc=sc,
                forcing=pk.forcing_matrix(met))


def _run(eng, w):
    d = dict(forc=eng.to_device(w["forcing"]), mem=eng.to_device(w["member"]), sc=eng.to_device(w["sc"]))
    out, diag = eng.run(d["forc"], d["mem"], d["sc"], w["topo"].parent_offsets, w["topo"].parent_ids, w["opt"])
    return d, out, diag


def _draws(eng, d, out, diag, desc, obs_error, seed=SEED):
    import torch
    V, (M, S, D) = len(desc), out.shape[:3]
    draws = torch.full((V, D, M), -7.0, dtype=torch.float64, device=eng.device)
    eng.predictive_draws(out, d["mem"], d["sc"], diag, eng.to_device(np.asarray(desc, dtype=np.int32)), draws, 0,
                         obs_error, seed)
    return draws.cpu().numpy()


def _expected(w, out_h, diag_h, desc):
    M = out_h.shape[0]
    sc = np.broadcast_to(w["sc"], (M,) + w["sc"].shape[1:])
    want = np.empty((len(desc), out_h.shape[2], M))
    for v, (s, kind) in enumerate(desc):
        for m in range(M):
            want[v, :, m] = ref.simulated(out_h[m, s], sc[m, s, ref.SC_A_CATCH], w["member"][m, ref.P_F_TDP], kind)
    failed = np.any(diag_h[:, :, 3] != 0, axis=1)
    want[:, :, failed] = np.nan
    return want


def _check_sim(got, want):
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert np.all(np.abs(got[ok] - want[ok]) <= ref.SIM_ULPS * ref.EPS * np.abs(want[ok]))


def test_draws_without_error_equal_reference_tarland(eng):
    w = _ensemble("tarland", 512)
    d, out, diag = _run(eng, w)
    desc = [(0, k) for k in range(6)]
    got = _draws(eng, d, out, diag, desc, False)
    _check_sim(got, _expected(w, out.cpu().numpy(), diag.cpu().numpy(), desc))


def test_draws_without_error_equal_reference_network5(eng):
    w = _ensemble("network5", 96)
    assert w["sc"].shape[0] == 96 and np.unique(w["sc"][:, 2, ref.SC_A_CATCH]).size == 96
    d, out, diag = _run(eng, w)
    desc = [(s, k) for s in (2, 4) for k in range(6)]
    got = _draws(eng, d, out, diag, desc, False)
    _check_sim(got, _expected(w, out.cpu().numpy(), diag.cpu().numpy(), desc))


def test_error_draws_equal_host_epsilon(eng):
    from tests import bands_host
    w = _ensemble("network5", 64)
    d, out, diag = _run(eng, w)
    desc = [(s, k) for s in (2, 4) for k in range(6)]
    sim = _draws(eng, d, out, diag, desc, False)
    y = _draws(eng, d, out, diag, desc, True)
    V, D, M = y.shape
    vv, dd, mm = np.meshgrid(np.arange(V), np.arange(D), np.arange(M), indexing="ij")
    eps_h = bands_host.epsilon(SEED, mm.ravel(), dd.ravel(), vv.ravel()).reshape(V, D, M)
    scale = np.stack([w["member"][:, ref.P_ERR_M[k]] for _, k in desc])[:, None, :] * sim
    ok = np.isfinite(sim) & (scale != 0)
    assert ok.mean() > 0.5
    with np.errstate(invalid="ignore", divide="ignore"):
        rec = (y - sim) / scale
    # host bound (8 ulp) + cospi on the device (4 ulp) + the roundings of y = sim + scale eps and of its recovery
    tol = 12 * np.spacing(np.abs(eps_h)) + 2 * (np.spacing(np.abs(y)) + np.spacing(np.abs(scale * eps_h))) / np.abs(scale)
    assert np.all(np.abs(rec[ok] - eps_h[ok]) <= tol[ok])
    assert np.array_equal(np.isnan(y), np.isnan(sim))


# --------------------------------------------------------------------------- 5. chunking
def test_chunking_changes_no_bit(eng):
    import torch
    from simplyp_b200 import ensemble as ens
    M = 74
    w = _ensemble("tarland", M, years=("2004-01-01", "2004-06-30"))
    series = [(1, "Q"), (1, "TDP"), (1, "SRP")]
    desc = np.array([(0, 0), (0, 2), (0, 5)], dtype=np.int32)
    d = dict(forc=eng.to_device(w["forcing"]), mem=eng.to_device(w["member"]), sc=eng.to_device(w["sc"]))
    draws, bands = [], []
    for chunk in (1, 37, M):
        D = w["forcing"].shape[0]
        x = torch.empty((3, D, M), dtype=torch.float64, device=eng.device)
        for m0 in range(0, M, chunk):
            n = min(chunk, M - m0)
            out, diag = eng.run(d["forc"], d["mem"][m0:m0 + n], d["sc"], w["topo"].parent_offsets,
                                w["topo"].parent_ids, w["opt"])
            eng.predictive_draws(out, d["mem"][m0:m0 + n], d["sc"], diag, eng.to_device(desc), x, m0, True, SEED)
        draws.append(x.cpu().numpy())
        bands.append(ens.predictive_bands(*w["inputs"], w["samples"], series, obs_error=True, seed=SEED,
                                          members_per_chunk=chunk, engine=eng))
    for k in (1, 2):
        assert np.array_equal(draws[k], draws[0], equal_nan=True)
        for f in ("quantiles", "mean", "count"):
            assert np.array_equal(getattr(bands[k], f), getattr(bands[0], f), equal_nan=True)
    assert _same(bands[0].quantiles, _np_nanquantile(draws[0], bands[0].q))


# --------------------------------------------------------------------------- 6. failed members
def test_failed_members_are_excluded(eng):
    import torch
    M = 128
    w = _ensemble("tarland", M, extra={"T_s:A": (1.0, 8.0), "E_M": (300.0, 3000.0)})
    d = dict(forc=eng.to_device(w["forcing"]), mem=eng.to_device(w["member"]), sc=eng.to_device(w["sc"]))
    desc = np.array([(0, 0), (0, 2)], dtype=np.int32)
    for steps in (2, 3, 4, 6, 8, 12, 16, 24, 32):
        w["opt"].max_steps_per_day = steps
        out, diag = eng.run(d["forc"], d["mem"], d["sc"], w["topo"].parent_offsets, w["topo"].parent_ids, w["opt"])
        status = diag.cpu().numpy()[:, :, 3]
        failed = np.any(status != 0, axis=1)
        if np.any(status & 1) and 0 < failed.sum() < M:
            break
    else:
        pytest.fail("no max_steps_per_day failed some members but not all")
    D = w["forcing"].shape[0]
    x = torch.empty((2, D, M), dtype=torch.float64, device=eng.device)
    eng.predictive_draws(out, d["mem"], d["sc"], diag, eng.to_device(desc), x, 0, True, SEED)
    quant, mean, count = eng.nanquantile(x.view(2 * D, M), Q)
    xh = x.cpu().numpy()
    assert np.all(np.isnan(xh[:, :, failed])) and not np.any(np.isnan(xh[:, :, ~failed]))
    assert np.all(count.cpu().numpy() == M - failed.sum())
    assert _same(quant.cpu().numpy(), _np_nanquantile(xh.reshape(2 * D, M), Q))


# --------------------------------------------------------------------------- 7. after the sampler
def test_bands_after_the_sampler(eng):
    from simplyp_b200 import ensemble as ens, mcmc
    w = _ensemble("tarland", 1)
    met, p_struc, p_SU, p_LU, p_SC, p, dyn = w["inputs"]
    priors = {"fc": (100.0, 400.0), "T_g": (20.0, 150.0), "a_Q": (0.2, 0.9), "err_m:Q": (0.05, 1.0),
              "err_m:TDP": (0.05, 1.0)}
    r = mcmc.sample(met, p_struc, p_SU, p_LU, p_SC, p, dyn, w["obs"], priors, 64, 20, engine=eng)
    samples = r.flat_samples(burn=10)
    series = [(1, "Q"), (1, "TDP")]
    b = ens.predictive_bands(met, p_struc, p_SU, p_LU, p_SC, p, dyn, samples, series, obs_error=True, seed=SEED,
                             engine=eng)
    from simplyp_b200 import packing as pk
    member, sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, w["topo"].sc_ids), samples)
    w2 = dict(w, member=member, sc=sc)
    d, out, diag = _run(eng, w2)
    x = _draws(eng, d, out, diag, [(0, 0), (0, 2)], True)
    assert b.n_failed == int(np.any(diag.cpu().numpy()[:, :, 3] != 0, axis=1).sum())
    assert _same(b.quantiles, _np_nanquantile(x, b.q))
    assert np.array_equal(b.count, np.sum(~np.isnan(x), axis=-1))
    cov = b.coverage(w["obs"], 0.025, 0.975)
    for v, lab in enumerate(series):
        o = w["obs"][1][lab[1]]
        o = o[~o.index.duplicated()].reindex(met.index).to_numpy(dtype="float64")
        seen = ~np.isnan(o)
        lo, hi = _np_nanquantile(x[v], [0.025, 0.975])
        inside = np.sum((lo[seen] <= o[seen]) & (o[seen] <= hi[seen]))
        assert cov[lab] == (int(seen.sum()), inside / seen.sum())


# --------------------------------------------------------------------------- 8. graph capture
@pytest.mark.parametrize("N", [5000, 40000])
def test_entry_points_capture_into_a_graph(eng, N):
    import torch
    w = _ensemble("tarland", 64, years=("2004-01-01", "2004-03-31"))
    d, out, diag = _run(eng, w)
    desc = eng.to_device(np.array([(0, 0), (0, 2)], dtype=np.int32))
    D = out.shape[2]
    x = torch.empty((2, D, 64), dtype=torch.float64, device=eng.device)
    big = eng.to_device(_matrix(16, N, 11))
    qa, ma, ca = (torch.empty((len(Q), 16), dtype=torch.float64, device=eng.device),
                  torch.empty(16, dtype=torch.float64, device=eng.device),
                  torch.empty(16, dtype=torch.int64, device=eng.device))
    eng.predictive_draws(out, d["mem"], d["sc"], diag, desc, x, 0, True, SEED)
    eng.nanquantile(big, Q, qa, ma, ca)
    torch.cuda.synchronize()
    direct = [t.cpu().numpy() for t in (x, qa, ma, ca)]
    for t in (x, qa, ma, ca):
        t.fill_(0)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        eng.predictive_draws(out, d["mem"], d["sc"], diag, desc, x, 0, True, SEED)
        eng.nanquantile(big, Q, qa, ma, ca)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(direct, (x, qa, ma, ca)):
        assert np.array_equal(a, b.cpu().numpy(), equal_nan=True)


# --------------------------------------------------------------------------- 9. memory check
def test_over_budget_draws_refused_before_any_launch(eng):
    from simplyp_b200 import _cabi, ensemble as ens
    from simplyp_b200.engine import Engine

    class Small(Engine):
        def free_bytes(self):
            return 1 << 20
    w = _ensemble("tarland", 400)
    n0 = _cabi.launch_count()
    with pytest.raises(ValueError, match="thin"):
        ens.predictive_bands(*w["inputs"], w["samples"], [(1, "Q"), (1, "TDP")], engine=Small())
    assert _cabi.launch_count() == n0
