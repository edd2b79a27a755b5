"""GPU tier of the fused fit statistics: every slot of every (member, series) of simplyp_calibrate_* against the exact
reference of tests/fit_stats_reference.py, rebuilt from the kernel's own full-output run of the same members.  Each
case also checks that the calibration run took the same steps as the full-output run (so the simulated values the
reference rebuilds are the calibration kernel's own), and runs with rank statistics off and on.

Not covered: Spearman's re-ranking of the observations when a member's simulated value is NaN on an observed day
(spearman_kernel's rerank_obs path); no valid input reaches it without a failing member."""
import numpy as np
import pytest

from tests import fit_stats_reference as ref

pytestmark = pytest.mark.gpu

# Disjoint ranges: the ensemble writes each err_m column by name (packing.MEMBER_INDEX) and the reference reads it by
# name, while the kernel reads SIMPLYP_P_ERR_M0 + kind; a header and packing order that disagree give another scale.
ERR_M_RANGES = {"err_m:Q": (0.05, 0.1), "err_m:SS": (0.2, 0.3), "err_m:TDP": (0.4, 0.5), "err_m:PP": (0.6, 0.7),
                "err_m:TP": (0.8, 0.9), "err_m:SRP": (1.0, 1.1)}


@pytest.fixture(scope="module")
def cabi():
    from simplyp_b200 import _cabi
    _cabi.require_device()
    return _cabi


def _tarland(M, seed=3, extra=None):
    from simplyp_b200 import ensemble as ens, model as spm, packing as pk, tarland
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load("2004-01-01", "2004-12-31", dynamic="y")
    topo = pk.build_topology(p_struc, p["SC_list"])
    opt = spm.make_options(p_SU, p, dyn, topo)
    ranges = {k: v for k, v in ens.TARLAND_RANGES.items() if not k.startswith("err_m:")}
    ranges.update(ERR_M_RANGES)
    ranges["f_TDP"] = (0.2, 0.8)
    ranges.update(extra or {})
    samples = ens.latin_hypercube(M, ranges, seed=seed)
    member, sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), samples)
    w = dict(forcing=pk.forcing_matrix(met), member=member, sc=sc, topo=topo, opt=opt, obs=obs, index=met.index)
    _assert_disjoint_error_scales(w)
    return w


def _network(kind, M, seed=5):
    from simplyp_b200 import ensemble as ens, model as spm, packing as pk, synthetic, tarland
    from tests.golden.networks import network5_inputs
    if kind == "network5":
        p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load("2004-01-01", "2004-12-31", dynamic="y")
        p, p_LU, p_SC, p_struc = network5_inputs(p, p_LU, p_SC, p_struc)
    else:                                   # the 64-reach synthetic network of the epoch-sweep test, 700 days
        p_SU, dyn, p, p_LU, p_SC0, p_struc0, met, obs = tarland.load("2003-06-01", "2005-04-30", dynamic="y")
        p, p_SC, p_struc = synthetic.random_network(p, p_SC0[1], n_sc=64, seed=3)
    pk.validate_land_use(p_SC, p["SC_list"])
    topo = pk.build_topology(p_struc, p["SC_list"])
    opt = spm.make_options(p_SU, p, dyn, topo)
    ranges = dict(ERR_M_RANGES, **{"fc": (100.0, 400.0), "T_g": (20.0, 150.0), "f_TDP": (0.2, 0.8),
                                   "sc:TDPeff": (0.0, 0.5)})
    samples = ens.latin_hypercube(M, ranges, seed=seed)
    member, sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), samples)
    w = dict(forcing=pk.forcing_matrix(met), member=member, sc=sc, topo=topo, opt=opt, obs=obs, index=met.index)
    _assert_disjoint_error_scales(w)
    return w


def _synthetic_obs(cabi, w, rows, seed=1, missing=0.2):
    """Observations of a truth member (member 0) for rows [(reach position, kind, mask or None)]: its simulated series
    with multiplicative noise, rounded to 3 significant digits (ties), about `missing` of the days removed."""
    out, _ = cabi.run_host(w["forcing"], w["member"][:1], w["sc"][:1], w["topo"].parent_offsets, w["topo"].parent_ids,
                           w["opt"])
    rng = np.random.default_rng(seed)
    D = w["forcing"].shape[0]
    obs = np.full((len(rows), D), np.nan)
    for v, (s, kind, mask) in enumerate(rows):
        sim = ref.simulated(out[0, s], w["sc"][0, s, ref.SC_A_CATCH], w["member"][0, ref.P_F_TDP], kind)
        x = sim * rng.lognormal(0.0, 0.2, D)
        x = np.array([float("%.3g" % t) for t in x])
        keep = rng.random(D) >= missing if mask is None else mask
        obs[v, keep] = x[keep]
    desc = np.array([(s, k) for s, k, _ in rows], dtype=np.int32)
    return obs, desc


def _assert_disjoint_error_scales(w):
    """Every member's err_m columns, found by name, lie in their own disjoint range (guards the fixture itself)."""
    for k, var in enumerate(ref.VAR_KINDS):
        lo, hi = ERR_M_RANGES["err_m:" + var]
        col = w["member"][:, ref.P_ERR_M[k]]
        assert np.all((col >= lo) & (col <= hi)), var


def _check(cabi, w, obs, desc, rank_modes=(0, 1), scaled_from=None):
    """Calibration statistics of w's members == the reference on the full-output run, every slot.  Returns the
    statistics of each rank mode.  scaled_from = (obs0, k): r^2 and Spearman are checked against the reference of
    the unscaled observations obs0 (= obs / 2^k)."""
    po, pid, opt = w["topo"].parent_offsets, w["topo"].parent_ids, w["opt"]
    out, dg = cabi.run_host(w["forcing"], w["member"], w["sc"], po, pid, opt)
    assert not np.any(dg[..., 3])
    want, bound = ref.reference_stats(out, w["member"], w["sc"], obs, desc)
    if scaled_from is not None:
        want0, bound0 = ref.reference_stats(out, w["member"], w["sc"], scaled_from[0], desc)
        for k in (ref.ST_R2, ref.ST_SPEARMAN):
            want[..., k], bound[..., k] = want0[..., k], bound0[..., k]
    res = {}
    try:
        for rs in rank_modes:
            opt.rank_stats = rs
            st, dgc = cabi.calibrate_host(w["forcing"], w["member"], w["sc"], po, pid, obs, desc, opt)
            assert np.array_equal(dgc, dg), "calibration and full-output runs took different steps"
            slots = [k for k in range(ref.NSTAT) if rs or k != ref.ST_SPEARMAN]
            bad = ref.compare(st, want, bound, slots)
            assert not bad, "rank_stats=%d: %d slots off, first %s: got %r want %r bound %r" % (
                rs, len(bad), bad[:5], st[bad[0][:2]], want[bad[0][:2]], bound[bad[0][:2]])
            if not rs:
                assert np.all(np.isnan(st[..., ref.ST_SPEARMAN]))
            res[rs] = st
    finally:
        opt.rank_stats = 0
    return res


def test_every_kind_and_every_error_scale_on_tarland(cabi):
    """Tarland 2004, all six observed series, 515 members: the pilot runs (ensembles of >= 512 members) and the last warp
    of 8 quads is ragged.  err_m of the six kinds, f_TDP and TDPeff are sampled, the err_m on disjoint ranges."""
    from simplyp_b200 import packing as pk
    w = _tarland(515)
    obs, desc, labels = pk.obs_arrays(w["obs"], w["topo"], w["index"], None)
    assert [k for _s, k in desc.tolist()] == list(range(6))
    _check(cabi, w, obs, desc)


def test_network_with_observations_inside_it(cabi):
    """5-reach network (1,2 -> 3; 3,4 -> 5), 13 members; six kinds on a headwater, the confluence and the outlet, the
    obs_desc rows interleaved across the reaches (the shared-memory slot is a row's rank among its reach's rows)."""
    w = _network("network5", 13)
    rows = [(s, k, None) for k in range(6) for s in (0, 2, 4)]
    obs, desc = _synthetic_obs(cabi, w, rows)
    _check(cabi, w, obs, desc)


def _overflow_rows(D, s, rng, extra=()):
    """Eight series on reach s: Q and TDP twice each with different missing days, then SS, PP, TP, SRP; the last two
    rows of the reach take the global-memory accumulators (slots 6 and 7)."""
    masks = [rng.random(D) >= 0.2 for _ in range(4)]
    return [(s, 0, masks[0]), (s, 2, masks[1]), (s, 1, None), (s, 3, None), (s, 4, None), (s, 5, None),
            (s, 0, masks[2]), (s, 2, masks[3])] + list(extra)


def _assert_permuted(cabi, w, obs, desc, st, perm):
    """Moving series between slot < 6 and slot >= 6 by reordering obs_desc permutes the rows bitwise: the two kinds of
    accumulator run the same operations in the same order, only their memory differs."""
    po, pid, opt = w["topo"].parent_offsets, w["topo"].parent_ids, w["opt"]
    stp, _ = cabi.calibrate_host(w["forcing"], w["member"], w["sc"], po, pid, obs[perm], desc[perm], opt)
    assert np.array_equal(stp, st[:, perm], equal_nan=True)


def test_more_than_six_series_on_a_reach_tarland(cabi):
    w = _tarland(515, seed=8)
    D = w["forcing"].shape[0]
    rows = _overflow_rows(D, 0, np.random.default_rng(2))
    obs, desc = _synthetic_obs(cabi, w, rows)
    st = _check(cabi, w, obs, desc)
    _assert_permuted(cabi, w, obs, desc, st[0], [6, 7, 2, 3, 4, 5, 0, 1])


def test_more_than_six_series_on_an_interior_reach_of_a_swept_network(cabi, monkeypatch):
    """64-reach network, 700 days in epochs of 128 days: eight series on an interior reach (parents and a child), a
    headwater series beside it, and series observed only across the epoch boundaries (days 127/128, 255/256)."""
    monkeypatch.setenv("SIMPLYP_EPOCH_DAYS", "128")
    w = _network("net64", 3)
    topo = w["topo"]
    po = np.asarray(topo.parent_offsets)
    S, D = len(po) - 1, w["forcing"].shape[0]
    assert D == 700
    children = set(np.asarray(topo.parent_ids).tolist())
    interior = [s for s in range(S - 1) if po[s + 1] > po[s] and s in children]
    head = [s for s in range(S) if po[s + 1] == po[s]]
    s_in = interior[len(interior) // 2]
    edges = np.zeros(D, bool)
    edges[[127, 128, 255, 256]] = True
    rows = [(head[0], 0, None)] + _overflow_rows(D, s_in, np.random.default_rng(3)) + [(head[1], 2, edges)]
    obs, desc = _synthetic_obs(cabi, w, rows)
    st = _check(cabi, w, obs, desc)
    perm = [0, 7, 8, 3, 4, 5, 6, 1, 2, 9]
    _assert_permuted(cabi, w, obs, desc, st[0], perm)


def test_where_the_observed_days_fall(cabi):
    """Tarland with the pilot (515 members; the pilot integrates days 0-7): series observed only on day 0, on days 7/8
    (the pilot hand-over), on days 127/128 (a forcing tile), on the last day, on no day, on 0/1/2 days, with an
    observation of 0 and a negative one.  err_m:SS is 0 on the even members: their SS series and lp are -inf."""
    import torch
    w = _tarland(515, seed=4)
    w["member"][0::2, ref.P_ERR_M[1]] = 0.0
    D = w["forcing"].shape[0]

    def days(*ds):
        m = np.zeros(D, bool)
        m[list(ds)] = True
        return m
    odd = np.random.default_rng(5).random(D) >= 0.3
    rows = [(0, 0, days(0)), (0, 2, days(7, 8)), (0, 1, days(127, 128)), (0, 3, days(D - 1)), (0, 4, days()),
            (0, 5, odd), (0, 0, days(0, 7, 8, 127, 128, D - 1)), (0, 2, odd)]
    obs, desc = _synthetic_obs(cabi, w, rows)
    obs[5, np.flatnonzero(odd)[:2]] = [0.0, -0.004]           # an observation of 0 and a negative one
    st = _check(cabi, w, obs, desc)[1]
    assert np.array_equal(st[:, 4, ref.ST_N], np.zeros(515)) and np.all(st[:, 0, ref.ST_N] == 1)
    assert np.all(st[0::2, 2, ref.ST_LOGLIK] == -np.inf) and np.all(np.isfinite(st[1::2, 2, ref.ST_LOGLIK]))
    # the sampler's lp over these statistics: the even members' -inf series makes their lp -inf
    from simplyp_b200 import _cabi
    M, V = 514, obs.shape[0]
    dev = torch.device("cuda", 0)
    t = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)
    stats, diag = t(st[:M]), torch.zeros((M, 1, 4), dtype=torch.int64, device=dev)
    walkers, lp = t(np.zeros((M, 1))), t(np.zeros(M))
    prop, log_z, oob = t(np.zeros((M // 2, 1))), t(np.zeros(M // 2)), t(np.zeros(M // 2), torch.int32)
    it, acc = t([0], torch.int64), t(np.zeros(M), torch.int64)
    chain, chain_lp = t(np.zeros((1, M, 1))), t(np.zeros((1, M)))
    mc = _cabi.make_mcmc(M, [(_cabi.MCMC_MEMBER, 2, 0)], [0.0], [1000.0], 1, V)
    state = _cabi.make_mcmc_state(walkers.data_ptr(), lp.data_ptr(), prop.data_ptr(), log_z.data_ptr(),
                                  oob.data_ptr(), it.data_ptr(), acc.data_ptr(), chain.data_ptr(), chain_lp.data_ptr(), 1)
    _cabi.mcmc_init_device(mc, state, stats.data_ptr(), diag.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    got = lp.cpu().numpy()
    assert np.all(got[0::2] == -np.inf)
    want = np.zeros(M // 2)
    for v in range(V):                                           # the device's order: series by series
        want = want + st[1:M:2, v, ref.ST_LOGLIK]
    assert np.all(np.isfinite(want)) and np.array_equal(got[1::2], want)


@pytest.mark.parametrize("k", [-10, 10, 20])
def test_scaled_observations(cabi, k):
    """Observations x 2^k (exact): r^2 and Spearman must equal the reference of the UNSCALED observations (both are
    invariant under scaling), every other slot the reference at that scale."""
    from simplyp_b200 import packing as pk
    w = _tarland(67, seed=6)
    obs, desc, labels = pk.obs_arrays(w["obs"], w["topo"], w["index"], None)
    _check(cabi, w, obs * 2.0 ** k, desc, scaled_from=(obs, k))


def test_chunked_calibrate_equals_one_launch(cabi, monkeypatch):
    """Engine.calibrate split into member chunks by max_workspace_bytes (three chunks, the last ragged) equals one
    launch bitwise: on the 5-reach network, and with rank statistics on Tarland."""
    import torch
    from simplyp_b200 import packing as pk
    from simplyp_b200.engine import Engine
    launches = []
    calibrate_device = cabi.calibrate_device

    def counted(dims, *args):
        launches.append(dims.n_members)
        return calibrate_device(dims, *args)
    monkeypatch.setattr(cabi, "calibrate_device", counted)
    eng = Engine(0)
    for kind in ("network5", "tarland"):
        if kind == "network5":
            w = _network("network5", 13)
            obs, desc = _synthetic_obs(cabi, w, [(s, k, None) for k in range(6) for s in (0, 2, 4)])
            S, D = 5, w["forcing"].shape[0]
            per_member, want_chunks = 32 * S * D, [5, 5, 3]
        else:
            w = _tarland(67, seed=7)
            obs, desc, _ = pk.obs_arrays(w["obs"], w["topo"], w["index"], None)
            w["opt"].rank_stats = 1
            per_member, want_chunks = 8 * obs.shape[0] * w["forcing"].shape[0], [30, 30, 7]
        try:
            args = (eng.to_device(w["forcing"]), eng.to_device(w["member"]), eng.to_device(w["sc"]),
                    w["topo"].parent_offsets, w["topo"].parent_ids, eng.to_device(obs), eng.to_device(desc), w["opt"])
            del launches[:]
            one, dg1 = eng.calibrate(*args)
            assert launches == [w["member"].shape[0]], kind
            del launches[:]
            chunked, dgc = eng.calibrate(*args, max_workspace_bytes=want_chunks[0] * per_member)
            torch.cuda.synchronize()
            assert launches == want_chunks, kind                    # the members of each launch
            assert torch.equal(torch.nan_to_num(one, nan=-7.0), torch.nan_to_num(chunked, nan=-7.0)), kind
            assert torch.equal(dg1, dgc), kind
        finally:
            w["opt"].rank_stats = 0


@pytest.mark.parametrize("row", [(-1, 0), ("S", 0), (0, -1), (0, 6)])
def test_bad_obs_desc_is_refused(cabi, row):
    """simplyp_calibrate_host checks every obs_desc row before any device work (a reach outside 0..S-1 was never
    finalised: silent zeros; a kind outside 0..5 read another parameter as its error scale)."""
    w = _network("network5", 2)
    obs, desc = _synthetic_obs(cabi, w, [(0, 0, None), (4, 2, None), (2, 1, None)])
    bad = (5 if row[0] == "S" else row[0], row[1])
    desc[1] = bad
    with pytest.raises(cabi.SimplypError, match="obs_desc row 1"):
        cabi.calibrate_host(w["forcing"], w["member"], w["sc"], w["topo"].parent_offsets, w["topo"].parent_ids, obs,
                            desc, w["opt"])
