"""GPU tier of the ensemble sampler (simplyp_mcmc_*_device, simplyp_b200.mcmc): the kernels against the NumPy
reference sampler, stored log-probabilities against fresh evaluations, graph replay against a hand-driven loop,
continuation, the prior box, and a twin experiment."""
import numpy as np
import pandas as pd
import pytest

from tests import mcmc_reference as ref

pytestmark = pytest.mark.gpu

FREE = {"fc": (100.0, 400.0), "T_g": (20.0, 150.0), "a_Q": (0.2, 0.9), "err_m:Q": (0.05, 1.0)}


@pytest.fixture(scope="module")
def cabi():
    from simplyp_b200 import _cabi
    _cabi.require_device()
    return _cabi


def _setup(kind):
    from simplyp_b200 import packing as pk, tarland
    from tests.golden.networks import network5_inputs
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(dynamic="y")
    priors = dict(FREE)
    if kind == "network5":
        p, p_LU, p_SC, p_struc = network5_inputs(p, p_LU, p_SC, p_struc)
        pk.validate_land_use(p_SC, p["SC_list"])
        obs = {5: obs[1]}
        priors["sc:TDPeff@2"] = (0.0, 0.5)
    return (met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs), priors


def _lp_sum(stats, diag):
    lp = np.zeros(stats.shape[0])
    for v in range(stats.shape[1]):
        lp = lp + stats[:, v, 3]
    lp[np.any(diag[..., 3] != 0, axis=1) | np.isnan(lp)] = -np.inf
    return lp


def test_kernels_equal_reference_sampler(cabi):
    import torch
    W, K, H, n, seed = 64, 5, 32, 100, 0xfeed_0000_0042
    rng = np.random.default_rng(8)
    A = rng.normal(size=(K, K))
    cov, mean = A @ A.T + np.eye(K), rng.normal(size=K)
    sd = np.sqrt(np.diag(cov))
    lo, hi = mean - 2.5 * sd, mean + 2.5 * sd        # some proposals leave the box
    lp_fn = ref.gaussian_lp(mean, cov)
    x0 = mean + rng.uniform(-1, 1, size=(W, K)) * sd
    dev = torch.device("cuda", 0)
    t = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)
    walkers, lp = t(x0), t(np.zeros(W))
    prop, log_z, oob = t(np.zeros((H, K))), t(np.zeros(H)), t(np.zeros(H), torch.int32)
    it, acc = t([0], torch.int64), t(np.zeros(W), torch.int64)
    chain, chain_lp = t(np.zeros((n, W, K))), t(np.zeros((n, W)))
    mem, sc = t(np.zeros((W, 40))), t(np.zeros((1, 1, 16)))
    stats = torch.zeros((W, 1, 10), dtype=torch.float64, device=dev)
    diag = torch.zeros((W, 1, 4), dtype=torch.int64, device=dev)
    mc = cabi.make_mcmc(W, [(cabi.MCMC_MEMBER, k, 0) for k in range(K)], lo, hi, 1, 1, seed=seed)
    st = cabi.make_mcmc_state(walkers.data_ptr(), lp.data_ptr(), prop.data_ptr(), log_z.data_ptr(), oob.data_ptr(),
                              it.data_ptr(), acc.data_ptr(), chain.data_ptr(), chain_lp.data_ptr(), n)
    stream = torch.cuda.current_stream().cuda_stream
    stats[:, 0, 3] = t(lp_fn(x0))
    cabi.mcmc_init_device(mc, st, stats.data_ptr(), diag.data_ptr(), stream)
    for i in range(n):
        for half in (0, 1):
            cabi.mcmc_propose_device(mc, st, half, mem.data_ptr(), sc.data_ptr(), stream)
            y = prop.cpu().numpy()
            rows = mem[half * H:(half + 1) * H, :K].cpu().numpy()
            flags = oob.cpu().numpy().astype(bool)
            assert np.array_equal(rows[~flags], y[~flags])
            stats[:H, 0, 3] = t(lp_fn(y))
            cabi.mcmc_accept_device(mc, st, half, stats.data_ptr(), diag.data_ptr(), stream)
    torch.cuda.synchronize()
    want_chain, want_lp, want_acc, _, _ = ref.sample(lp_fn, x0, lo, hi, n, seed)
    assert np.array_equal(chain.cpu().numpy(), want_chain)
    assert np.array_equal(chain_lp.cpu().numpy(), want_lp)
    assert np.array_equal(acc.cpu().numpy(), want_acc)
    assert int(it.item()) == n and want_acc.sum() > 0


@pytest.mark.parametrize("kind", ["tarland", "network5"])
def test_every_stored_lp_is_a_fresh_evaluation(cabi, kind):
    """Stored lp == Engine.calibrate of the stored states (all of them in one launch) + the box prior (0), bitwise —
    a member's statistics do not depend on launch composition, pilot or placement."""
    from simplyp_b200 import ensemble as ens, mcmc
    args, priors = _setup(kind)
    W, n, seed = 64, 40, 21
    r = mcmc.sample(*args, priors, W, n, seed=seed)
    K = len(priors)
    assert r.chain.shape == (n, W, K) and r.iterations == n
    stats, labels, diag = ens.calibrate_ensemble(*args, r.flat_samples())
    lp = _lp_sum(stats.cpu().numpy(), diag.cpu().numpy())
    assert np.isfinite(r.log_prob).all()
    assert np.array_equal(lp, r.log_prob.ravel())
    b = r.bounds
    assert np.all((r.chain >= b[:, 0]) & (r.chain <= b[:, 1]))
    lhs = ens.latin_hypercube(W, {k: v for k, v in priors.items()}, seed)
    x0 = np.stack([lhs[k] for k in priors], axis=1)
    prev = np.concatenate([x0[None], r.chain[:-1]])
    changes = np.any(r.chain != prev, axis=2).sum(axis=0)
    assert np.array_equal(changes, r.accepted)
    assert 0 < r.acceptance_fraction.mean() < 1


def test_graph_replay_equals_hand_driven_loop(cabi):
    from simplyp_b200 import mcmc
    args, priors = _setup("tarland")
    kw = dict(seed=3, thin=2)
    s = mcmc._Sampler(*args, priors, 32, 12, **kw)
    s.evaluate_all()
    for _ in range(12):
        s.iteration_step()
    hand = s.result()
    graph = mcmc.sample(*args, priors, 32, 12, **kw)
    for f in ("chain", "log_prob", "accepted", "last", "last_log_prob"):
        assert np.array_equal(getattr(hand, f), getattr(graph, f)), f
    assert hand.iterations == graph.iterations == 12 and graph.chain.shape[0] == 6


@pytest.mark.parametrize("thin", [1, 4])
def test_continuation_equals_one_run(cabi, thin):
    from simplyp_b200 import mcmc
    args, priors = _setup("tarland")
    one = mcmc.sample(*args, priors, 32, 50, seed=9, thin=thin)
    a = mcmc.sample(*args, priors, 32, 30, seed=9, thin=thin)
    b = mcmc.sample(*args, priors, 32, 20, seed=9, thin=thin, initial=a, start_iteration=a.iterations)
    assert b.iterations == 50
    assert np.array_equal(np.concatenate([a.chain, b.chain]), one.chain)
    assert np.array_equal(np.concatenate([a.log_prob, b.log_prob]), one.log_prob)
    assert np.array_equal(a.accepted + b.accepted, one.accepted)
    assert np.array_equal(b.last, one.last) and np.array_equal(b.last_log_prob, one.last_log_prob)


def test_rows_handed_to_the_integrator_lie_inside_the_box(cabi):
    import torch
    from simplyp_b200 import mcmc, packing as pk
    args, _ = _setup("tarland")
    priors = {"fc": (280.0, 300.0), "T_g": (60.0, 70.0), "a_Q": (0.45, 0.55), "err_m:Q": (0.4, 0.6)}
    names = list(priors)
    b = np.array([priors[k] for k in names])
    W = 32
    x0 = b[:, 0] + np.random.default_rng(5).uniform(0, 0.02, size=(W, len(names))) * (b[:, 1] - b[:, 0])
    s = mcmc._Sampler(*args, priors, W, 10, seed=4, initial=x0)
    s.evaluate_all()
    cols = [pk.MEMBER_INDEX[k] for k in names]
    n_out = n_all = 0
    for _ in range(10):
        for half in (0, 1):
            s.propose(half)
            rows = s.d_mem[half * s.H:(half + 1) * s.H].cpu().numpy()[:, cols]
            assert np.all((rows >= b[:, 0]) & (rows <= b[:, 1]))
            oob = s.out_of_box.cpu().numpy().astype(bool)
            assert np.all(np.any((s.proposals.cpu().numpy() < b[:, 0]) | (s.proposals.cpu().numpy() > b[:, 1]),
                                 axis=1) == oob)
            n_out += int(oob.sum())
            n_all += oob.size
            s.evaluate(half)
            s.accept(half)
    r = s.result()
    assert np.all((r.chain >= b[:, 0]) & (r.chain <= b[:, 1]))
    assert n_out > 0.25 * n_all, (n_out, n_all)
    torch.cuda.synchronize()


def test_twin_experiment_recovers_the_truth(cabi):
    """Q of a known member with 10 % multiplicative Gaussian noise: the posterior covers the truth."""
    from simplyp_b200 import ensemble as ens, mcmc, model as spm, packing as pk, tarland
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, _ = tarland.load(dynamic="y")
    topo = pk.build_topology(p_struc, p["SC_list"])
    opt = spm.make_options(p_SU, p, dyn, topo)
    out, diag = cabi.run_host(pk.forcing_matrix(met), pk.member_vector(p, p_LU)[None], pk.sc_matrix(p_SC, topo.sc_ids),
                              topo.parent_offsets, topo.parent_ids, opt)
    assert not diag[..., 3].any()
    q = out[0, 0, :, pk.RAW_COLS.index("Qr")] * float(p_SC.loc["A_catch", 1]) * 1000 / 86400
    q_obs = q * (1.0 + 0.1 * np.random.default_rng(2004).normal(size=q.size))
    obs = {1: pd.DataFrame({"Q": q_obs}, index=met.index)}
    truth = {"fc": float(p["fc"]), "T_g": float(p["T_g"]), "alpha": float(p["alpha"])}
    priors = {k: ens.TARLAND_RANGES[k] for k in list(truth) + ["err_m:Q"]}
    r = mcmc.sample(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, priors, 128, 400, variables=("Q",), seed=77)
    post = r.flat_samples(burn=200)
    for k, v in truth.items():
        lo, hi = np.quantile(post[k], [0.025, 0.975])
        assert lo <= v <= hi, (k, v, lo, hi)
    assert 0.08 <= np.median(post["err_m:Q"]) <= 0.12
