"""CPU tier of the ensemble sampler: the host build of simplyp_mcmc.cuh against the NumPy reference sampler
(tests/mcmc_reference.py), the reference sampler on a known target, the input checks of mcmc.sample and the
autocorrelation estimate."""
import numpy as np
import pytest

from tests import mcmc_reference as ref

KAT = [  # Random123 known-answer vectors of Philox4x32-10: counter, key, result
    ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
     [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
]


@pytest.fixture(scope="module")
def host():
    from tests import mcmc_host
    mcmc_host.load()
    return mcmc_host


def _mc(W, K, lo, hi, seed, stretch=2.0):
    from simplyp_b200 import _cabi
    return _cabi.make_mcmc(W, [(_cabi.MCMC_MEMBER, k, 0) for k in range(K)], lo, hi, 1, 1, seed=seed, stretch=stretch)


def test_philox_known_answers_and_numpy_restatement(host):
    for ctr, key, want in KAT:
        assert ref.philox4x32_10([ctr], key)[0].tolist() == want
        assert host.philox([ctr], key)[0].tolist() == want
    rng = np.random.default_rng(1)
    ctr = rng.integers(0, 2 ** 32, size=(10000, 4), dtype=np.uint64).astype(np.uint32)
    key = rng.integers(0, 2 ** 32, size=(10000, 2), dtype=np.uint64).astype(np.uint32)
    assert np.array_equal(host.philox(ctr, key), ref.philox4x32_10(ctr, key))


def test_host_propose_and_accept_equal_reference(host):
    """Proposals bit for bit, ln z within 1 ulp, the same decisions — over iterations with both halves, a seed with
    a high word and a box that some proposals leave."""
    W, K, seed = 64, 5, 0x1234_5678_9abc_def0
    lo, hi = np.full(K, -3.0), np.full(K, 3.0)
    mc = _mc(W, K, lo, hi, seed, stretch=2.5)
    lp_fn = ref.gaussian_lp(np.zeros(K), np.eye(K) + 0.5)
    x = np.random.default_rng(2).uniform(-2, 2, size=(W, K))
    xh, lp, lph = x.copy(), lp_fn(x), lp_fn(x)
    acc, acch = np.zeros(W, np.int64), np.zeros(W, np.int64)
    n_oob = n_acc = 0
    for t in (0, 1, 7, 2 ** 32 + 3):
        for half in (0, 1):
            y, lz, oob = ref.propose(x, t, half, seed, lo, hi, a=2.5)
            yh, lzh, oobh = host.propose(mc, xh, t, half)
            assert np.array_equal(y.view(np.int64), yh.view(np.int64))
            assert np.all(np.abs(lz.view(np.int64) - lzh.view(np.int64)) <= 1)
            assert np.array_equal(oob, oobh.astype(bool))
            lp_new = lp_fn(y)
            lp_new[oob] = -np.inf
            ok = ref.accept(x, lp, acc, y, lz, lp_new, t, half, seed)
            okh = host.accept(mc, t, half, lp_new, lzh, yh, xh, lph, acch)
            assert np.array_equal(ok, okh.astype(bool))
            n_oob += int(oob.sum())
            n_acc += int(ok.sum())
    assert np.array_equal(x, xh) and np.array_equal(lp, lph) and np.array_equal(acc, acch)
    assert n_oob > 0 and n_acc > 0


def test_reference_sampler_recovers_a_correlated_gaussian():
    K = 5
    rng = np.random.default_rng(3)
    A = rng.normal(size=(K, K))
    cov = A @ A.T + 0.5 * np.eye(K)
    mean = rng.normal(size=K) * 3
    sd = np.sqrt(np.diag(cov))
    lo, hi = mean - 50 * sd, mean + 50 * sd
    x0 = mean + rng.normal(size=(64, K)) * sd * 0.1
    chain, chain_lp, acc, _, _ = ref.sample(ref.gaussian_lp(mean, cov), x0, lo, hi, 4000, seed=11)
    s = chain[1000:].reshape(-1, K)
    assert np.all(np.abs(s.mean(axis=0) - mean) <= 0.1 * sd)
    c = np.cov(s.T)
    assert np.all(np.abs(c - cov) <= 0.1 * np.sqrt(np.outer(np.diag(cov), np.diag(cov))))
    assert 0.2 < acc.mean() / 4000 < 0.7


def test_autocorr_time_of_ar1():
    from simplyp_b200.mcmc import autocorr_time
    rho, n_t, n_w = 0.9, 20000, 16
    rng = np.random.default_rng(4)
    e = rng.normal(size=(n_t, n_w)) * np.sqrt(1 - rho ** 2)
    x = np.zeros((n_t, n_w))
    x[0] = rng.normal(size=n_w)
    for i in range(1, n_t):
        x[i] = rho * x[i - 1] + e[i]
    tau = autocorr_time(x[:, :, None])
    assert tau.shape == (1,)
    assert abs(tau[0] - 19.0) <= 0.15 * 19.0


def _tarland():
    from simplyp_b200 import tarland
    return tarland.load(dynamic="y")


@pytest.mark.parametrize("priors, W, kw, match", [
    ({"nope": (0, 1)}, 8, {}, "unknown"),
    ({"sc:nope": (0, 1)}, 8, {}, "unknown"),
    ({"sc:TDPeff@1": (0, 1)}, 8, {}, "position"),
    ({"fc": (200.0, 100.0)}, 8, {}, "lo < hi"),
    ({"fc": (100.0, 100.0)}, 8, {}, "lo < hi"),
    ({"fc": (100.0, np.inf)}, 8, {}, "finite"),
    ({"fc": (np.nan, 1.0)}, 8, {}, "finite"),
    ({"fc": (100.0, 400.0)}, 7, {}, "even"),
    ({"fc": (100.0, 400.0), "T_g": (20.0, 150.0)}, 2, {}, "twice"),
    ({"d_maxE_spr": (60.0, 120.0)}, 8, {}, "integer"),
    ({"d_maxE_aut": (200.0, 300.0)}, 8, {}, "integer"),
    ({"sc:f_Ar": (0.1, 0.3)}, 8, {}, "land-use"),
    ({"sc:f_IG": (0.1, 0.3)}, 8, {}, "land-use"),
    ({"sc:f_S": (0.1, 0.3)}, 8, {}, "land-use"),
    ({"sc:f_NC_Ar@0": (0.1, 0.3)}, 8, {}, "land-use"),
    ({"sc:f_NC_IG": (0.1, 0.3)}, 8, {}, "land-use"),
    ({"sc:f_NC_S": (0.1, 0.3)}, 8, {}, "land-use"),
    ({"D_snow_0": (0.0, 10.0)}, 8, {}, "snow_on_device"),
    ({"f_DDSM": (1.0, 4.0)}, 8, {}, "snow_on_device"),
    ({"fc": (100.0, 400.0)}, 8, {"initial": np.full((8, 1), 500.0)}, "inside"),
    ({"fc": (100.0, 400.0)}, 8, {"initial": np.full((6, 1), 200.0)}, "shape"),
    ({"fc": (100.0, 400.0)}, 8, {"thin": 0}, "thin"),
    ({"fc": (100.0, 400.0)}, 8, {"stretch": 1.0}, "stretch"),
])
def test_sample_rejects_bad_input_before_device_work(priors, W, kw, match, monkeypatch):
    from simplyp_b200 import engine, mcmc

    def no_device(*a, **k):
        raise AssertionError("device work before the input check")
    monkeypatch.setattr(engine, "Engine", no_device)
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = _tarland()
    with pytest.raises(ValueError, match=match):
        mcmc.sample(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, priors, W, 10, **kw)


def test_tarland_ranges_are_accepted_as_priors():
    from simplyp_b200 import ensemble as ens, mcmc
    names, targets, bounds = mcmc._check_priors(ens.TARLAND_RANGES, 1, False)
    assert names == list(ens.TARLAND_RANGES) and len(targets) == 18
    assert bounds.tolist() == [list(v) for v in ens.TARLAND_RANGES.values()]


def test_flat_samples_feed_pack_members():
    from simplyp_b200 import ensemble as ens, mcmc, packing as pk
    chain = np.arange(3 * 4 * 2, dtype=np.float64).reshape(3, 4, 2)
    r = mcmc.McmcResult(chain=chain, log_prob=np.zeros((3, 4)), accepted=np.zeros(4, np.int64),
                        names=["fc", "sc:TDPeff@0"], bounds=np.array([[0, 100.0], [0, 100.0]]), iterations=3,
                        n_steps=3, last=chain[-1], last_log_prob=np.zeros(4))
    s = r.flat_samples(burn=1)
    assert s["fc"].tolist() == chain[1:, :, 0].ravel().tolist()
    member, sc = ens.pack_members(np.zeros(pk.NP_MEMBER), np.zeros((1, pk.NP_SC)), s)
    assert member[:, pk.MEMBER_INDEX["fc"]].tolist() == s["fc"].tolist()
    assert sc[:, 0, pk.SC_INDEX["TDPeff"]].tolist() == s["sc:TDPeff@0"].tolist()
    assert r.acceptance_fraction.shape == (4,)


def test_mcmc_entry_points_raise_without_device():
    import ctypes as C
    from simplyp_b200 import _cabi
    lib = _cabi.load()
    if lib.simplyp_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    mc = _mc(8, 2, [0, 0], [1, 1], 0)
    st = _cabi.make_mcmc_state(*([8] * 9), 1)
    for call in (lambda: _cabi.mcmc_propose_device(mc, st, 0, 8, 8, None),
                 lambda: _cabi.mcmc_accept_device(mc, st, 1, 8, 8, None),
                 lambda: _cabi.mcmc_init_device(mc, st, 8, 8, None)):
        with pytest.raises(_cabi.SimplypError):
            call()
    # the library itself answers SIMPLYP_ENODEVICE (the wrapper's own device check aside)
    assert lib.simplyp_mcmc_propose_device(C.byref(mc), C.byref(st), 0, 8, 8, None) == -2
    assert lib.simplyp_mcmc_accept_device(C.byref(mc), C.byref(st), 0, 8, 8, None) == -2
    assert lib.simplyp_mcmc_init_device(C.byref(mc), C.byref(st), 8, 8, None) == -2
    bad = _mc(8, 2, [0, 0], [1, 1], 0)
    bad.n_walkers = 3
    assert lib.simplyp_mcmc_init_device(C.byref(bad), C.byref(st), 8, 8, None) == -1
