"""GPU tier: the device at vertices of the prior box (tests/box_vertices.py), every vertex of a combination of options in
ONE launch so that lock-step warps mix the heaviest members, against the oracle under the bound of box_vertices and
against the host build of the same program (tests/hostemu: what the CPU tier finds about it holds on the device):
outputs within the same bound, step attempts within STEP_RATIO.  Then the vertices planted among 10^4 Latin-hypercube
members (cost pilot, planned placement, warps led by one heavy member) must give the bits of their runs alone."""
import numpy as np
import pytest

from simplyp_b200 import ensemble as ens
from tests import box_vertices as bv
from tests import hostemu
from tests.test_box_vertices_cpu import N_NETWORK, N_SNOW, N_TARLAND

pytestmark = pytest.mark.gpu

# Device and host build differ in the last bits (FMA contraction, sp_rcp / sp_div), which can flip an accept/reject
# decision; over a year of ~5,000 attempts per member that moves the count by far less than this ratio.
STEP_RATIO = 1.05


@pytest.fixture(scope="module")
def cabi():
    from simplyp_b200 import _cabi
    _cabi.require_device()
    return _cabi


@pytest.fixture(scope="module")
def pool():
    p = bv.oracle_pool()
    yield p
    p.close()
    p.join()


def _check(cabi, case, pool, label, out=None, dg=None):
    if out is None:
        out, dg = case.run(cabi.run_host)
    assert np.all(np.isfinite(out)) and not np.any(dg[..., 3]), (label, np.nonzero(dg[..., 3]))
    out_t, _ = case.run(cabi.run_host, tighten=100.0)
    bv.compare_with_oracle(case, out, bv.oracle_runs(pool, case), "device " + label, out_tight=out_t).check()
    out_h, dg_h = case.run(hostemu.run_quad)
    host = [{SC: r[bv.FLOW_CONC_COLS].to_numpy(float) for SC, r in case.frames(out_h[i], i).items()}
            for i in range(case.M)]
    bv.compare_with_oracle(case, out, host, "device vs host build " + label).check()
    ratio = dg[..., 0] / dg_h[..., 0]
    print("%s: step attempts device / host build %.4f ... %.4f" % (label, ratio.min(), ratio.max()))
    assert np.all(ratio <= STEP_RATIO) and np.all(ratio >= 1.0 / STEP_RATIO), label


@pytest.mark.parametrize("k", range(len(bv.OPTIONS)), ids=bv.OPTION_IDS)
def test_tarland_vertices_on_device(cabi, pool, k):
    case = bv.Case(bv.OPTIONS[k], bv.vertices(N_TARLAND, seed=100 + k))
    _check(cabi, case, pool, "tarland " + bv.OPTION_IDS[k])


@pytest.mark.parametrize("k", range(0, len(bv.OPTIONS), 3), ids=bv.OPTION_IDS[::3])
def test_network_vertices_on_device(cabi, pool, k, monkeypatch):
    """Per-member sub-catchment rows on the 5-reach network, in one piece and swept in epochs of 128 days (the
    midnight state of every reach handed over twice in 2004): the same bits, and within the bound."""
    ranges = {**ens.TARLAND_RANGES, **bv.NETWORK_SC_RANGES}
    case = bv.Case(bv.OPTIONS[k], bv.vertices(N_NETWORK, seed=200 + k, ranges=ranges), network=True)
    monkeypatch.setenv("SIMPLYP_EPOCH_DAYS", "0")
    out, dg = case.run(cabi.run_host)
    monkeypatch.setenv("SIMPLYP_EPOCH_DAYS", "128")
    out_e, dg_e = case.run(cabi.run_host)
    assert np.array_equal(out, out_e) and np.array_equal(dg, dg_e)
    _check(cabi, case, pool, "network " + bv.OPTION_IDS[k], out_e, dg_e)


@pytest.mark.parametrize("k", [0, 15], ids=[bv.OPTION_IDS[0], bv.OPTION_IDS[15]])
def test_snow_vertices_on_device(cabi, pool, k):
    ranges = {**ens.TARLAND_RANGES, **bv.SNOW_RANGES}
    samples = bv.vertices(N_SNOW, seed=300 + k, ranges=ranges)
    samples["D_snow_0"][:4], samples["f_DDSM"][:4] = [0.0, 0.0, 40.0, 40.0], [1.0, 4.0, 1.0, 4.0]
    _check(cabi, bv.Case(bv.OPTIONS[k], samples, snow=True), pool, "snow " + bv.OPTION_IDS[k])


def test_vertices_planted_in_a_large_ensemble(cabi):
    """32 vertices written over members of the 10^4-member Latin-hypercube ensemble bench.py times (dynamic options on,
    'cal', step 1): at the first and last ranks, at block and warp edges and spread over the rest.  The launch runs the
    8-day cost pilot, the planned placement and 100 warps led by one heavy member; each vertex must give the bits of
    its run alone (outputs and counters)."""
    M = 10000
    samples = ens.latin_hypercube(M, seed=20260101)
    verts = bv.vertices(32, seed=400)
    at = np.array([0, 1, 7, 8, 31, 32, 33, 63, 64, 255, 256, 1000, 2047, 2048, 3001, 4095, 4096, 5000, 5031, 5032,
                   6000, 6543, 7001, 8191, 8192, 9000, 9500, 9967, 9968, 9990, 9998, 9999])
    for name, vals in verts.items():
        samples[name][at] = vals
    case = bv.Case(bv.OPTIONS[0], samples)
    out, dg = case.run(cabi.run_host)
    assert not np.any(dg[..., 3])
    for j in at:
        out1, dg1 = case.run(cabi.run_host, members=[int(j)])
        assert np.array_equal(out1[0], out[j]) and np.array_equal(dg1[0], dg[j]), int(j)
    spd = dg[:, 0, 0] / len(case.met)
    print("planted vertices: attempts per day %.1f ... %.1f, ensemble median %.1f"
          % (spd[at].min(), spd[at].max(), float(np.median(spd))))

