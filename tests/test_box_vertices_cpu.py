"""CPU tier: the host build of the quad program (tests/hostemu) against the oracle at vertices of the prior box, under
every combination of the dynamic options, run mode and step length (tests/box_vertices.py: the vertices, the option
matrix and the bound).  Every member must end with status 0 at the default max_steps_per_day, and every daily flow and
concentration must lie within 1e-5 relative above the floor, within the floor's absolute bound below it and, below
it, come closer to the oracle when the member is integrated again at rtol/100, atol/100."""
import numpy as np
import pytest

from simplyp_b200 import ensemble as ens
from tests import box_vertices as bv
from tests import hostemu

N_TARLAND, N_NETWORK, N_SNOW = 16, 6, 12


@pytest.fixture(scope="module")
def pool():
    p = bv.oracle_pool()
    yield p
    p.close()
    p.join()


def _check(case, pool, label):
    out, dg = case.run(hostemu.run_quad)
    assert not np.any(dg[..., 3]), (label, np.nonzero(dg[..., 3]))
    out_t, _ = case.run(hostemu.run_quad, tighten=100.0)
    bv.compare_with_oracle(case, out, bv.oracle_runs(pool, case), label, out_tight=out_t).check()


@pytest.mark.parametrize("k", range(len(bv.OPTIONS)), ids=bv.OPTION_IDS)
def test_tarland_vertices_vs_oracle(pool, k):
    """Tarland 2004: all-low, all-high and 14 seeded vertices of TARLAND_RANGES."""
    case = bv.Case(bv.OPTIONS[k], bv.vertices(N_TARLAND, seed=100 + k))
    _check(case, pool, "tarland " + bv.OPTION_IDS[k])


@pytest.mark.parametrize("k", range(0, len(bv.OPTIONS), 3), ids=bv.OPTION_IDS[::3])
def test_network_vertices_vs_oracle(pool, k):
    """The 5-reach network with per-member sub-catchment rows (sc_params [M][S][NP_SC]): every reach of every member."""
    ranges = {**ens.TARLAND_RANGES, **bv.NETWORK_SC_RANGES}
    case = bv.Case(bv.OPTIONS[k], bv.vertices(N_NETWORK, seed=200 + k, ranges=ranges), network=True)
    assert case.sc.shape[0] == case.M
    _check(case, pool, "network " + bv.OPTION_IDS[k])


@pytest.mark.parametrize("k", [0, 15], ids=[bv.OPTION_IDS[0], bv.OPTION_IDS[15]])
def test_snow_vertices_vs_oracle(pool, k):
    """snow_on_device with D_snow_0 / f_DDSM at the faces of their box (all four corners among the vertices), against
    the oracle on the forcing snow_hydrol_inputs makes on the host with each member's own snow parameters."""
    ranges = {**ens.TARLAND_RANGES, **bv.SNOW_RANGES}
    samples = bv.vertices(N_SNOW, seed=300 + k, ranges=ranges)
    samples["D_snow_0"][:4], samples["f_DDSM"][:4] = [0.0, 0.0, 40.0, 40.0], [1.0, 4.0, 1.0, 4.0]
    case = bv.Case(bv.OPTIONS[k], samples, snow=True)
    _check(case, pool, "snow " + bv.OPTION_IDS[k])
