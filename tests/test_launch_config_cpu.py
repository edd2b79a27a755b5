"""CPU tier: the launch policy of the quad kernel (launch_config() and read_launch_overrides() in simplyp_plan.cuh,
compiled for the host by tests/hostemu) against a restatement of the rules it was moved from.

The policy decides whether a cost pilot runs, which register variant (resident blocks per SM) every launch uses, the
planned placement of an ensemble and the epochs of a network.  None of this shows in the results, so these tests are
what pins it."""
import re

import pytest

from tests import hostemu

OVERRIDES = ("SIMPLYP_QUAD_MINBLOCKS", "SIMPLYP_PILOT_MINBLOCKS", "SIMPLYP_SM_PLAN", "SIMPLYP_PLAN_QMAX",
             "SIMPLYP_SOLO_WARPS", "SIMPLYP_EPOCH_DAYS", "SIMPLYP_NET_MINBLOCKS")
TILE = 128                # FORC_TILE: days per forcing tile
PLAN_MAX_SM = 1024


def atoi(s):
    m = re.match(r"[ \t\n\v\f\r]*([+-]?[0-9]+)", s)
    return int(m.group(1)) if m else 0


def cdiv(a, b):
    """C integer division (truncates toward zero)."""
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b > 0) else -q


def plan_shape(B, n_sm, resident):
    if n_sm <= 0 or B <= n_sm or B >= 3 * n_sm:
        return None
    Q = B - 2 * n_sm if B > 2 * n_sm else 0
    nY = n_sm - Q
    nP = B - nY - 3 * Q
    if nY <= 0 or nP <= 0 or nP > nY:
        return None
    res = 3 if resident == 3 and Q > 0 else 2
    return dict(nY=nY, nP=nP, Q=Q, resident=res, n_launch=3 * n_sm if res == 3 else n_sm + nP + Q)


def expected(M, D, n_sm, env, network=False, n_levels=0, grid_one_epoch=0, pilot_days=0, workspace=True):
    """The rules as the launcher applied them before they moved into launch_config()."""
    cfg = dict.fromkeys(hostemu.LAUNCH_CONFIG_FIELDS, 0)

    def quad_minblocks(grid):
        if "SIMPLYP_QUAD_MINBLOCKS" in env and 2 <= atoi(env["SIMPLYP_QUAD_MINBLOCKS"]) <= 4:
            return atoi(env["SIMPLYP_QUAD_MINBLOCKS"])
        return 2 if grid <= 2 * n_sm else 3 if grid <= 9 * n_sm else 4

    if not network:
        grid = ((M + 7) // 8 * 8 + 31) // 32
        cfg.update(grid=grid, minb=quad_minblocks(grid))
        # order_members_by_cost
        days = pilot_days if pilot_days > 0 else 8
        if pilot_days < 0 or not workspace or M < 512 or D < 8 * days:
            return cfg
        grid = (M + 31) // 32
        pilot_minb = quad_minblocks(grid)
        if pilot_minb == 2 and n_sm > 0 and grid > 2 * n_sm:
            pilot_minb = 3
        if "SIMPLYP_PILOT_MINBLOCKS" in env and 2 <= atoi(env["SIMPLYP_PILOT_MINBLOCKS"]) <= 4:
            pilot_minb = atoi(env["SIMPLYP_PILOT_MINBLOCKS"])
        cfg.update(pilot_days=days, pilot_minb=pilot_minb)
        minb = quad_minblocks(grid)
        q_max = atoi(env["SIMPLYP_PLAN_QMAX"]) if "SIMPLYP_PLAN_QMAX" in env else n_sm - 1
        shape = plan_shape(grid, n_sm, minb)
        if ((minb == 2 or (minb == 3 and grid <= 2 * n_sm + q_max)) and n_sm <= PLAN_MAX_SM and M >= 2048
                and not ("SIMPLYP_SM_PLAN" in env and atoi(env["SIMPLYP_SM_PLAN"]) == 0) and shape):
            solo = M // 100 // 4 * 4
            if "SIMPLYP_SOLO_WARPS" in env and atoi(env["SIMPLYP_SOLO_WARPS"]) >= 0:
                solo = atoi(env["SIMPLYP_SOLO_WARPS"])
            cfg.update(plan=1, solo=solo, grid=shape["n_launch"],
                       **{k: shape[k] for k in ("nY", "nP", "Q", "resident")})
        return cfg
    # launch_levels, network
    grid = grid_one_epoch
    epoch_days = max(2 * TILE, (4 * n_levels + TILE - 1) // TILE * TILE)
    if grid <= n_sm:
        epoch_days = 0
    if "SIMPLYP_EPOCH_DAYS" in env:
        epoch_days = cdiv(atoi(env["SIMPLYP_EPOCH_DAYS"]), TILE) * TILE
    n_epochs = -(-D // epoch_days) if epoch_days > 0 else 0
    if epoch_days > 0 and D > epoch_days and grid * n_epochs < 2 ** 30:
        cfg.update(epoch_days=epoch_days, n_epochs=n_epochs)
        grid *= n_epochs
    minb = 3 if grid_one_epoch >= 6 * n_sm else 2
    if "SIMPLYP_NET_MINBLOCKS" in env and atoi(env["SIMPLYP_NET_MINBLOCKS"]) in (2, 3):
        minb = atoi(env["SIMPLYP_NET_MINBLOCKS"])
    cfg.update(grid=grid, minb=minb)
    return cfg


def ensemble_cases(n_sm):
    q_max = n_sm - 1
    Ms = {10 ** 4, 10 ** 6}
    for t in (512, 2048, n_sm * 32, 2 * n_sm * 32, (2 * n_sm + q_max) * 32, 9 * n_sm * 32):
        Ms |= {t - 1, t, t + 1}
    for M in sorted(Ms):
        for pilot_days in (-1, 0, 3, 40):
            days = pilot_days if pilot_days > 0 else 8
            for D in (8 * days - 1, 8 * days, 8 * days + 1, 366):
                for workspace in (True, False):
                    yield dict(M=M, D=D, n_sm=n_sm, pilot_days=pilot_days, workspace=workspace)


def network_cases(n_sm):
    # 2**27 blocks: 7 epochs stay under the 2**30-block cap, 8 reach it
    for grid in (n_sm, n_sm + 1, 6 * n_sm - 1, 6 * n_sm, 2 ** 27):
        for n_levels in (1, 32, 487):
            E = max(2 * TILE, (4 * n_levels + TILE - 1) // TILE * TILE)
            for D in (E - 1, E, E + 1, 7 * E, 8 * E, 10958):
                yield dict(M=8, D=D, n_sm=n_sm, network=True, n_levels=n_levels, grid_one_epoch=grid)


def check(cases, env):
    n = 0
    for case in cases:
        got = hostemu.launch_config(**case)
        assert got == expected(env=env, **case), case
        n += 1
    assert n > 0


@pytest.fixture
def no_overrides(monkeypatch):
    for name in OVERRIDES:
        monkeypatch.delenv(name, raising=False)
    return monkeypatch


@pytest.mark.parametrize("n_sm", [60, 132, 148])     # on 60 SMs the plan's floor of 2048 members is what decides
def test_policy_equals_the_rules(no_overrides, n_sm):
    check(ensemble_cases(n_sm), {})
    check(network_cases(n_sm), {})


# valid and ignored values of every override (atoi: leading blanks and trailing junk are accepted, no digits read 0)
OVERRIDE_VALUES = {
    "SIMPLYP_QUAD_MINBLOCKS": ["2", "3", "4", " 3", "4x", "1", "5", "x", ""],
    "SIMPLYP_PILOT_MINBLOCKS": ["2", "3", "4", "1", "5", "x"],
    "SIMPLYP_SM_PLAN": ["0", "x", "", "1", "2"],
    "SIMPLYP_PLAN_QMAX": ["0", "16", "17", "147", "-5", "x"],
    "SIMPLYP_SOLO_WARPS": ["0", "24", "240", "-1", "x"],
    "SIMPLYP_EPOCH_DAYS": ["0", "127", "128", "200", "512", "-300", "x"],
    "SIMPLYP_NET_MINBLOCKS": ["2", "3", "1", "4", "x"],
}


@pytest.mark.parametrize("name,value", [(k, v) for k, vs in OVERRIDE_VALUES.items() for v in vs])
def test_overrides(no_overrides, name, value):
    no_overrides.setenv(name, value)
    for n_sm in (132, 148):
        check(ensemble_cases(n_sm), {name: value})
        check(network_cases(n_sm), {name: value})


def test_bench_workloads(no_overrides):
    """What the benchmark's workloads get on a 148-SM B200."""
    # config 2: 10^4 members of Tarland 2004 (366 days)
    c = hostemu.launch_config(M=10 ** 4, D=366, n_sm=148)
    assert (c["pilot_days"], c["pilot_minb"]) == (8, 3)
    assert (c["minb"], c["plan"], c["resident"], c["grid"], c["solo"]) == (3, 1, 3, 444, 100)
    assert (c["nY"], c["nP"], c["Q"]) == (131, 131, 17)
    # config 4: 10^6 members
    c = hostemu.launch_config(M=10 ** 6, D=366, n_sm=148)
    assert (c["minb"], c["plan"], c["grid"], c["pilot_days"], c["pilot_minb"]) == (4, 0, 31250, 8, 4)
    # config 3: 256 reaches on 32 levels, 64 members (512 blocks per epoch), 10958 days
    c = hostemu.launch_config(M=64, D=10958, n_sm=148, network=True, n_levels=32, grid_one_epoch=512)
    assert (c["minb"], c["epoch_days"], c["n_epochs"], c["grid"]) == (2, 256, 43, 43 * 512)
    # config 5: 4096 reaches on 487 levels, 8 members (1024 blocks per epoch), 18262 days
    c = hostemu.launch_config(M=8, D=18262, n_sm=148, network=True, n_levels=487, grid_one_epoch=1024)
    assert (c["minb"], c["epoch_days"], c["n_epochs"], c["grid"]) == (3, 2048, 9, 9 * 1024)
