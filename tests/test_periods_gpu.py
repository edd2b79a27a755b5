"""GPU tier of the period aggregates (simplyp_period_aggregates_device, ensemble.period_statistics): the kernel on the
library's own full output against the host build, reach means against the predictive draws and water-body loads
against Engine.sum_to_waterbody bitwise, chunking, failed members, the quantiles of the returned values, graph
capture and the memory check."""
import warnings

import numpy as np
import pytest

from tests import fit_stats_reference as ref
from tests.test_bands_gpu import _ensemble, _run

pytestmark = pytest.mark.gpu

ALL_STATS = [(k, st) for k in range(6) for st in range(3) if not (st == 2 and k == 0)]


@pytest.fixture(scope="module")
def eng():
    from simplyp_b200.engine import Engine
    return Engine()


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def _aggregate(eng, d, out, diag, desc, bounds, wb):
    import torch
    M = out.shape[0]
    values = torch.full((len(desc) * len(bounds), M), -7.0, dtype=torch.float64, device=eng.device)
    eng.period_aggregates(out, d["mem"], d["sc"], diag, np.asarray(desc, dtype=np.int32),
                          np.asarray(bounds, dtype=np.int32), np.asarray(wb, dtype=np.int32), values)
    return values.cpu().numpy()


def _check_against_host(got, want, desc, n_periods):
    """Bitwise, except reach means: sim_series_value forms its quotients with a reciprocal and one fma on the device
    and with IEEE division on the host (simplyp_core.cuh sp_div), which can differ in the last bit."""
    assert np.array_equal(np.isnan(got), np.isnan(want))
    for v, (t, _, st) in enumerate(desc):
        g, w = got[v * n_periods:(v + 1) * n_periods], want[v * n_periods:(v + 1) * n_periods]
        if st == 0 and t >= 0:
            ok = ~np.isnan(w)
            assert np.all(np.abs(g[ok] - w[ok]) <= ref.SIM_ULPS * ref.EPS * np.abs(w[ok])), (t, st)
        else:
            assert _same(g, w), desc[v]


@pytest.mark.parametrize("kind", ["tarland", "network5"])
def test_kernel_equals_host_build(eng, kind):
    from tests import periods_host
    from simplyp_b200 import ensemble as ens
    w = _ensemble(kind, 96 if kind == "network5" else 256)
    d, out, diag = _run(eng, w)
    wb, reaches = ([2, 3, 4], [2, 4]) if kind == "network5" else ([0], [0])
    desc = [(t, k, st) for t in reaches + [-1] for k, st in ALL_STATS]
    bounds, _ = ens.period_bounds(w["inputs"][0].index, "month")
    bounds = np.concatenate([bounds, [[0, out.shape[2] - 1], [40, 200]]]).astype(np.int32)
    got = _aggregate(eng, d, out, diag, desc, bounds, wb)
    want = periods_host.aggregate(out.cpu().numpy(), w["member"], w["sc"], diag.cpu().numpy(), desc, bounds, wb)
    assert np.isfinite(got).mean() > 0.9
    _check_against_host(got, want, desc, len(bounds))


def test_reach_mean_equals_draws_and_waterbody_load_equals_sum_to_waterbody(eng):
    import torch
    from simplyp_b200 import ensemble as ens
    w = _ensemble("network5", 64)
    d, out, diag = _run(eng, w)
    bounds, _ = ens.period_bounds(w["inputs"][0].index, "month")
    wb = [2, 3, 4]
    desc = [(4, k, 0) for k in range(6)] + [(-1, k, 1) for k in range(6)] + [(-1, k, 0) for k in range(6)]
    got = _aggregate(eng, d, out, diag, desc, bounds, wb)
    P, (M, S, D) = len(bounds), out.shape[:3]
    draws = torch.empty((6, D, M), dtype=torch.float64, device=eng.device)
    eng.predictive_draws(out, d["mem"], d["sc"], diag, eng.to_device(np.array([(4, k) for k in range(6)], np.int32)),
                         draws, 0, False, 0)
    x = draws.cpu().numpy()
    wbc = eng.sum_to_waterbody(out, d["mem"], d["sc"], wb).cpu().numpy()           # [M][D][11]
    flux_col = [None, 1, 2, 3, 8, 10]
    value_col = [0, 4, 5, 6, 7, 9]
    for p, (a, b) in enumerate(bounds):
        for k in range(6):
            s_mean, s_load, s_wmean = np.zeros(M), np.zeros(M), np.zeros(M)
            for dd in range(a, b + 1):
                s_mean = s_mean + x[k, dd]
                s_load = s_load + (wbc[:, dd, 0] * 86400.0 if k == 0 else wbc[:, dd, flux_col[k]])
                s_wmean = s_wmean + wbc[:, dd, value_col[k]]
            n = np.float64(b - a + 1)
            assert _same(got[k * P + p], s_mean / n)
            assert _same(got[(6 + k) * P + p], s_load)
            assert _same(got[(12 + k) * P + p], s_wmean / n)


def test_chunking_and_repetition_change_no_bit(eng):
    from simplyp_b200 import ensemble as ens
    M = 23
    w = _ensemble("tarland", M, years=("2004-01-01", "2005-06-30"))
    series = [(1, "Q", "load"), (1, "TDP", "fwmc"), (1, "TP", "mean"), (1, "SRP", "load")]
    runs = [ens.period_statistics(*w["inputs"], w["samples"], series, periods="month", members_per_chunk=c,
                                  engine=eng) for c in (1, 7, M, M)]
    for r in runs[1:]:
        for f in ("values", "quantiles", "mean", "count"):
            assert np.array_equal(getattr(r, f), getattr(runs[0], f), equal_nan=True)
    r = runs[0]
    assert r.values.shape == (4 * 18, M) and r.n_days.tolist()[:3] == [31, 29, 31]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        assert _same(r.quantiles, np.nanquantile(r.values, r.q, axis=-1))
    assert np.array_equal(r.count, np.sum(~np.isnan(r.values), axis=-1))
    ok = r.count > 0
    assert np.allclose(r.mean[ok], np.nanmean(r.values[ok], axis=-1), rtol=1e-13, atol=0)


def test_failed_members_give_nan_and_are_counted(eng):
    from simplyp_b200 import ensemble as ens
    M = 128
    w = _ensemble("tarland", M, extra={"T_s:A": (1.0, 8.0), "E_M": (300.0, 3000.0)})
    met, p_struc, p_SU, p_LU, p_SC, p, dyn = w["inputs"]
    d = dict(forc=eng.to_device(w["forcing"]), mem=eng.to_device(w["member"]), sc=eng.to_device(w["sc"]))
    for steps in (2, 3, 4, 6, 8, 12, 16, 24, 32):
        w["opt"].max_steps_per_day = steps
        out, diag = eng.run(d["forc"], d["mem"], d["sc"], w["topo"].parent_offsets, w["topo"].parent_ids, w["opt"])
        failed = np.any(diag.cpu().numpy()[:, :, 3] != 0, axis=1)
        if 0 < failed.sum() < M:
            break
    else:
        pytest.fail("no max_steps_per_day failed some members but not all")
    got = _aggregate(eng, d, out, diag, [(0, 2, 1), (0, 0, 0)], [[0, 100], [101, 365]], [])
    assert np.all(np.isnan(got[:, failed])) and not np.any(np.isnan(got[:, ~failed]))
    import simplyp_b200.model as spm
    orig = spm.make_options

    def capped(*a, **k):
        o = orig(*a, **k)
        o.max_steps_per_day = steps
        return o
    spm.make_options = capped
    try:
        r = ens.period_statistics(met, p_struc, p_SU, p_LU, p_SC, p, dyn, w["samples"], [(1, "TDP", "load")],
                                  periods="all", engine=eng)
    finally:
        spm.make_options = orig
    assert r.n_failed == int(failed.sum())
    assert np.array_equal(np.isnan(r.values[0]), failed) and r.count[0] == M - failed.sum()


def test_entry_point_captures_into_a_graph(eng):
    import torch
    from simplyp_b200 import ensemble as ens
    w = _ensemble("network5", 64, years=("2004-01-01", "2004-06-30"))
    d, out, diag = _run(eng, w)
    desc = np.array([(-1, 4, 1), (4, 2, 2), (2, 5, 0)], dtype=np.int32)
    bounds, _ = ens.period_bounds(w["inputs"][0].index, "month")
    wb = np.array([2, 3, 4], dtype=np.int32)
    values = torch.empty((3 * len(bounds), 64), dtype=torch.float64, device=eng.device)
    eng.period_aggregates(out, d["mem"], d["sc"], diag, desc, bounds, wb, values)
    torch.cuda.synchronize()
    direct = values.cpu().numpy()
    values.fill_(0)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        eng.period_aggregates(out, d["mem"], d["sc"], diag, desc, bounds, wb, values)
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(direct, values.cpu().numpy(), equal_nan=True)


def test_over_budget_values_refused_before_any_launch(eng):
    from simplyp_b200 import _cabi, ensemble as ens
    from simplyp_b200.engine import Engine

    class Small(Engine):
        def free_bytes(self):
            return 1 << 20
    w = _ensemble("tarland", 4000)
    n0 = _cabi.launch_count()
    with pytest.raises(ValueError, match="thin"):
        ens.period_statistics(*w["inputs"], w["samples"], [(1, "Q", "load"), (1, "TDP", "fwmc")], periods="month",
                              engine=Small())
    assert _cabi.launch_count() == n0
