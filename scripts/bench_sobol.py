"""Timing of the Sobol' sensitivity analysis (sensitivity.sobol_indices) on one GPU: one JSON line per case.

Per case, after one warm-up pass, CUDA events time the phases of a second pass: the design kernel, the integration
(one fused-statistics ``Engine.calibrate`` for objectives; chunked ``Engine.run`` for series), the outputs kernel or
the draw kernel, the point estimates (the indices entry point with n_boot = 0) and the whole indices entry point with
the bootstrap (its difference to the former is the bootstrap).  Beside them, a host NumPy restatement of the
estimators and the bootstrap runs on the same Y with a host clock, over the first rows only; its per-row time is
scaled to all rows.  The card's name and power limit are read in the same run.

    python scripts/bench_sobol.py [--out lines.jsonl] [--host-rows 2]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 20260103
OBJ = ["NSE", "log_NSE", "loglik", "r2", "pbias", "nRMSD", "SSE", "lp"]


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def host_indices(y, K, P, n_boot, picks):
    """NumPy restatement of the point estimates and the bootstrap of one row (all samples finite)."""
    U = y.reshape(-1, P)
    c = U.mean()
    X = U - c
    a, b, ab = X[:, 0], X[:, -1], X[:, 1:K + 1]
    V = np.concatenate([a, b]).var()
    s1 = (b[:, None] * (ab - a[:, None])).mean(axis=0) / V
    st = 0.5 * ((a[:, None] - ab) ** 2).mean(axis=0) / V
    bs1, bst = np.empty((n_boot, K)), np.empty((n_boot, K))
    for t in range(n_boot):
        i = picks[t]
        at, bt, abt = a[i], b[i], ab[i]
        Vt = np.concatenate([at, bt]).var()
        bs1[t] = (bt[:, None] * (abt - at[:, None])).mean(axis=0) / Vt
        bst[t] = 0.5 * ((at[:, None] - abt) ** 2).mean(axis=0) / Vt
    return s1, st, bs1.std(axis=0, ddof=1), bst.std(axis=0, ddof=1)


def run_case(name, years, n_base, second_order, kind, n_boot, card, power, host_rows):
    import torch
    from simplyp_b200 import _cabi, ensemble as ens, mcmc, model as spm, packing as pk, tarland
    from simplyp_b200.engine import Engine
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(years[0], years[1], dynamic="y")
    eng = Engine()
    topo = pk.build_topology(p_struc, p["SC_list"])
    names, targets, bounds = mcmc._check_priors(ens.TARLAND_RANGES, topo.n_sc, False)
    K, S, D = len(names), topo.n_sc, len(met)
    P = 2 * K + 2 if second_order else K + 2
    M = n_base * P
    opt = spm.make_options(p_SU, p, dyn, topo)
    base_m, base_sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), {})
    sb = _cabi.make_sobol(targets, bounds[:, 0], bounds[:, 1], S, n_base, 0, True, second_order)
    d_forc = eng.to_device(pk.forcing_matrix(met))
    d_mem = eng.to_device(base_m).expand(M, pk.NP_MEMBER).contiguous()
    d_sc = eng.to_device(base_sc).expand(M, S, pk.NP_SC).contiguous()
    if kind == "objectives":
        o, odesc, labels = pk.obs_arrays(obs, topo, met.index, ("Q", "TDP"))
        d_obs, d_odesc = eng.to_device(o), eng.to_device(odesc)
        rows = [(v, pk.STAT_NAMES.index(s)) for v in range(len(labels)) for s in OBJ if s != "lp"] + [(0, -1)]
        d_rows = eng.to_device(np.asarray(rows, dtype=np.int32))
        R = len(rows)
    else:
        desc = np.array([(0, 0), (0, 2)], dtype=np.int32)
        d_desc = eng.to_device(desc)
        R = 2 * D
        chunk = max(1, (1 << 30) // (S * D * pk.NOUT * 8))
        out = torch.empty((min(chunk, M), S, D, pk.NOUT), dtype=torch.float64, device=eng.device)
        diag = torch.zeros((M, S, pk.NDIAG), dtype=torch.int64, device=eng.device)
    y = torch.empty((R, M), dtype=torch.float64, device=eng.device)
    z = statistics.NormalDist().inv_cdf(0.975)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]

    def one_pass():
        ev[0].record()
        eng.sobol_design(sb, d_mem, d_sc)
        ev[1].record()
        if kind == "objectives":
            stats, dg = eng.calibrate(d_forc, d_mem, d_sc, topo.parent_offsets, topo.parent_ids, d_obs, d_odesc, opt)
            ev[2].record()
            eng.sobol_outputs(stats, dg, d_rows, y)
            ev[3].record()
            times = None
        else:
            t_run, t_draw = 0.0, 0.0
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            for m0 in range(0, M, chunk):
                n = min(chunk, M - m0)
                e[0].record()
                eng.run(d_forc, d_mem[m0:m0 + n], d_sc[m0:m0 + n], topo.parent_offsets, topo.parent_ids, opt,
                        out=out[:n], diag=diag[m0:m0 + n])
                e[1].record()
                eng.predictive_draws(out[:n], d_mem[m0:m0 + n], d_sc[m0:m0 + n], diag[m0:m0 + n], d_desc,
                                     y.view(2, D, M), m0)
                e[2].record()
                torch.cuda.synchronize()
                t_run += e[0].elapsed_time(e[1])
                t_draw += e[1].elapsed_time(e[2])
            ev[2].record()
            ev[3].record()
            times = (t_run, t_draw)
        eng.sobol_indices(sb, y, 0, z, SEED)
        ev[4].record()
        res = eng.sobol_indices(sb, y, n_boot, z, SEED)
        ev[5].record()
        torch.cuda.synchronize()
        if times is None:
            times = (ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]))
        point = ev[3].elapsed_time(ev[4])
        total = ev[4].elapsed_time(ev[5])
        return dict(design_ms=ev[0].elapsed_time(ev[1]), integration_ms=times[0], outputs_ms=times[1],
                    point_ms=point, indices_with_bootstrap_ms=total, bootstrap_ms=total - point), res

    one_pass()
    t, res = one_pass()
    yh = y[:host_rows].cpu().numpy()
    n_used = res["n_used"].cpu().numpy()
    from tests import sobol_host
    picks = sobol_host.picks(SEED, n_boot, n_base)
    h0 = time.perf_counter()
    worst = 0.0
    for r in range(host_rows):
        s1, st, c1, cT = host_indices(yh[r], K, P, n_boot, picks)
        worst = max(worst, float(np.nanmax(np.abs(s1 - res["S1"][r].cpu().numpy()))),
                    float(np.nanmax(np.abs(c1 * z - res["S1_conf"][r].cpu().numpy()))))
    host_s = (time.perf_counter() - h0) / host_rows * R
    draws = R * n_boot * n_base
    line = dict(case=name, card=card, power_limit=power, K=K, n_base=n_base, second_order=second_order,
                members=M, rows=R, n_boot=n_boot, n_used_min=int(n_used.min()),
                **{k: round(v, 3) for k, v in t.items()},
                bootstrap_draws_per_s=draws / (t["bootstrap_ms"] * 1e-3),
                host_numpy_estimators_s_scaled=round(host_s, 2), host_rows_timed=host_rows,
                host_vs_device_max_abs_diff_S1_and_conf=worst)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--host-rows", type=int, default=2)
    a = ap.parse_args()
    card, power = gpu_info()
    cases = [("tarland2004_objectives_first_order", ("2004-01-01", "2004-12-31"), 1 << 12, False, "objectives", 1000),
             ("tarland2004_objectives_second_order", ("2004-01-01", "2004-12-31"), 1 << 12, True, "objectives", 1000),
             ("tarland2004_series_Q_TDP", ("2004-01-01", "2004-12-31"), 1 << 12, False, "series", 1000),
             ("tarland1981_2010_series_Q_TDP", ("1981-01-01", "2010-12-31"), 1 << 10, False, "series", 100)]
    lines = []
    for c in cases:
        line = run_case(*c, card, power, a.host_rows)
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
