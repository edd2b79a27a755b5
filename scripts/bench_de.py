"""Timing of differential evolution (simplyp_b200.optimize) on one GPU: one JSON line per population size.

Per case: one generation (trial, zero diag, fused-statistics ``Engine.calibrate`` of all N members, objective rows,
selection) is captured into a CUDA graph; after 20 warm-up replays, CUDA events time 100 replays.  The same events
time a graph of the bare ``Engine.calibrate`` launch of the same N members, and a graph of the DE steps alone (trial,
zero diag, objective rows, selection, without the integration): the difference of the first two and the third are
the optimiser's own cost per generation.  Free parameters: the 18 of ``ensemble.TARLAND_RANGES``; objective ``lp``;
``tol = 0`` so that no run converges inside the timed window.  The card's name and power limit are read in the same
run.

    python scripts/bench_de.py [--out lines.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CASES = [("tarland_2004", "2004-01-01", "2004-12-31", 2048), ("tarland_2004", "2004-01-01", "2004-12-31", 10000),
         ("tarland_2004", "2004-01-01", "2004-12-31", 20000)]
WARMUP, TIMED = 20, 100


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def _time_graph(torch, g):
    for _ in range(WARMUP):
        g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(TIMED):
        g.replay()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / TIMED


def _graph(torch, fn):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def run_case(name, st, en, N, card, power):
    import torch
    from simplyp_b200 import ensemble as ens, optimize, tarland

    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(st, en, dynamic="y")
    n_gen = 1 + 3 * (WARMUP + TIMED)
    o = optimize._Optimizer(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, ens.TARLAND_RANGES, N, n_gen, seed=1,
                            tol=0.0)
    o.evaluate_initial()
    o.generation_step()

    def calibrate():
        o.diag.zero_()
        o.eng.calibrate(o.d_forc, o.d_mem, o.d_sc, o.topo.parent_offsets, o.topo.parent_ids, o.d_obs, o.d_desc,
                        o.opt, stats=o.stats, diag=o.diag)

    def de_steps():
        o.trial_step()
        o.diag.zero_()
        o.eng.sobol_outputs(o.stats, o.diag, o.d_rows, o.y)
        o.select()
    with o._device():
        ms_gen = _time_graph(torch, o.capture())
        ms_cal = _time_graph(torch, _graph(torch, calibrate))
        ms_de = _time_graph(torch, _graph(torch, de_steps))
    r = o.result()
    assert not r.converged
    return dict(case=name, gpu=card, power_limit=power, n_population=N, n_free=len(r.names), days=len(met),
                n_obs_series=o.V, objective_rows=o.R, ms_per_generation=round(ms_gen, 4),
                ms_bare_calibration=round(ms_cal, 4), ms_de_overhead=round(ms_gen - ms_cal, 4),
                ms_de_steps_alone=round(ms_de, 4), member_sc_days_per_s=round(N * o.S * len(met) / (ms_gen * 1e-3), 1),
                best_objective_after_run=r.best_objective, generations=r.generations, timed_replays=TIMED,
                warmup_replays=WARMUP)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    card, power = gpu_info()
    lines = []
    for c in CASES:
        line = run_case(*c, card, power)
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
