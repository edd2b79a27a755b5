"""Timing of NSGA-II (simplyp_b200.optimize.nsga2) on one GPU: one JSON line per (population size, objectives).

Per case: one generation (offspring, zero diag, fused-statistics ``Engine.calibrate`` of the N offspring, objective
rows, survival) is captured into a CUDA graph; after 20 warm-up replays, CUDA events time 100 replays.  The same events
time a graph of the bare ``Engine.calibrate`` launch of the same N members, a graph of the NSGA-II steps alone
(offspring, zero diag, objective rows, survival, without the integration) and a graph of the survival alone.  Free
parameters: the 18 of ``ensemble.TARLAND_RANGES``; M = 2 (NSE of Q and TDP) or 4 (also log_NSE of Q and NSE of TP).
``fronts_ranked`` is the number of fronts the last survival ranked.  The card's name and power limit are read in the
same run.  Lines are appended to ``profiles/r03_nsga2_bench_lines.jsonl`` (or ``--out``).

    python scripts/bench_nsga2.py [--out lines.jsonl] [--sizes 2048,10000,20000]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OBJECTIVES = {2: [(1, "Q", "NSE"), (1, "TDP", "NSE")],
              4: [(1, "Q", "NSE"), (1, "TDP", "NSE"), (1, "Q", "log_NSE"), (1, "TP", "NSE")]}
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


def run_case(N, M, card, power):
    import torch
    from simplyp_b200 import ensemble as ens, optimize, tarland

    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load("2004-01-01", "2004-12-31", dynamic="y")
    n_gen = 1 + 4 * (WARMUP + TIMED)
    o = optimize._Nsga2(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, ens.TARLAND_RANGES, N, n_gen, seed=1,
                        objectives=OBJECTIVES[M], variables=("Q", "TDP", "TP"))
    o.evaluate_initial()
    o.generation_step()

    def calibrate():
        o.diag.zero_()
        o.eng.calibrate(o.d_forc, o.d_mem, o.d_sc, o.topo.parent_offsets, o.topo.parent_ids, o.d_obs, o.d_desc,
                        o.opt, stats=o.stats, diag=o.diag)

    def nsga2_steps():
        o.offspring_step()
        o.diag.zero_()
        o.eng.sobol_outputs(o.stats, o.diag, o.d_rows, o.y)
        o.survive()
    with o._device():
        ms_gen = _time_graph(torch, o.capture())
        fronts = int(o.history[min(int(o.counters[0].item()), n_gen)][1].item())
        ms_cal = _time_graph(torch, _graph(torch, calibrate))
        ms_steps = _time_graph(torch, _graph(torch, nsga2_steps))
        ms_survive = _time_graph(torch, _graph(torch, o.survive))
    r = o.result()
    return dict(case="tarland_2004", gpu=card, power_limit=power, n_population=N, n_free=len(r.names),
                n_objectives=M, days=len(met), ms_per_generation=round(ms_gen, 4),
                ms_bare_calibration=round(ms_cal, 4), ms_nsga2_steps_alone=round(ms_steps, 4),
                ms_survival_alone=round(ms_survive, 4), survival_share_of_generation=round(ms_survive / ms_gen, 4),
                fronts_ranked=fronts, first_front_size=int((r.rank == 0).sum()), generations=r.generations,
                timed_replays=TIMED, warmup_replays=WARMUP)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_nsga2_bench_lines.jsonl"))
    ap.add_argument("--sizes", default="2048,10000,20000")
    a = ap.parse_args()
    card, power = gpu_info()
    for N in (int(s) for s in a.sizes.split(",")):
        for M in (2, 4):
            line = run_case(N, M, card, power)
            print(json.dumps(line), flush=True)
            with open(a.out, "a") as f:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
