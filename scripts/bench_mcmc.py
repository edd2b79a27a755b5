"""Timing of the ensemble sampler (simplyp_b200.mcmc) on one GPU: one JSON line per case.

Per case: one iteration (propose / integrate / accept for each half) is captured into a CUDA graph; after 20 warm-up
replays, CUDA events time 100 replays.  The same events time a graph of the two bare ``Engine.calibrate`` launches of
W/2 members each: the difference is the sampler's own cost per iteration.  Free parameters: the 18 of
``ensemble.TARLAND_RANGES``.  The card's name and power limit are read in the same run.

    python scripts/bench_mcmc.py [--out lines.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CASES = [("tarland_2004", "2004-01-01", "2004-12-31", 64), ("tarland_2004", "2004-01-01", "2004-12-31", 2048),
         ("tarland_2004", "2004-01-01", "2004-12-31", 20000), ("tarland_1981_2010", "1981-01-01", "2010-12-31", 2048)]
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


def run_case(name, st, en, W, card, power):
    import torch
    from simplyp_b200 import ensemble as ens, mcmc, tarland

    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(st, en, dynamic="y")
    s = mcmc._Sampler(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, ens.TARLAND_RANGES, W, 1 + WARMUP + TIMED, seed=1)
    s.evaluate_all()
    s.iteration_step()
    with s._device():
        ms_iter = _time_graph(torch, s.capture())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for half in (0, 1):
                lo, hi = half * s.H, (half + 1) * s.H
                mem, sc = s._rows(lo, hi)
                s.eng.calibrate(s.d_forc, mem, sc, s.topo.parent_offsets, s.topo.parent_ids, s.d_obs, s.d_desc, s.opt,
                                stats=s.stats[lo:hi], diag=s.diag[lo:hi])
        ms_cal = _time_graph(torch, g)
    r = s.result()
    D = len(met)
    return {"case": name, "gpu": card, "power_limit": power, "n_walkers": W, "n_free": s.K, "days": D,
            "n_obs_series": s.V, "ms_per_iteration": round(ms_iter, 4), "ms_two_calibrations": round(ms_cal, 4),
            "ms_sampler_overhead": round(ms_iter - ms_cal, 4),
            "member_sc_days_per_s": round(W * D * s.S / (ms_iter * 1e-3), 1),
            "acceptance_fraction": round(float(r.acceptance_fraction.mean()), 4),
            "iterations": r.iterations, "timed_replays": TIMED, "warmup_replays": WARMUP}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", help="also append the lines to this file")
    a = ap.parse_args()
    from simplyp_b200 import _cabi
    _cabi.require_device()
    card, power = gpu_info()
    for name, st, en, W in CASES:
        line = json.dumps(run_case(name, st, en, W, card, power))
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
