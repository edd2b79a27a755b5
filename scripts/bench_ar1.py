"""Cost of the AR(1) error model of the log-likelihood on one GPU: one JSON line per case.

Case ``mcmc``: ``mcmc.sample``'s captured iteration on Tarland 2004 with 2×10⁴ walkers and the 18 free parameters of
``ensemble.TARLAND_RANGES``, without and with ``err_phi:Q`` / ``err_phi:TDP`` in (0, 0.95) (20 free parameters);
after 20 warm-up replays CUDA events time 100 replays, and the two samplers alternate three times.  Beside them, a
graph of the two bare half-ensemble calibrations (``Engine.calibrate``) without and with phi: the difference is what
the AR(1) path adds per iteration (the NaN fill of the simulated values, their stores, the AR(1) kernel).

Case ``ar1_kernel``: the device time of ``ar1_loglik_kernel`` alone, from ``torch.profiler`` (CUDA activities) over
100 replays of the calibration graph with phi, in a run of its own after the timed runs; its bytes are the simulated
values it reads, W/2 * V * D * 8 per launch.  The card's name and power limit are read in the same run.

    python scripts/bench_ar1.py [--out lines.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, WARMUP, TIMED, ROUNDS = 20000, 20, 100, 3
PHI = {"err_phi:Q": (0.0, 0.95), "err_phi:TDP": (0.0, 0.95)}


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


def _sampler(priors):
    from simplyp_b200 import mcmc, tarland
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load("2004-01-01", "2004-12-31", dynamic="y")
    s = mcmc._Sampler(met, p_struc, p_SU, p_LU, p_SC, p, dyn, obs, priors, W, 1 + ROUNDS * (WARMUP + TIMED), seed=1)
    s.evaluate_all()
    s.iteration_step()
    return s


def _calibration_graph(torch, s):
    g = torch.cuda.CUDAGraph()
    with s._device():
        with torch.cuda.graph(g):
            for half in (0, 1):
                s.evaluate(half)
    return g


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", help="also append the lines to this file")
    a = ap.parse_args()
    import torch
    from simplyp_b200 import _cabi
    from simplyp_b200 import ensemble as ens
    _cabi.require_device()
    card, power = gpu_info()
    iid, ar1 = _sampler(dict(ens.TARLAND_RANGES)), _sampler(dict(ens.TARLAND_RANGES, **PHI))
    graphs = {}
    for name, s in (("iid", iid), ("ar1", ar1)):
        with s._device():
            graphs[name] = (s.capture(), _calibration_graph(torch, s))
    ms = {k: {"iteration": [], "calibrations": []} for k in graphs}
    for _ in range(ROUNDS):
        for name, (g_iter, g_cal) in graphs.items():
            ms[name]["iteration"].append(round(_time_graph(torch, g_iter), 4))
            ms[name]["calibrations"].append(round(_time_graph(torch, g_cal), 4))
    lines = [{"case": "mcmc_tarland_2004", "gpu": card, "power_limit": power, "n_walkers": W,
              "days": int(ar1.d_forc.shape[0]), "n_obs_series": ar1.V, "n_free_iid": iid.K, "n_free_ar1": ar1.K,
              "ms_per_iteration_iid": ms["iid"]["iteration"], "ms_per_iteration_ar1": ms["ar1"]["iteration"],
              "ms_two_calibrations_iid": ms["iid"]["calibrations"],
              "ms_two_calibrations_ar1": ms["ar1"]["calibrations"],
              "timed_replays": TIMED, "warmup_replays": WARMUP, "rounds_alternated": ROUNDS}]
    g_cal = graphs["ar1"][1]
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(TIMED):
            g_cal.replay()
        torch.cuda.synchronize()
    from torch.autograd import DeviceType
    ev = [e.time_range.elapsed_us() for e in prof.events()
          if "ar1_loglik_kernel" in e.name and e.device_type == DeviceType.CUDA]
    n = len(ev)
    us = sum(ev) / max(n, 1)
    D = int(ar1.d_forc.shape[0])
    read = ar1.H * ar1.V * D * 8
    lines.append({"case": "ar1_kernel", "gpu": card, "power_limit": power, "members_per_launch": ar1.H, "days": D,
                  "n_obs_series": ar1.V, "launches_profiled": n, "us_per_launch": round(us, 2),
                  "MB_sim_obs_per_launch": round(read / 1e6, 2),
                  "GB_per_s": round(read / (us * 1e-6) / 1e9, 1) if us > 0 else None,
                  "source": "torch.profiler device time, 100 replays of the two-half calibration graph"})
    for line in lines:
        text = json.dumps(line)
        print(text, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(text + "\n")


if __name__ == "__main__":
    main()
