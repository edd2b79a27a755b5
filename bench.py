#!/usr/bin/env python
"""Benchmark of the SimplyP daily mass-balance integration path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5]
                    [--members M] [--period 2004|full] [--dump-outputs DIR]

One "step" = one pass of the whole workload over its whole period.  Metric (BASELINE.json): member-sub-catchment-days
per second, whole job.  Workloads = BASELINE.json `configs` (SURVEY.md §8d):

  --config 2 (default)  Tarland (1 sub-catchment, 2004, both dynamic options on), Latin-hypercube ensemble of 10^4
                        parameter sets PER GPU (weak scaling), fused goodness-of-fit statistics vs observed Q and TDP,
                        all-gather of the statistics inside the timed step; e2e = simplyp_calibrate_host.
  --config 4            the same ensemble with 10^6 members IN TOTAL, sharded over the GPUs (strong scaling).
  --config 3            synthetic 256-sub-catchment branching network, 30-year daily forcing, both dynamic options on,
                        --members parameter sets per GPU (default 64), full daily output kept in HBM;
                        e2e = simplyp_run_host on a member subset whose output fits pinned host memory.
  --config 5            synthetic 4096-sub-catchment x 3 land-use network, 50-year daily run, full daily output written
                        to HBM (200 B per member-SC-day), --members per GPU (default 8).

Members are sharded over ranks with no data-path collective; the only collective is the all-gather of the per-member
statistics (configs 2 and 4).  Prints ONE JSON line (rank 0).  See DESIGN.md §5 for how each field is obtained.
`--impl reference` times the reference's own CPU algorithm (oracle port: per-day scipy odeint/LSODA at the reference's
rtol=0.01) on all host cores, on a bounded sample of the same workload.
`--dump-outputs DIR` writes what the last timed step returned (see dump_outputs) so that two builds can be compared
output for output: every input is generated from fixed seeds, so the same arguments give the same inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "member-sub-catchment-days/sec"
UNIT = "member-SC-days/s"
F_RHS, F_STEP_EXTRA, F_DAY = 140.0, 700.0, 120.0      # SURVEY.md §8(d) algorithmic flop counts
B_DAY = 200.0                                         # SURVEY.md §8(d): bytes written per member-SC-day (full output)
FP64_DFMA_PER_SM_CLK = 64                             # B200: 64 DFMA per SM per clock (nominal)
DUMP_BYTES = 64 * 10 ** 6                             # --dump-outputs: all files together
ST_SPEARMAN = 8                                       # SIMPLYP_ST_SPEARMAN: first stats slot after SIMPLYP_ST_SSE


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--members", type=int, default=None,
                    help="members per GPU (configs 2, 3, 5; defaults 10000 / 64 / 8) or in total (config 4; 10^6)")
    ap.add_argument("--period", default="2004", choices=["2004", "full"], help="configs 2 and 4: Tarland period")
    ap.add_argument("--rtol", type=float, default=None)
    ap.add_argument("--atol", type=float, default=None)
    ap.add_argument("--pilot-days", type=int, default=0, help="cost pilot: 0 = library default, -1 = off")
    ap.add_argument("--e2e-members", type=int, default=None,
                    help="configs 3 and 5: members of the end-to-end leg (default: as many as fit 48 GB of pinned host memory)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=24.0, help="sizes the cpu_baseline samples (about this many seconds of CPU work in total)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm keeps no outputs")
    if args.members is None:
        args.members = {2: 10000, 3: 64, 4: 1000000, 5: 8}[args.config]
    return args


def period_dates(period):
    return ("2004-01-01", "2004-12-31") if period == "2004" else ("1981-01-01", "2010-12-31")


# ------------------------------------------------------------------------------------------ workloads
def build_workload(period, n_members, seed=20260101, member_offset=0):
    """Configs 2/4: arrays of the calibration call for `n_members` members (deterministic in the member index)."""
    from simplyp_b200 import ensemble as ens, model as spm, packing as pk, tarland
    st, end = period_dates(period)
    p_SU, dyn, p, p_LU, p_SC, p_struc, met, obs = tarland.load(st, end, dynamic="y")
    topo = pk.build_topology(p_struc, p["SC_list"])
    samples = ens.latin_hypercube(n_members, seed=seed + member_offset)
    member, sc = ens.pack_members(pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids), samples)
    obs_m, desc, labels = pk.obs_arrays(obs, topo, met.index, ("Q", "TDP"))
    return dict(p_SU=p_SU, dyn=dyn, p=p, p_LU=p_LU, p_SC=p_SC, p_struc=p_struc, met=met, obs=obs, topo=topo,
                samples=samples, member=member, sc=sc, forcing=pk.forcing_matrix(met), obs_m=obs_m, desc=desc,
                labels=labels)


def workload_text(args, M_local, D, S):
    if args.config in (2, 4):
        how = ("%d-member LHS ensemble per GPU" % M_local) if args.config == 2 else \
              ("%d-member LHS ensemble in total, sharded over the GPUs" % args.members)
        return ("Tarland %s (D=%d days, S=1), %s, fused NSE/log-NSE/log-likelihood vs observed Q and TDP, "
                "Dynamic_EPC0/erodibility on" % (args.period, D, how))
    if args.config == 3:
        return ("synthetic 256-sub-catchment branching reach network (seed 3), 30-year daily forcing (D=%d), all "
                "dynamic options on, %d parameter sets per GPU, full daily output kept in HBM" % (D, M_local))
    return ("synthetic 4096-sub-catchment x 3 land-use network (seed 3), 50-year daily run (D=%d), full daily output "
            "written to HBM (200 B per member-SC-day), %d parameter sets per GPU" % (D, M_local))


# ------------------------------------------------------------------------------------------ CPU legs (oracle port)
def _cpu_worker(args):
    """Integrate `count` members with the oracle port; returns (member_sc_days, seconds)."""
    period, first, count, rtol, atol, seed, n_total = args
    sys.path.insert(0, ROOT)
    from oracle import simplyp_oracle as orc
    from simplyp_b200 import ensemble as ens
    w = build_workload(period, n_total, seed=seed)
    t0 = time.perf_counter()
    days = 0
    for i in range(first, first + count):
        pi, pLUi, pSCi = ens.apply_member_to_pandas(w["samples"], i, w["p"], w["p_LU"], w["p_SC"])
        orc.run_simply_p(w["met"], w["p_struc"], w["p_SU"], pLUi, pSCi, pi, w["dyn"], rtol=rtol, atol=atol,
                         mxstep=50000)
        days += len(w["met"])
    return days, time.perf_counter() - t0


def cpu_port_throughput(period, members_per_core, cores, rtol, atol):
    """Oracle port (scipy LSODA, one member per task) on `cores` processes; member-SC-days/s aggregate."""
    import multiprocessing as mp
    tasks = [(period, c * members_per_core, members_per_core, rtol, atol, 20260101, members_per_core * cores)
             for c in range(cores)]
    t0 = time.perf_counter()
    if cores == 1:
        res = [_cpu_worker(tasks[0])]
    else:
        with mp.get_context("spawn").Pool(cores) as pool:
            res = pool.map(_cpu_worker, tasks)
    wall = time.perf_counter() - t0
    days = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    return days / busy, days, busy, wall


_NET = {}


def cpu_network_throughput(cfg, n_days, processes, rtol, atol):
    """Oracle port on the first `n_days` of a network configuration (all reaches, one parameter set): the reference's
    SC-major loop nest, the reaches of a topological level spread over `processes` host processes
    (oracle/parallel.py; bit-identical to the serial call).  Returns (SC-days/s, SC-days, seconds)."""
    from oracle import parallel as opar, simplyp_oracle as orc
    from simplyp_b200 import synthetic
    if cfg not in _NET:
        _NET[cfg] = synthetic.scale_config(cfg)
    w = _NET[cfg]
    met = w["met"].iloc[:n_days]
    p, lu, sc, ups = orc.unpack_pandas(w["p_struc"], w["p_LU"], w["p_SC"], w["p"])
    a = (met["P"].to_numpy(), met["PET"].to_numpy(), met.index.dayofyear.to_numpy(), p, lu, sc, ups)
    kw = dict(run_mode="cal", dynamic_EPC0=True, dynamic_erodibility=True, rtol=rtol, atol=atol, mxstep=500000)
    t0 = time.perf_counter()
    if processes == 1:
        orc.run_network(*a, **kw)
    else:
        opar.run_network_parallel(*a, processes=processes, **kw)
    dt = time.perf_counter() - t0
    units = len(sc) * n_days
    return units / dt, units, dt


def cpu_baseline_legs(args, rtol, atol, D):
    """SURVEY.md §8(d): the reference's algorithm on the host cores — all cores and one process, at the GPU run's
    tolerance and at the reference's own (rtol=0.01, model.py:640).  Bounded samples of the same workload."""
    cores = os.cpu_count() or 1
    legs = {}
    if args.config in (2, 4):
        per_core = 1 if args.period == "full" else max(1, int(round(args.cpu_seconds / 1.2)))
        v, days, busy, _ = cpu_port_throughput(args.period, per_core, cores, rtol, atol)
        legs["all"] = (v, "%d members x %d days (same LHS members), one member per task on %d processes (%.1f s)"
                       % (per_core * cores, D, cores, busy))
        v1, _, b1, _ = cpu_port_throughput(args.period, max(1, per_core // 2), 1, rtol, atol)
        vr, _, br, _ = cpu_port_throughput(args.period, per_core, cores, 0.01, None)
        vr1, _, br1, _ = cpu_port_throughput(args.period, max(1, per_core // 2), 1, 0.01, None)
    else:
        S = 256 if args.config == 3 else 4096
        n_all = max(2, int(args.cpu_seconds * 350.0 * cores * 0.5 / S))     # ~350 SC-days/s/core at 1e-7, level-limited
        v, units, dt = cpu_network_throughput(args.config, n_all, cores, rtol, atol)
        legs["all"] = (v, "first %d days of the %d-reach network, one parameter set, reaches of a level on %d processes (%.1f s)"
                       % (n_all, S, cores, dt))
        n_one = max(1, int(args.cpu_seconds * 350.0 / S))
        v1, _, b1 = cpu_network_throughput(args.config, n_one, 1, rtol, atol)
        vr, _, br = cpu_network_throughput(args.config, n_all, cores, 0.01, None)
        vr1, _, br1 = cpu_network_throughput(args.config, n_one, 1, 0.01, None)
    return {"value": legs["all"][0], "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "oracle port = per-day scipy odeint/LSODA with a Python RHS at the GPU run's rtol/atol; " + legs["all"][1],
            "rtol": rtol, "atol": atol,
            "single_process": {"value": v1, "cores": 1, "seconds": b1},
            "reference_tolerance": {"rtol": 0.01, "atol": "odeint default", "value": vr, "cores": cores, "seconds": br,
                                    "single_process": {"value": vr1, "cores": 1, "seconds": br1}}}


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU algorithm (oracle port: per-day scipy odeint/LSODA at the
    reference's rtol=0.01 with a Python RHS callback) on all host cores.  The reference is pure Python and
    cannot travel to the GPU box, so the port stands in for it (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    times, units = [], 0
    if args.config in (2, 4):
        D = 366 if args.period == "2004" else 10957
        S = 1
        per_core = 2 if args.period == "2004" else 1
        sample = ("each step integrates a %d-member Latin-hypercube sample drawn by the same generator and seed, one member "
                  "per task on %d processes (bounded sample; member-SC-days/s does not depend on the ensemble size on the CPU)"
                  % (per_core * cores, cores))
        extra = {"members_per_step": per_core * cores}
        for it in range(args.warmup + args.steps):
            v, d, busy, wall = cpu_port_throughput(args.period, per_core, cores, 0.01, None)
            if it >= args.warmup:
                times.append(busy)
                units = d
    else:
        S, D = (256, 10958) if args.config == 3 else (4096, 18262)
        n_days = max(2, int(2.0 * 1500.0 * cores * 0.5 / S))       # about 2 s per step
        sample = ("each step integrates the first %d days of the %d-reach network for one parameter set, the reaches of a "
                  "topological level spread over %d processes (bounded sample of the %d-day record)" % (n_days, S, cores, D))
        extra = {"days_per_step": n_days}
        for it in range(args.warmup + args.steps):
            v, u, dt = cpu_network_throughput(args.config, n_days, cores, 0.01, None)
            if it >= args.warmup:
                times.append(dt)
                units = u
    ms = 1e3 * float(np.mean(times))
    value = units / (ms * 1e-3)
    cfg = {"workload": workload_text(args, args.members if args.config != 4 else args.members // max(args.gpus, 1), D, S),
           "bench_config": args.config, "sample": sample, "days": D, "sub_catchments": S, "rtol": 0.01,
           "atol": "odeint default (the reference's own solver settings, model.py:640)"}
    cfg.update(extra)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong" if args.config == 4 else "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic: Tarland forcing/obs example data or seeded synthetic network; seeded parameter sets",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": sample + "; scipy odeint (LSODA) rtol=0.01 as the reference calls it"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.gpu_index = gpu_index
        self.path = "/tmp/simplyp_clocks_%d_%d.csv" % (os.getpid(), gpu_index)

    def start(self):
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.fh,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, smax, reasons = [], [], set()
        try:
            for ln in open(self.path):
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    smax.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons), samples=len(sm),
                       window="warm-up + timed steps")
        return out


# ------------------------------------------------------------------------------------------ our arm
def _pinned(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


def dump_outputs(dirname, outputs):
    """Write each tensor of `outputs` (name -> tensor, last axis = one row) as DIR/<name>.npy in float64.
    A tensor larger than its share of DUMP_BYTES (the full daily output of configs 3 and 5 is tens of GB) is written as
    a sample of its rows, drawn with seed 0 from its shape alone, with the flat row indices in DIR/<name>_rows.npy:
    runs with the same arguments write the same rows."""
    import torch
    os.makedirs(dirname, exist_ok=True)
    share = DUMP_BYTES // len(outputs) - 1024         # an equal share per output, less its two .npy headers
    for name, t in outputs.items():
        rows = t.reshape(-1, t.shape[-1])
        n_keep = share // (8 * (rows.shape[1] + 1))   # a sampled row costs its values and its index
        if rows.shape[0] > n_keep:
            pick = np.sort(np.random.default_rng(0).choice(rows.shape[0], n_keep, replace=False))
            np.save(os.path.join(dirname, name + "_rows.npy"), pick.astype(np.float64))
            t = rows.index_select(0, torch.from_numpy(pick).to(rows.device))
        np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy().astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist

    from simplyp_b200 import _cabi, ensemble as ens, model as spm, packing as pk, synthetic
    from simplyp_b200.engine import Engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = Engine(local_rank)
    calibration = args.config in (2, 4)

    # ---- workload: this rank's member block [lo, hi) of M_total
    if calibration:
        M_total = args.members * world if args.config == 2 else args.members
        w = build_workload(args.period, M_total)
        opt = spm.make_options(w["p_SU"], w["p"], w["dyn"], w["topo"], 1.0, args.rtol, args.atol)
        kernel_name = "simplyp_quad_kernel<cal>"
        data = "Tarland forcing/obs example data (simplyp_b200/data/tarland); Latin-hypercube parameter sets, seed 20260101"
    else:
        M_total = args.members * world
        w = synthetic.scale_config(args.config, M_total)
        opt = w["opt"]
        if args.rtol is not None:
            opt.rtol = args.rtol
        if args.atol is not None:
            opt.atol = args.atol
        kernel_name = "simplyp_quad_kernel<run,stiff>"
        data = ("seeded synthetic network (simplyp_b200/synthetic.py: random_network seed 3, synthetic_met seed 11), Tarland "
                "parameters, members differ in a_Q (0.8x..1.2x)")
    opt.pilot_days = args.pilot_days
    lo, hi = ens.shard_bounds(M_total, world, rank)
    M_local = hi - lo
    topo = w["topo"]
    S, D = topo.n_sc, w["forcing"].shape[0]
    po, pid = topo.parent_offsets, topo.parent_ids
    sc_local = w["sc"][lo:hi] if w["sc"].shape[0] > 1 else w["sc"]

    # ---- device-resident leg ("value"): inputs already in HBM
    d_forc = eng.to_device(w["forcing"])
    d_mem = eng.to_device(w["member"][lo:hi])
    d_sc = eng.to_device(sc_local)
    diag = torch.zeros((M_local, S, pk.NDIAG), dtype=torch.int64, device=eng.device)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=eng.device)   # > 126 MB L2
    if calibration:
        V = w["obs_m"].shape[0]
        d_obs = eng.to_device(w["obs_m"])
        d_desc = eng.to_device(w["desc"])
        # the kernel writes this rank's statistics straight into its slot of the pre-allocated gather buffer
        gb = ens.GatherBuffers(M_total, (V, pk.NSTAT), eng.device)
        stats = gb.local
        # N > 1: the all-gather is fused into the calibration kernel (peer stores into every rank's buffer + a flag
        # exchange, ensemble.PeerGather) where CUDA IPC between the ranks works; SIMPLYP_GATHER=nccl keeps NCCL
        pg = None
        if world > 1 and os.environ.get("SIMPLYP_GATHER", "peer") != "nccl":
            try:           # (collective inside: succeeds or fails on all ranks together)
                pg = ens.PeerGather(M_total, (V, pk.NSTAT), eng.device)
            except Exception as e:
                pg = None
                sys.stderr.write("rank %d: peer gather unavailable (%r), using NCCL\n" % (rank, e))
        gather_mode = ("peer-memory stores fused into the calibration kernel + flag exchange" if pg is not None
                       else ("NCCL all_gather_into_tensor, in place" if world > 1 else "none (one rank)"))
        last = {}

        def step(mid=None):
            if pg is not None:
                last["g"], _ = eng.calibrate(d_forc, d_mem, d_sc, po, pid, d_obs, d_desc, opt, diag=diag, peer_gather=pg)
                if mid is not None:
                    mid.record()
                return last["g"]
            eng.calibrate(d_forc, d_mem, d_sc, po, pid, d_obs, d_desc, opt, stats=stats, diag=diag)
            if mid is not None:
                mid.record()               # this rank's own integration ends here; the all-gather waits for the slowest rank
            return gb.gather()
    else:
        out = torch.empty((M_local, S, D, pk.NOUT), dtype=torch.float64, device=eng.device)

        def step(mid=None):
            eng.run(d_forc, d_mem, d_sc, po, pid, opt, out=out, diag=diag)
            if mid is not None:
                mid.record()
            return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks are sampled from before the warm-up steps (nvidia-smi needs ~0.1 s to start and a timed region of 10
    # steps of config 2 lasts 0.15 s) to the end of the timed steps: every sample is taken under the bench load
    sampler = ClockSampler(local_rank)
    sampler.start()
    warmup = max(args.warmup, 3)
    for _ in range(warmup):
        flush.zero_()
        step()
    barrier()

    launches0 = _cabi.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    mid = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for k in range(args.steps):
        flush.zero_()                      # L2 flush between timed iterations (outside the events)
        ev[k][0].record()
        result = step(mid[k])
        ev[k][1].record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = _cabi.launch_count() - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:   # what a caller of the step receives; diag is this rank's
        if calibration:
            # the statistics the call computes: Spearman's r (slot 8) is a NaN placeholder unless opt.rank_stats is
            # set, and the last slot is reserved (include/simplyp_b200.h, SIMPLYP_ST_*)
            result = result[..., :ST_SPEARMAN + 1 if opt.rank_stats else ST_SPEARMAN]
        dump_outputs(args.dump_outputs, {"stats" if calibration else "out": result, "diag": diag})
    del result                            # configs 3 and 5: `out` must be freed before the end-to-end leg
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([float(sum(step_ms))], dtype=torch.float64, device=eng.device)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(total_ms.item()) / args.steps
    value = M_total * S * D / (ms_per_step * 1e-3)
    # every rank's OWN integration time per step (start of the step to the end of its kernels, before the all-gather):
    # the ranks integrate different members, and a step lasts as long as the slowest of them
    own_ms = torch.tensor([float(np.mean([a.elapsed_time(m) for (a, _b), m in zip(ev, mid)]))], dtype=torch.float64,
                          device=eng.device)
    ranks_own_ms = [own_ms.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(ranks_own_ms, own_ms)
    ranks_own_ms = [round(float(t.item()), 4) for t in ranks_own_ms]

    # ---- integrator work counters for the roofline (device-counted)
    dg = diag.sum(dim=(0, 1)).cpu().numpy().astype(float)
    n_steps, n_rej, n_rhs = dg[0], dg[1], dg[2]
    status_any = int(diag[..., 3].max().item())
    units_local = M_local * S * D
    flops_local = n_rhs * F_RHS + n_steps * F_STEP_EXTRA + units_local * F_DAY
    # work of the ACCEPTED attempts only (a rejected attempt is integrator overhead, not algorithmic work)
    acc_frac = 1.0 - n_rej / max(n_steps, 1.0)
    flops_accepted = (n_rhs * F_RHS + n_steps * F_STEP_EXTRA) * acc_frac + units_local * F_DAY
    kernel_ms = float(np.mean(step_ms))
    fp64_peak = _cabi.measure_fp64_peak(local_rank, 3) if rank == 0 else None
    if calibration:
        stats_ref = (last["g"][lo:hi] if pg is not None else stats).clone()
        alg_bytes = (d_forc.numel() + d_mem.numel() + d_sc.numel() + d_obs.numel()) * 8 + stats.numel() * 8 * 2
    else:
        alg_bytes = units_local * B_DAY + (d_forc.numel() + d_mem.numel() + d_sc.numel()) * 8
        ref_rows = out[0, S - 1, :64].clone()         # the outlet's first days, to compare with the end-to-end leg

    # ---- end-to-end leg: host buffers through the C-ABI, H2D + D2H inside the timed region
    if calibration:
        M_e2e = M_local
        h = {k: _pinned(v) for k, v in (("forcing", w["forcing"]), ("member", w["member"][lo:hi]), ("sc", sc_local),
                                        ("obs", w["obs_m"]))}
        st_host = _pinned(np.empty((M_e2e, V, pk.NSTAT)))
        dg_host = _pinned(np.zeros((M_e2e, S, pk.NDIAG), dtype=np.int64))
        h2d = sum(v.nbytes for v in h.values()) + w["desc"].nbytes
        d2h = st_host.nbytes + dg_host.nbytes

        def e2e_step():
            _cabi.calibrate_host(h["forcing"], h["member"], h["sc"], po, pid, h["obs"], w["desc"], opt, device=local_rank,
                                 stats=st_host, diag=dg_host)
        api = "simplyp_calibrate_host (C-ABI, pinned host buffers)"
        e2e_reps = args.steps
    else:
        del out
        torch.cuda.empty_cache()
        # as many members as fit a pinned host buffer of at most a quarter of the free host memory (48 GB at most)
        per_member = S * D * pk.NOUT * 8
        try:
            avail = [int(l.split()[1]) * 1024 for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0]
        except Exception:
            avail = 64 << 30
        fit = max(1, int(min(avail // 4, 48 << 30) // per_member))
        M_e2e = min(M_local, args.e2e_members if args.e2e_members else fit)
        h = {k: _pinned(v) for k, v in (("forcing", w["forcing"]), ("member", w["member"][lo:lo + M_e2e]),
                                        ("sc", sc_local[:M_e2e] if sc_local.shape[0] > 1 else sc_local))}
        out_host = torch.empty((M_e2e, S, D, pk.NOUT), dtype=torch.float64, pin_memory=True).numpy()
        dg_host = _pinned(np.zeros((M_e2e, S, pk.NDIAG), dtype=np.int64))
        h2d = sum(v.nbytes for v in h.values())
        d2h = out_host.nbytes + dg_host.nbytes

        def e2e_step():
            _cabi.run_host(h["forcing"], h["member"], h["sc"], po, pid, opt, device=local_rank, out=out_host, diag=dg_host)
        api = "simplyp_run_host (C-ABI, pinned host buffers; %d of the %d members per GPU)" % (M_e2e, M_local)
        e2e_reps = max(2, min(args.steps, 3))
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_reps):
        e2e_step()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=eng.device)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = M_e2e * world * S * D * e2e_reps / float(e2e_s.item())
    if calibration:
        same = bool(np.array_equal(st_host, stats_ref.cpu().numpy(), equal_nan=True))
    else:
        same = bool(np.array_equal(out_host[0, S - 1, :64], ref_rows.cpu().numpy()))

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        traffic, traffic_src = None, None
        try:     # measured DRAM traffic of this kernel at this size, from the committed ncu capture (null if none)
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            ent = tj.get("%s|%d|%d|%d" % (kernel_name, M_local, S, D)) or tj.get("%s|%d|%d" % (kernel_name, M_local, D))
            if ent:
                traffic, traffic_src = ent["bytes"], ent["source"]
        except Exception:
            pass
        achieved_tf = flops_accepted / (kernel_ms * 1e-3) / 1e12
        achieved_tf_all = flops_local / (kernel_ms * 1e-3) / 1e12
        achieved_gbs = alg_bytes / (kernel_ms * 1e-3) / 1e9
        sm_mhz = clocks.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
        n_sm = torch.cuda.get_device_properties(local_rank).multi_processor_count
        fp64_nominal = n_sm * FP64_DFMA_PER_SM_CLK * 2 * sm_mhz * 1e6 / 1e12
        fp64 = {"achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": (achieved_tf / fp64_peak) if fp64_peak else None,
                "achieved_incl_rejected_attempts": achieved_tf_all,
                "frac_incl_rejected_attempts": (achieved_tf_all / fp64_peak) if fp64_peak else None,
                "peak_source": "simplyp_measure_fp64_peak (DFMA probe, this run); MEASURED_PEAKS.json has no FP64 figure",
                "peak_nominal_at_clock": fp64_nominal,
                "peak_nominal_note": "%d SMs x 64 DFMA/clk x 2 flop x %.0f MHz (median SM clock of this run)" % (n_sm, sm_mhz),
                "algorithmic_flops_per_launch": flops_accepted,
                "algorithmic_flops_per_launch_incl_rejected": flops_local,
                "flops_per_member_sc_day": flops_accepted / units_local}
        hbm = {"achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
               "algorithmic_bytes_per_launch": int(alg_bytes),
               "bytes_per_member_sc_day": (B_DAY if not calibration else alg_bytes / units_local),
               "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"}
        primary = hbm if args.config == 5 else fp64
        roofline = {"bound": "hbm" if args.config == 5 else "fp64"}
        roofline.update({k: primary[k] for k in ("achieved", "peak", "unit", "frac")})
        roofline.update({"traffic": traffic, "traffic_source": traffic_src, "kernel": kernel_name, "kernel_ms": kernel_ms,
                         "steps_per_member_sc_day": n_steps / units_local, "rejected_frac": n_rej / max(n_steps, 1.0),
                         "rhs_per_member_sc_day": n_rhs / units_local, "fp64": fp64, "hbm": hbm})
        if args.config == 5:
            roofline["note"] = ("BASELINE.json names this the output-bandwidth-bound case; measured, the step is bound by the "
                                "FP64/issue rate of the integration (fp64 sub-object): at 200 B per member-SC-day the HBM "
                                "ceiling is %.2e member-SC-days/s, the FP64 ceiling at this workload's %.0f flop per "
                                "member-SC-day is %.2e" % (hbm_peak * 1e9 / B_DAY, flops_accepted / units_local,
                                                           (fp64_peak or fp64_nominal) * 1e12 / (flops_accepted / units_local)))
        if calibration:
            launches_text = ("pilot pass (days 0-7, member order) + counting sort (2) + observation constants + main pass "
                             "(days 8-end, cost order, blocks placed by SM)" + (" + NCCL all-gather" if world > 1 else ""))
        else:
            launches_text = "stiff/non-stiff grouping of the reaches (1 block) + the network launch (routing wavefront inside)"
        cfg = {"workload": workload_text(args, M_local, D, S), "bench_config": args.config,
               "members_total": M_total, "members_per_gpu": M_local, "days": D, "sub_catchments": S,
               "rtol": opt.rtol, "atol": opt.atol, "parallelism": "ensemble members sharded over %d GPU(s)" % world,
               "l2": "256 MB buffer written between timed steps (outside the per-step CUDA events)"
                     + ("" if calibration else "; the output written per step (%.1f GB) is far larger than L2" % (units_local * B_DAY / 1e9)),
               "launches_per_step": launches_text}
        if calibration:
            cfg["obs_series"] = [list(l) for l in w["labels"]]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if args.config == 4 else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic: " + data,
            "config": cfg,
            "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "api": api, "members_per_gpu": M_e2e, "steps": e2e_reps, "matches_device_leg": same},
            "roofline": roofline,
            "clocks": clocks, "integrator_status_bits": status_any, "wall_s_timed_region": t_wall,
            "ranks_own_ms_per_step": ranks_own_ms if not (calibration and pg is not None) else None,
        }
        if calibration:
            line["config"]["gather"] = gather_mode
        if not args.no_cpu_baseline and world == 1:
            try:
                line["cpu_baseline"] = cpu_baseline_legs(args, opt.rtol, opt.atol, D)
            except Exception as e:  # keep the bench line even if the CPU leg cannot run
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                                        "sample": "failed: %r" % (e,)}
        print(json.dumps(line), flush=True)
    if calibration and pg is not None:
        pg.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
