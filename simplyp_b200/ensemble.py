"""Parameter ensembles: sampling, packing, sharding over GPUs, fused calibration statistics.

The reference has no ensemble driver in its release; the only construct of this kind is the
development notebook's emcee sampler over an IPython.parallel pool
(``Development/2016/MCMC.ipynb:29-31,380``), i.e. independent parameter sets evaluated in parallel.
Here the members of an ensemble are the threads of one kernel launch, and the ranks of a
``torch.distributed`` job each take a contiguous block of members (SURVEY.md §8e); the only
collective is one all-gather of the per-member fit statistics.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import packing as pk

#: Latin-hypercube ranges bracketing the Tarland values (SURVEY.md §8d, config 2).
#: key: member field (``packing.MEMBER_FIELDS``), or ``sc:<row>`` for a p_SC row applied to every SC.
TARLAND_RANGES = {
    "f_quick": (0.0, 0.1), "alpha": (0.5, 1.2), "fc": (100.0, 400.0), "beta": (0.3, 0.9), "T_g": (20.0, 150.0),
    "T_s:A": (1.0, 8.0), "T_s:S": (3.0, 20.0), "a_Q": (0.2, 0.9), "b_Q": (0.3, 0.6), "Qg_min": (0.05, 0.6),
    "E_M": (300.0, 3000.0), "k_M": (1.2, 2.5), "E_PP": (1.0, 3.0), "TDPg": (0.0, 0.05),
    "EPC0_init_mgl:A": (0.03, 0.3), "sc:TDPeff": (0.0, 0.5),
    "err_m:Q": (0.05, 1.0), "err_m:TDP": (0.05, 1.0),
}


def latin_hypercube(n, ranges=None, seed=20260101):
    """``n`` stratified samples per parameter; returns dict name -> array [n]."""
    ranges = TARLAND_RANGES if ranges is None else ranges
    rng = np.random.default_rng(seed)
    out = {}
    for name, (lo, hi) in ranges.items():
        strata = (rng.permutation(n) + rng.random(n)) / n
        out[name] = lo + (hi - lo) * strata
    return out


def pack_members(base_member, base_sc, samples, return_phi=False):
    """Broadcast the base parameter vectors over the ensemble and apply the sampled columns.

    base_member [NP_MEMBER], base_sc [S][NP_SC], samples: dict name -> [M].
    Returns (member_params [M][NP_MEMBER], sc_params [1 or M][S][NP_SC]).  The AR(1) error-model parameters
    ``err_phi:<kind>`` are in neither: with ``return_phi`` they come back separately as a third item, a dict
    name -> [M] in the order of ``samples``.
    """
    M = len(next(iter(samples.values()))) if samples else 1
    member = np.repeat(np.asarray(base_member, dtype=np.float64)[None, :], M, axis=0)
    sc = np.asarray(base_sc, dtype=np.float64)[None, :, :]
    per_member_sc = any(k.startswith("sc:") for k in samples)
    if per_member_sc:
        sc = np.repeat(sc, M, axis=0)
    phi = {}
    for name, vals in samples.items():
        vals = np.asarray(vals, dtype=np.float64)
        if name.startswith(pk.ERR_PHI):
            phi[name] = vals
        elif name.startswith("sc:"):
            row = name[3:]
            if "@" in row:                       # sc:<row>@<position in run order>
                row, at = row.split("@")
                sc[:, int(at), pk.SC_INDEX[row]] = vals
            else:
                sc[:, :, pk.SC_INDEX[row]] = vals[:, None]
        else:
            member[:, pk.MEMBER_INDEX[name]] = vals
    if return_phi:
        return np.ascontiguousarray(member), np.ascontiguousarray(sc), phi
    return np.ascontiguousarray(member), np.ascontiguousarray(sc)


@dataclass
class _ModelInputs:
    """What :func:`_model_inputs` returns: the host inputs every ensemble driver starts from."""
    topo: pk.Topology
    opt: object                 # SimplypOptions
    member: np.ndarray          # base member vector [NP_MEMBER]
    sc: np.ndarray              # base SC matrix [S][NP_SC]
    forcing: np.ndarray         # [D][NF]


def _model_inputs(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, step_len=1.0, rtol=None, atol=None,
                  snow_on_device=False):
    """The reference's checks of the land use and the erosion windows, the topology, the options (with
    ``snow_on_device``), the base parameter vectors :func:`pack_members` broadcasts and the forcing matrix (raw
    precipitation with ``snow_on_device``).  Host work only, on copies of the frames: a driver calls it before any
    device work."""
    from .model import make_options

    p_LU, p_SC = p_LU.copy(deep=True), p_SC.copy(deep=True)
    pk.validate_land_use(p_SC, p["SC_list"])
    pk.check_erosion_windows(p)
    topo = pk.build_topology(p_struc, p["SC_list"])
    opt = make_options(p_SU, p, dynamic_options, topo, step_len, rtol, atol)
    opt.snow_on_device = 1 if snow_on_device else 0
    return _ModelInputs(topo, opt, pk.member_vector(p, p_LU), pk.sc_matrix(p_SC, topo.sc_ids),
                        pk.forcing_matrix(met_df, raw_snow=bool(snow_on_device)))


def apply_member_to_pandas(samples, i, p, p_LU, p_SC):
    """Copies of the reference's pandas objects with member ``i``'s sampled values written in — this is how
    the oracle / the reference is run on the same member."""
    p, p_LU, p_SC = p.copy(deep=True), p_LU.copy(deep=True), p_SC.copy(deep=True)
    for name, vals in samples.items():
        v = float(vals[i])
        if name.startswith("err_m:") or name.startswith(pk.ERR_PHI):
            continue
        if name.startswith("sc:"):
            row = name[3:]
            if "@" in row:
                row, at = row.split("@")
                p_SC.loc[row, p_SC.columns[int(at)]] = v
            else:
                p_SC.loc[row, :] = v
        elif ":" in name:
            row, col = name.split(":")
            p_LU.loc[row, col] = v
        else:
            p[name] = v
    return p, p_LU, p_SC


def shard_bounds(n_members, world_size, rank):
    """Contiguous block [lo, hi) of members for ``rank`` (sizes differ by at most one)."""
    base, extra = divmod(n_members, world_size)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


class GatherBuffers:
    """Pre-allocated buffers of the one collective of the path: the all-gather of the per-member fit statistics.

    ``local`` is this rank's slot INSIDE the gather buffer — hand it to ``Engine.calibrate(stats=...)`` and the kernel
    writes its statistics where the collective reads them; ``gather()`` is then one ``all_gather_into_tensor`` with no
    allocation, no padding copy and (when the shards are equal) no concatenation: the returned tensor is the buffer.
    NCCL gathers in place (send buffer = own slot of the receive buffer); gloo (CPU tests) gets a copy of the slot.
    """

    def __init__(self, n_members, tail_shape, device, dtype=None, group=None):
        import torch
        import torch.distributed as dist

        self.group = group
        self.n_members = int(n_members)
        on = dist.is_available() and dist.is_initialized()
        self.world = dist.get_world_size(group) if on else 1
        self.rank = dist.get_rank(group) if on else 0
        self.sizes = [shard_bounds(self.n_members, self.world, r) for r in range(self.world)]
        self.mmax = max(hi - lo for lo, hi in self.sizes)
        self.equal = all(hi - lo == self.mmax for lo, hi in self.sizes)
        dtype = torch.float64 if dtype is None else dtype
        self.buffer = torch.zeros((self.world * self.mmax,) + tuple(tail_shape), dtype=dtype, device=device)
        lo, hi = self.sizes[self.rank]
        self.slot = self.buffer[self.rank * self.mmax:(self.rank + 1) * self.mmax]
        self.local = self.slot[:hi - lo]
        self.compact = None if self.equal else torch.empty((self.n_members,) + tuple(tail_shape), dtype=dtype, device=device)

    def gather(self):
        """All ranks' statistics, [M][...] in member order (a view of the buffer when the shards are equal)."""
        import torch
        import torch.distributed as dist

        if self.world > 1:
            src = self.slot if self.buffer.is_cuda else self.slot.clone()
            dist.all_gather_into_tensor(self.buffer, src, group=self.group)
        if self.equal:
            return self.buffer
        torch.cat([self.buffer[r * self.mmax: r * self.mmax + (hi - lo)] for r, (lo, hi) in enumerate(self.sizes)],
                  dim=0, out=self.compact)
        return self.compact


class PeerGather:
    """The all-gather of the per-member fit statistics FUSED into the calibration kernel (one process per GPU of one
    NVLink / NVSwitch box): every rank maps every other rank's gather buffer (CUDA IPC) and its kernel stores each
    finished member's statistics straight into all of them; after the integration only a flag exchange is left
    (``simplyp_calibrate_gather_device``, include/simplyp_b200.h).  Replaces ``GatherBuffers`` + NCCL on this path;
    ``torch.distributed`` is used once, to exchange the IPC handles.

    Two buffer sets alternate from call to call (a fast rank may write step k+1 while a slow one still reads step k):
    the tensor :meth:`Engine.calibrate` returns is valid until the call after the next one.
    Raises ``SimplypError`` where CUDA IPC or peer access is not available — fall back to ``GatherBuffers``.
    """

    def __init__(self, n_members, tail_shape, device, group=None):
        import torch
        import torch.distributed as dist
        from . import _cabi

        self.group = group
        self.n_members = int(n_members)
        self.tail = tuple(int(x) for x in tail_shape)
        self.device = torch.device(device)
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        if self.world > _cabi.MAX_RANKS:
            raise _cabi.SimplypError("PeerGather: at most %d ranks" % _cabi.MAX_RANKS)
        self.lo, self.hi = shard_bounds(self.n_members, self.world, self.rank)
        self.buf_bytes = (8 * self.n_members * int(np.prod(self.tail)) + 255) // 256 * 256
        self.flag_bytes = 256
        self.step = 0
        self._peers = []
        # Every rank takes part in the exchange whatever happened locally (a rank that could not allocate or export
        # sends None), so that a failure is seen by all ranks together and nobody waits in a collective alone.
        self.base, handle, err = 0, None, None
        self.bases = []

        def local_export():
            with torch.cuda.device(self.device):
                self.base = _cabi.peer_alloc(self.flag_bytes + 2 * self.buf_bytes)
                return _cabi.ipc_export(self.base)

        def local_import(handles):
            with torch.cuda.device(self.device):
                for r, h in enumerate(handles):
                    if r == self.rank:
                        self.bases.append(self.base)
                    else:
                        ptr = _cabi.ipc_import(h)
                        self._peers.append(ptr)
                        self.bases.append(ptr)

        try:
            handle = local_export()
        except Exception as e:          # no device, no memory, IPC not permitted ...
            err = e
        handles = [None] * self.world
        dist.all_gather_object(handles, handle, group=group)
        if err is None and all(h is not None for h in handles):
            try:
                local_import(handles)
            except Exception as e:
                err = e
        elif err is None:
            err = _cabi.SimplypError("PeerGather: a peer could not export its buffer")
        oks = [None] * self.world
        dist.all_gather_object(oks, err is None, group=group)
        if not all(oks):
            try:
                self.close()
            except Exception:
                pass
            msg = "PeerGather unavailable: %r" % (err,) if err is not None else "PeerGather: a peer could not map the buffers"
            raise _cabi.SimplypError(msg)
        self._views = [self._tensor(self.base + self.flag_bytes + k * self.buf_bytes) for k in range(2)]

    def _tensor(self, ptr):
        import torch

        shape = (self.n_members,) + self.tail

        class _Mem:
            __cuda_array_interface__ = {"shape": shape, "typestr": "<f8", "data": (int(ptr), False), "version": 3,
                                        "strides": None}
        return torch.as_tensor(_Mem(), device=self.device)

    def descriptor(self):
        """SimplypPeerGather of the NEXT call (advances the step) and the tensor its result will be in."""
        from . import _cabi

        self.step += 1
        k = self.step % 2
        g = _cabi.SimplypPeerGather()
        g.n_ranks, g.rank = self.world, self.rank
        g.member_offset, g.n_members_total, g.step = self.lo, self.n_members, self.step
        for r in range(self.world):
            g.stats_bufs[r] = self.bases[r] + self.flag_bytes + k * self.buf_bytes
            g.flag_bufs[r] = self.bases[r]
        return g, self._views[k]

    def close(self):
        from . import _cabi
        import torch

        import torch.distributed as dist

        if self._peers or self.base:
            torch.cuda.synchronize(self.device)
            with torch.cuda.device(self.device):
                for ptr in self._peers:
                    _cabi.ipc_close(ptr)
        self._peers = []
        # (an exported allocation must outlive its mappings in the other processes: every rank calls close())
        if self.world > 1 and dist.is_initialized():
            dist.barrier(group=self.group)
        if self.base:
            with torch.cuda.device(self.device):
                _cabi.peer_free(self.base)
            self.base = 0


_gather_cache = {}


def all_gather_stats(local_stats, n_members, group=None):
    """All-gather the per-member statistics [M_local][V][10] of every rank into [M][V][10] (rank order).

    Uses ``torch.distributed`` (NCCL on GPUs, gloo in the CPU tests) through a cached :class:`GatherBuffers`; callers
    that run many passes should hold a ``GatherBuffers`` themselves and let the kernel write into ``.local``.
    """
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()):
        return local_stats
    key = (int(n_members), tuple(local_stats.shape[1:]), str(local_stats.device), local_stats.dtype, id(group))
    gb = _gather_cache.get(key)
    if gb is None:
        gb = _gather_cache[key] = GatherBuffers(n_members, local_stats.shape[1:], local_stats.device, local_stats.dtype, group)
    gb.local.copy_(local_stats)
    return gb.gather()


def calibrate_ensemble(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, obs_dict, samples,
                       variables=("Q", "TDP"), step_len=1.0, rtol=None, atol=None, engine=None, gather=True,
                       snow_on_device=False, rank_stats=False):
    """Fused-statistics run of an ensemble; this rank integrates its shard and (optionally) all-gathers.

    ``snow_on_device``: ``met_df`` carries the raw ``Precipitation`` and ``T_air``; the degree-day snow module
    (reference ``inputs.py:159-210``) runs per member on the device, so ``D_snow_0`` and ``f_DDSM`` may be sampled.
    ``rank_stats``: also reduce Spearman's r (the whole table of ``goodness_of_fit_stats``).
    ``err_phi:<variable>`` in ``samples`` gives the log-likelihood of that variable's series the AR(1) error model with
    that lag-one autocorrelation (``simplyp_calibrate_ar1_device``); the other statistics do not change.  An
    ``err_phi`` name of an unknown variable or of one not among ``variables`` raises ``ValueError`` before any device
    work.

    Returns ``(stats [M][V][10] torch tensor on the device, labels [(reach, variable)], diag)``.
    """
    import torch
    import torch.distributed as dist

    from .engine import Engine

    inp = _model_inputs(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, step_len, rtol, atol, snow_on_device)
    topo, opt = inp.topo, inp.opt
    opt.rank_stats = 1 if rank_stats else 0
    member, sc, phi = pack_members(inp.member, inp.sc, samples, return_phi=True)
    M = member.shape[0]
    rank, world = (dist.get_rank(), dist.get_world_size()) if (dist.is_available() and dist.is_initialized()) else (0, 1)
    lo, hi = shard_bounds(M, world, rank)
    obs, desc, labels = pk.obs_arrays(obs_dict, topo, met_df.index, variables)
    phi_col = pk.ar1_columns(list(phi), labels, variables)
    eng = engine or Engine()
    d_forc = eng.to_device(inp.forcing)
    d_mem = eng.to_device(member[lo:hi])
    d_sc = eng.to_device(sc if sc.shape[0] == 1 else sc[lo:hi])
    d_obs = eng.to_device(obs)
    d_desc = eng.to_device(desc)
    d_phi = eng.to_device(np.stack(list(phi.values()), axis=1)[lo:hi]) if phi else None
    stats, diag = eng.calibrate(d_forc, d_mem, d_sc, topo.parent_offsets, topo.parent_ids, d_obs, d_desc, opt,
                                phi=d_phi, phi_col=phi_col if phi else None)
    if gather and world > 1:
        stats = all_gather_stats(stats, M)
    torch.cuda.synchronize(eng.device)
    return stats, labels, diag


# --------------------------------------------------------------------------- full-output ensemble container
def _safe_name(col):
    return col.replace("/", "_per_")


def run_ensemble_to_dir(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, samples, out_dir, columns=None,
                        members_per_chunk=None, step_len=1.0, rtol=None, atol=None, engine=None):
    """Full daily output of an ensemble written as one ``.npy`` per raw variable (SURVEY.md §8f rank 4).

    The members are integrated in chunks; while the GPU integrates chunk k+1 (compute stream), chunk k travels to
    PINNED host memory on a copy stream and is scattered by the host into memory-mapped ``<variable>.npy`` files of
    shape ``[M][S][D]`` (float64) — the reference's raw columns (``model.py:737-745``), ``/`` in a name written as
    ``_per_``.  ``manifest.json`` lists variables, shapes, member parameters (``samples.npz``), sub-catchment ids,
    dates and the integrator diagnostics (``diag.npy`` [M][S][4]).  Two device buffers and two pinned buffers of
    ``members_per_chunk * S * D * 200`` bytes each are used (default: about 1 GiB per buffer).

    Returns the manifest dict.  Ranks of a ``torch.distributed`` job each write their member shard
    (``shard_bounds``) into files of the full shape opened in ``r+`` mode, rank 0 creating them first.
    """
    import json
    import os

    import torch
    import torch.distributed as dist

    from .engine import Engine

    inp = _model_inputs(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, step_len, rtol, atol)
    topo, opt = inp.topo, inp.opt
    member, sc = pack_members(inp.member, inp.sc, samples)
    M, S, D = member.shape[0], len(topo.sc_ids), len(met_df)
    cols = list(pk.RAW_COLS) if columns is None else list(columns)
    col_idx = [pk.RAW_COLS.index(c) for c in cols]
    rank, world = (dist.get_rank(), dist.get_world_size()) if (dist.is_available() and dist.is_initialized()) else (0, 1)
    lo, hi = shard_bounds(M, world, rank)

    os.makedirs(out_dir, exist_ok=True)
    paths = {c: os.path.join(out_dir, _safe_name(c) + ".npy") for c in cols}
    diag_path = os.path.join(out_dir, "diag.npy")
    if rank == 0:
        for c in cols:
            np.lib.format.open_memmap(paths[c], mode="w+", dtype=np.float64, shape=(M, S, D)).flush()
        np.lib.format.open_memmap(diag_path, mode="w+", dtype=np.int64, shape=(M, S, pk.NDIAG)).flush()
        np.savez(os.path.join(out_dir, "samples.npz"), **{k.replace(":", "__"): np.asarray(v) for k, v in samples.items()})
    if world > 1:
        dist.barrier()
    files = {c: np.load(paths[c], mmap_mode="r+") for c in cols}
    diag_file = np.load(diag_path, mmap_mode="r+")

    eng = engine or Engine()
    row_bytes = S * D * pk.NOUT * 8
    if members_per_chunk is None:
        members_per_chunk = max(1, (1 << 30) // max(row_bytes, 1))
    chunk = int(max(1, min(members_per_chunk, hi - lo))) if hi > lo else 1
    d_forc = eng.to_device(inp.forcing)
    d_mem = eng.to_device(member[lo:hi]) if hi > lo else None
    d_sc = eng.to_device(sc if sc.shape[0] == 1 else sc[lo:hi]) if hi > lo else None
    dev_buf = [torch.empty((chunk, S, D, pk.NOUT), dtype=torch.float64, device=eng.device) for _ in range(2)]
    dev_diag = [torch.zeros((chunk, S, pk.NDIAG), dtype=torch.int64, device=eng.device) for _ in range(2)]
    pin_buf = [torch.empty((chunk, S, D, pk.NOUT), dtype=torch.float64, pin_memory=True) for _ in range(2)]
    pin_diag = [torch.empty((chunk, S, pk.NDIAG), dtype=torch.int64, pin_memory=True) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=eng.device)
    computed = [torch.cuda.Event() for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    pending = []                                      # (buffer, first member, count) in flight to the host

    def drain(item):
        b, m0, n = item
        copied[b].synchronize()
        host = pin_buf[b].numpy()
        for c, j in zip(cols, col_idx):
            files[c][m0:m0 + n] = host[:n, :, :, j]
        diag_file[m0:m0 + n] = pin_diag[b].numpy()[:n]

    with torch.cuda.device(eng.device):
        compute_stream = torch.cuda.current_stream()
        k = 0
        for m0 in range(lo, hi, chunk):
            n = min(chunk, hi - m0)
            b = k % 2
            if len(pending) == 2:                     # buffer b is still travelling / being scattered
                drain(pending.pop(0))
            scp = d_sc if d_sc.shape[0] == 1 else d_sc[m0 - lo:m0 - lo + n]
            eng.run(d_forc, d_mem[m0 - lo:m0 - lo + n], scp, topo.parent_offsets, topo.parent_ids, opt,
                    out=dev_buf[b][:n], diag=dev_diag[b][:n])
            computed[b].record(compute_stream)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(computed[b])
                pin_buf[b][:n].copy_(dev_buf[b][:n], non_blocking=True)
                pin_diag[b][:n].copy_(dev_diag[b][:n], non_blocking=True)
                copied[b].record(copy_stream)
            pending.append((b, m0, n))
            k += 1
        while pending:
            drain(pending.pop(0))
    for f in files.values():
        f.flush()
    diag_file.flush()
    if world > 1:
        dist.barrier()
    manifest = {
        "format": "simplyp_b200 ensemble container v1",
        "variables": {c: os.path.basename(paths[c]) for c in cols},
        "shape": [M, S, D], "dtype": "float64", "axes": ["member", "sub_catchment", "day"],
        "sub_catchments": [int(s) for s in topo.sc_ids],
        "dates": [str(met_df.index[0].date()), str(met_df.index[-1].date())],
        "diag": "diag.npy", "samples": "samples.npz",
        "options": {"rtol": float(opt.rtol), "atol": float(opt.atol),
                    "dynamic_epc0": int(opt.dynamic_epc0), "dynamic_erodibility": int(opt.dynamic_erodibility)},
        "members_per_chunk": chunk, "world_size": world,
    }
    if rank == 0:
        with open(os.path.join(out_dir, "manifest.json"), "w") as f:
            json.dump(manifest, f, indent=1)
    return manifest


# --------------------------------------------------------------------------- posterior predictive bands
DEFAULT_BAND_SEED = 20260102


@dataclass
class PredictiveBands:
    """What :func:`predictive_bands` returns.  ``quantiles`` [n_q][V][D] is the layout of
    ``np.nanquantile(draws, q, axis=-1)``; ``mean`` [V][D] and ``count`` [V][D] are the mean and the number of the
    members that entered every (series, day) — all members but the ``n_failed`` whose integration raised a status bit.
    ``labels`` [(sc_id, variable)] name the series, ``dates`` the days."""
    q: np.ndarray
    quantiles: np.ndarray
    mean: np.ndarray
    count: np.ndarray
    n_failed: int
    labels: list
    dates: object

    def band(self, q):
        """The band [V][D] of quantile value ``q`` (one of ``self.q``)."""
        hits = np.flatnonzero(self.q == float(q))
        if hits.size == 0:
            raise ValueError("%r is not one of the computed quantiles %s" % (q, list(self.q)))
        return self.quantiles[hits[0]]

    def coverage(self, obs_dict, lo, hi):
        """Per series label: ``(observed days, fraction of them with band_lo <= obs <= band_hi)`` for the bands of
        the quantile values ``lo`` and ``hi``; ``obs_dict`` as ``calibrate_ensemble`` takes it."""
        b_lo, b_hi = self.band(lo), self.band(hi)
        out = {}
        for v, (sc_id, var) in enumerate(self.labels):
            df = obs_dict.get(sc_id)
            if df is None or var not in df.columns:
                out[(sc_id, var)] = (0, float("nan"))
                continue
            ser = df[var]
            o = ser[~ser.index.duplicated()].reindex(self.dates).to_numpy(dtype="float64")
            seen = ~np.isnan(o)
            n = int(seen.sum())
            inside = int(np.sum((b_lo[v][seen] <= o[seen]) & (o[seen] <= b_hi[v][seen])))
            out[(sc_id, var)] = (n, inside / n if n else float("nan"))
        return out


def _check_band_quantiles(quantiles):
    q = np.asarray(quantiles, dtype=np.float64).reshape(-1)
    if q.size == 0 or q.size > 16:
        raise ValueError("1..16 quantile values, got %d" % q.size)
    if not np.all(np.isfinite(q)) or np.any(q < 0.0) or np.any(q > 1.0):
        raise ValueError("quantile values must be finite and lie in [0, 1], got %s" % list(q))
    return q


def _band_series(series, topo):
    series = list(series)
    if not series:
        raise ValueError("no series: give a list of (sc_id, variable)")
    pos = {s: i for i, s in enumerate(topo.sc_ids)}
    desc = []
    for sc_id, var in series:
        if var not in pk.VAR_INDEX:
            raise ValueError("unknown variable %r: one of %s" % (var, pk.VAR_KINDS))
        try:
            sc_key = int(sc_id)
        except (TypeError, ValueError):
            sc_key = None
        if sc_key not in pos:
            raise ValueError("reach %r is not in SC_list" % (sc_id,))
        desc.append((pos[sc_key], pk.VAR_INDEX[var]))
    return np.asarray(desc, dtype=np.int32).reshape(-1, 2), [(int(s), v) for s, v in series]


def _integrate_in_chunks(eng, d_forc, d_mem, d_sc, topo, opt, members_per_chunk, consume):
    """Integrate the member rows ``d_mem`` [M][NP_MEMBER] / ``d_sc`` [1 or M][S][NP_SC] with the forcing ``d_forc``
    (all on the device) in full-output chunks of ``members_per_chunk`` (default: about 1 GiB of output a chunk) into
    one reused device buffer, and after each chunk enqueue ``consume(out [n][S][D][25], member rows [n], sc rows
    [1 or n], diag rows [n], first member)``, which reads the chunk's output in place before the next chunk overwrites
    it.  Returns the per-member diagnostics [M][S][4] on the device; asynchronous."""
    import torch

    M, S, D = d_mem.shape[0], topo.n_sc, d_forc.shape[0]
    row_bytes = S * D * pk.NOUT * 8
    if members_per_chunk is None:
        members_per_chunk = max(1, (1 << 30) // max(row_bytes, 1))
    chunk = int(max(1, min(int(members_per_chunk), M)))
    out = torch.empty((chunk, S, D, pk.NOUT), dtype=torch.float64, device=eng.device)
    diag = torch.zeros((M, S, pk.NDIAG), dtype=torch.int64, device=eng.device)
    for m0 in range(0, M, chunk):
        n = min(chunk, M - m0)
        scp = d_sc if d_sc.shape[0] == 1 else d_sc[m0:m0 + n]
        eng.run(d_forc, d_mem[m0:m0 + n], scp, topo.parent_offsets, topo.parent_ids, opt, out=out[:n],
                diag=diag[m0:m0 + n])
        consume(out[:n], d_mem[m0:m0 + n], scp, diag[m0:m0 + n], m0)
    return diag


def _n_failed(diag):
    """Members whose integration raised a status bit at any reach (diag after a synchronise)."""
    return int(np.any(diag.cpu().numpy()[:, :, 3] != 0, axis=1).sum())


def predictive_bands(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, samples, series,
                     quantiles=(0.025, 0.25, 0.5, 0.75, 0.975), obs_error=False, seed=DEFAULT_BAND_SEED,
                     members_per_chunk=None, step_len=1.0, rtol=None, atol=None, snow_on_device=False, engine=None):
    """Posterior predictive bands: quantiles over the members of ``samples`` (e.g. ``McmcResult.flat_samples``) of
    the simulated series ``series`` [(sc_id, variable)], variable in ``packing.VAR_KINDS`` — Q_cumecs or a
    concentration in mg/l, the values the fused statistics compare with the observations.

    The members are integrated in full-output chunks of ``members_per_chunk`` (default: about 1 GiB of output a
    chunk); each chunk is turned on the device into its columns of a [V][D][M] matrix of draws, and one selection
    launch gives ``np.nanquantile`` of every (series, day) over the members, bitwise.  With ``obs_error`` every draw
    also carries the likelihood's error model, y = s + m s eps with eps ~ N(0, 1) and m the member's ``err_m:<var>``,
    keyed by ``seed``: a draw depends on (seed, member, day, series) only, not on the chunking.  A member whose
    integration raised a status bit enters no band (``n_failed``).  ``snow_on_device`` as in
    ``calibrate_ensemble``.  AR(1) error-model columns ``err_phi:<var>`` of ``samples`` (a posterior sampled with
    them) are accepted and ignored: the AR(1) process has unit variance, so each day's marginal N(s, (m s)^2) does not
    depend on phi, and neither does a daily quantile.

    Raises ``ValueError`` before any device work for an unknown variable, a reach not in ``SC_list``, an empty
    ``series``, quantile values that are not finite, lie outside [0, 1] or number more than 16, and a matrix of
    draws (8 V D M bytes) larger than half of the free device memory.
    """
    import torch

    from .engine import Engine, check_device_memory

    q = _check_band_quantiles(quantiles)
    inp = _model_inputs(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, step_len, rtol, atol, snow_on_device)
    desc, labels = _band_series(series, inp.topo)
    member, sc = pack_members(inp.member, inp.sc, samples)
    M, D, V = member.shape[0], len(met_df), desc.shape[0]
    eng = engine or Engine()
    check_device_memory(eng, 8 * V * D * M, "the draws need", "thin the samples (e.g. flat_samples(burn, thin=n))")
    dev = eng.device
    d_desc = eng.to_device(desc)
    draws = torch.empty((V, D, M), dtype=torch.float64, device=dev)

    def draw(out, d_mem, scp, diag, m0):
        eng.predictive_draws(out, d_mem, scp, diag, d_desc, draws, m0, obs_error, seed)
    diag = _integrate_in_chunks(eng, eng.to_device(inp.forcing), eng.to_device(member), eng.to_device(sc), inp.topo,
                                inp.opt, members_per_chunk, draw)
    with torch.cuda.device(dev):
        quant, mean, count = eng.nanquantile(draws.view(V * D, M), q)
    torch.cuda.synchronize(dev)
    n_failed = _n_failed(diag)
    return PredictiveBands(q=q, quantiles=quant.cpu().numpy().reshape(len(q), V, D),
                           mean=mean.cpu().numpy().reshape(V, D), count=count.cpu().numpy().reshape(V, D),
                           n_failed=n_failed, labels=labels, dates=met_df.index)


# --------------------------------------------------------------------------- period loads and concentrations
PERIOD_STATISTICS = ("mean", "load", "fwmc")


def period_bounds(dates, periods):
    """``periods`` as (bounds [P][2] int32 = first and last day index of each period, inclusive, labels [P] str).

    ``"year"``: calendar years (labels ``"2004"``), ``"month"``: calendar months (``"2004-01"``), ``"all"``: the whole
    record, or a list of ``(start, end)`` dates, inclusive (labels ``"start/end"``), which may overlap.  A partial
    first or last year or month is kept."""
    import pandas as pd

    idx = pd.DatetimeIndex(dates)
    D = len(idx)
    if D == 0:
        raise ValueError("an empty record has no periods")
    if isinstance(periods, str):
        if periods == "all":
            keys = np.zeros(D, dtype=np.int64)
            names = ["%s/%s" % (idx[0].date(), idx[-1].date())]
        elif periods == "year":
            keys = idx.year.to_numpy()
            names = None
        elif periods == "month":
            keys = idx.year.to_numpy() * 12 + (idx.month.to_numpy() - 1)
            names = None
        else:
            raise ValueError("unknown periods %r: 'year', 'month', 'all' or a list of (start, end) dates" % periods)
        change = np.flatnonzero(np.diff(keys)) + 1
        first = np.concatenate([[0], change])
        last = np.concatenate([change - 1, [D - 1]])
        if names is None:
            names = [str(idx[i].year) if periods == "year" else "%04d-%02d" % (idx[i].year, idx[i].month)
                     for i in first]
        return np.stack([first, last], axis=1).astype(np.int32), names
    ranges = list(periods)
    if not ranges:
        raise ValueError("no periods: give 'year', 'month', 'all' or a list of (start, end) dates")
    bounds, names = [], []
    for rng in ranges:
        try:
            start, end = (pd.Timestamp(t) for t in rng)
        except (TypeError, ValueError):
            raise ValueError("a period is a (start, end) pair of dates, got %r" % (rng,))
        if start > end:
            raise ValueError("period %s/%s is reversed" % (start.date(), end.date()))
        if start < idx[0] or end > idx[-1]:
            raise ValueError("period %s/%s is not inside the record %s/%s"
                             % (start.date(), end.date(), idx[0].date(), idx[-1].date()))
        lo, hi = int(idx.searchsorted(start, "left")), int(idx.searchsorted(end, "right")) - 1
        if hi < lo:
            raise ValueError("period %s/%s holds no day of the record" % (start.date(), end.date()))
        bounds.append((lo, hi))
        names.append("%s/%s" % (start.date(), end.date()))
    return np.asarray(bounds, dtype=np.int32).reshape(-1, 2), names


def _period_series(series, topo, p_struc):
    """(desc [V][3] int32 for ``simplyp_period_aggregates_device``, labels [(target, variable, statistic)],
    run-order water-body reaches)."""
    from . import _cabi

    series = list(series)
    if not series:
        raise ValueError("no series: give a list of (target, variable, statistic)")
    pos = {s: i for i, s in enumerate(topo.sc_ids)}
    desc, labels, wb = [], [], None
    for item in series:
        try:
            target, var, stat = item
        except (TypeError, ValueError):
            raise ValueError("a series is (target, variable, statistic), got %r" % (item,))
        if var not in pk.VAR_INDEX:
            raise ValueError("unknown variable %r: one of %s" % (var, pk.VAR_KINDS))
        if stat not in PERIOD_STATISTICS:
            raise ValueError("unknown statistic %r: one of %s" % (stat, list(PERIOD_STATISTICS)))
        if stat == "fwmc" and var == "Q":
            raise ValueError("the flow-weighted mean concentration of Q is undefined")
        if isinstance(target, str) and target == "waterbody":
            if wb is None:
                flag = p_struc["In_final_flux?"]
                wb = [pos[int(r)] for r in flag[flag == 1].index.values if int(r) in pos]
                if not wb:
                    raise ValueError("'waterbody' needs at least one reach flagged In_final_flux? == 1")
            code, label = _cabi.PERIOD_WATERBODY, "waterbody"
        else:
            try:
                key = int(target)
            except (TypeError, ValueError):
                key = None
            if key not in pos:
                raise ValueError("reach %r is not in SC_list" % (target,))
            code, label = pos[key], key
        desc.append((code, pk.VAR_INDEX[var], _cabi.PERIOD_STATS[stat]))
        labels.append((label, var, stat))
    if len(desc) > _cabi.PERIOD_MAX_SERIES:
        raise ValueError("at most %d series, got %d" % (_cabi.PERIOD_MAX_SERIES, len(desc)))
    if wb is not None and len(wb) > _cabi.PERIOD_MAX_REACHES:
        raise ValueError("at most %d reaches in the water body" % _cabi.PERIOD_MAX_REACHES)
    return np.asarray(desc, dtype=np.int32).reshape(-1, 3), labels, np.asarray(wb or [], dtype=np.int32)


@dataclass
class PeriodStatistics:
    """What :func:`period_statistics` returns.  Row r = v * n_periods + p is series v (``series[v]``, a
    (target, variable, statistic)) over period p (``periods[p]``).  ``values`` [R][M] holds every member's aggregate
    (NaN for the ``n_failed`` members whose integration raised a status bit), ``quantiles`` [n_q][R] is
    ``np.nanquantile(values, q, axis=-1)``, ``mean`` [R] and ``count`` [R] are the mean and the number of the non-NaN
    entries of a row.  ``bounds`` [P][2] are the first and last day index of each period, ``n_days`` [P] its days."""
    q: np.ndarray
    quantiles: np.ndarray
    values: np.ndarray
    mean: np.ndarray
    count: np.ndarray
    n_failed: int
    series: list
    periods: list
    bounds: np.ndarray
    n_days: np.ndarray
    dates: object

    @property
    def labels(self):
        """Row labels: (target, variable, statistic, period), series-major."""
        return [s + (p,) for s in self.series for p in self.periods]

    def row(self, row_or_label):
        """The row index of an int or of a label (target, variable, statistic, period); the period may be given as
        its label or, for a year, as the int year."""
        if isinstance(row_or_label, (int, np.integer)):
            r = int(row_or_label)
            if not 0 <= r < self.values.shape[0]:
                raise ValueError("row %d outside 0..%d" % (r, self.values.shape[0] - 1))
            return r
        lab = tuple(row_or_label)
        if len(lab) != 4:
            raise ValueError("a row label is (target, variable, statistic, period), got %r" % (row_or_label,))
        key = (lab[0], lab[1], lab[2], str(lab[3]))
        for r, l in enumerate(self.labels):
            if l == key:
                return r
        raise ValueError("no row %r" % (row_or_label,))

    def exceedance(self, row_or_label, threshold):
        """Fraction of the finite entries of a row of ``values`` greater than ``threshold`` (NaN if none)."""
        v = self.values[self.row(row_or_label)]
        v = v[np.isfinite(v)]
        return float(np.count_nonzero(v > threshold)) / v.size if v.size else float("nan")

    def table(self):
        """A DataFrame with one row per (target, variable, statistic, period): the period's first and last date and
        number of days, the quantiles (columns ``q<value>``), the mean and the count."""
        import pandas as pd

        P = len(self.periods)
        rows = []
        for r, (target, var, stat, period) in enumerate(self.labels):
            p = r % P
            row = {"target": target, "variable": var, "statistic": stat, "period": period,
                   "start": self.dates[self.bounds[p, 0]], "end": self.dates[self.bounds[p, 1]],
                   "n_days": int(self.n_days[p])}
            for k, qv in enumerate(self.q):
                row["q%g" % qv] = self.quantiles[k, r]
            row["mean"] = self.mean[r]
            row["count"] = int(self.count[r])
            rows.append(row)
        return pd.DataFrame(rows)


def period_statistics(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, samples, series, periods="year",
                      quantiles=(0.025, 0.5, 0.975), members_per_chunk=None, step_len=1.0, rtol=None, atol=None,
                      snow_on_device=False, engine=None):
    """Period loads, flow-weighted mean concentrations and means over the members of ``samples`` (e.g.
    ``McmcResult.flat_samples``), with their quantiles: what a catchment delivers per year, month or any set of date
    ranges, per reach and into the receiving water body, with its uncertainty.

    ``series`` [(target, variable, statistic)]: target a reach id of ``SC_list`` or ``"waterbody"`` (the reaches flagged
    ``In_final_flux? == 1``, summed as ``sum_to_waterbody`` sums them), variable in ``packing.VAR_KINDS``, statistic
      ``"mean"``  mean over the period's days of the daily value (Q_cumecs, or a concentration in mg/l); for a reach the
                  value the fit statistics and ``predictive_bands`` see;
      ``"load"``  sum of the daily flux in kg (for Q the volume in m3, the sum of Q_cumecs * 86400);
      ``"fwmc"``  flow-weighted mean concentration in mg/l, sum of the flux / sum of Q_cumecs * 1000/86400 (not Q).
    ``periods``: ``"year"``, ``"month"``, ``"all"`` or a list of (start, end) dates, inclusive (:func:`period_bounds`).

    The members are integrated in full-output chunks as in :func:`predictive_bands`; each chunk is reduced on the
    device over the days of every period in ascending order (one rounding per addition, so every value is bitwise
    independent of the chunking) into its columns of a [R][M] matrix, R = len(series) * n_periods, series-major, and
    one selection launch gives ``np.nanquantile`` of every row, bitwise.  A member whose integration raised a status
    bit gives NaN in every row (``n_failed``).  AR(1) error-model columns ``err_phi:<var>`` of ``samples`` are accepted
    and ignored: the aggregates are of the simulated series, which do not depend on phi.

    Raises ``ValueError`` before any device work for an unknown variable or statistic, ``"fwmc"`` of Q, a reach not in
    ``SC_list``, ``"waterbody"`` with no flagged reach, an empty ``series``, unknown ``periods``, an explicit range
    that is reversed, not inside the record or holds no day of it, bad quantile values, more series, periods or
    water-body reaches than ``simplyp_period_aggregates_device`` takes, and a values matrix (8 R M bytes) larger than
    half of the free device memory.
    """
    import torch

    from . import _cabi
    from .engine import Engine, check_device_memory

    q = _check_band_quantiles(quantiles)
    inp = _model_inputs(met_df, p_struc, p_SU, p_LU, p_SC, p, dynamic_options, step_len, rtol, atol, snow_on_device)
    desc, labels, wb = _period_series(series, inp.topo, p_struc)
    bounds, names = period_bounds(met_df.index, periods)
    if bounds.shape[0] > _cabi.PERIOD_MAX_PERIODS:
        raise ValueError("at most %d periods, got %d" % (_cabi.PERIOD_MAX_PERIODS, bounds.shape[0]))
    member, sc = pack_members(inp.member, inp.sc, samples)
    M, R = member.shape[0], desc.shape[0] * bounds.shape[0]
    eng = engine or Engine()
    check_device_memory(eng, 8 * R * M, "the values need", "thin the samples (e.g. flat_samples(burn, thin=n)) or ask "
                        "for fewer series or periods")
    dev = eng.device
    values = torch.empty((R, M), dtype=torch.float64, device=dev)

    def aggregate(out, d_mem, scp, diag, m0):
        eng.period_aggregates(out, d_mem, scp, diag, desc, bounds, wb, values, m0)
    diag = _integrate_in_chunks(eng, eng.to_device(inp.forcing), eng.to_device(member), eng.to_device(sc), inp.topo,
                                inp.opt, members_per_chunk, aggregate)
    with torch.cuda.device(dev):
        quant, mean, count = eng.nanquantile(values, q)
    torch.cuda.synchronize(dev)
    return PeriodStatistics(q=q, quantiles=quant.cpu().numpy(), values=values.cpu().numpy(),
                            mean=mean.cpu().numpy(), count=count.cpu().numpy(), n_failed=_n_failed(diag),
                            series=labels, periods=names, bounds=bounds,
                            n_days=(bounds[:, 1] - bounds[:, 0] + 1).astype(np.int64), dates=met_df.index)
