"""NumPy restatement of NSGA-II (simplyp_b200/csrc/simplyp_nsga2.cuh and the NSGA-II kernels): the Philox words, the
tournaments, SBX and polynomial mutation, the orientation of the objectives, the non-dominated ranks, the crowding
distances, the survivors and the history row, and a driver over a Python objective.  The oracle of the NSGA-II
arithmetic in the tests: ranks, crowding, survivors and history agree with the device bit for bit; offspring agree up
to the pow calls of SBX and mutation (OFFSPRING_ULP)."""
import numpy as np

from tests import mcmc_reference as mref

#: Offspring of the device (or the host build) and of this restatement differ by at most this many units in the last
#: place of 1.0 (2^-52): the only inexact calls are pow's, which the device and the host's libm round differently.
OFFSPRING_ULP = 64
EPS = 1e-14
UNRANKED = np.iinfo(np.int32).max


def words(seed, g, pairs, group):
    """The four words of group ``group`` of ``pairs`` (array) at generation g: counter (p, g lo, g hi, 5 + 256 q)."""
    p = np.asarray(pairs, dtype=np.uint64)
    ctr = np.stack([p, np.full_like(p, g & 0xFFFFFFFF), np.full_like(p, (g >> 32) & 0xFFFFFFFF),
                    np.full_like(p, 5 + 256 * group)], axis=1)
    return mref.philox4x32_10(ctr, [seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF])


def _mulhi(w, n):
    return ((w.astype(np.uint64) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


def picks(N, g, seed):
    """[N/2][4] tournament picks a, b, c, d of every pair (b != a, d != c)."""
    w = words(seed, g, np.arange(N // 2), 0)
    out = np.empty((N // 2, 4), dtype=np.int64)
    for t in range(2):
        a = _mulhi(w[:, 2 * t], N)
        b = _mulhi(w[:, 2 * t + 1], N - 1)
        out[:, 2 * t], out[:, 2 * t + 1] = a, b + (b >= a)
    return out


def better(rank, crowd, a, b):
    """Lower rank, then larger crowding, then lower index."""
    ra, rb, ca, cb = rank[a], rank[b], crowd[a], crowd[b]
    a_wins = (ra < rb) | ((ra == rb) & ((ca > cb) | ((ca == cb) & (a < b))))
    return np.where(a_wins, a, b)


def _betaq(beta, rand, eta_c):
    expo = eta_c + 1.0
    alpha = 2.0 - np.power(beta, -expo)
    lo = rand <= 1.0 / alpha
    with np.errstate(all="ignore"):
        return np.where(lo, np.power(rand * alpha, 1.0 / expo), np.power(1.0 / (2.0 - rand * alpha), 1.0 / expo))


def mutate(y, rnd, eta_m):
    expo = eta_m + 1.0
    mut_pow = 1.0 / expo
    with np.errstate(all="ignore"):
        lo = rnd <= 0.5
        val_lo = 2.0 * rnd + (1.0 - 2.0 * rnd) * np.power(1.0 - y, expo)
        val_hi = 2.0 * (1.0 - rnd) + 2.0 * (rnd - 0.5) * np.power(1.0 - (1.0 - y), expo)
        dq = np.where(lo, np.power(val_lo, mut_pow) - 1.0, 1.0 - np.power(val_hi, mut_pow))
    return np.clip(y + dq, 0.0, 1.0)


def offspring(pop, rank, crowd, g, seed, crossover, mutation, eta_c, eta_m):
    """(children [N][K] (pair p: rows 2p, 2p + 1), decisions [N/2][3 + K]: parent 1, parent 2, crossed, then the bits
    SBX 1 / swap 2 / mutate child 1 4 / mutate child 2 8 of every variable)."""
    N, K = pop.shape
    P = N // 2
    pk = picks(N, g, seed)
    p1, p2 = better(rank, crowd, pk[:, 0], pk[:, 1]), better(rank, crowd, pk[:, 2], pk[:, 3])
    w = words(seed, g, np.arange(P), 1)
    cross = mref.u53(w[:, 0], w[:, 1]) < crossover
    dec = np.zeros((P, 3 + K), dtype=np.int64)
    dec[:, 0], dec[:, 1], dec[:, 2] = p1, p2, cross
    out = np.empty((N, K))
    for j in range(K):
        a, b = pop[p1, j].copy(), pop[p2, j].copy()
        w = words(seed, g, np.arange(P), 2 + 4 * j)
        rand = mref.u53(w[:, 2], w[:, 3])
        sbx = cross & (mref.u53(w[:, 0], w[:, 1]) < 0.5) & (np.fabs(a - b) > EPS)
        y1, y2 = np.minimum(a, b), np.maximum(a, b)
        with np.errstate(all="ignore"):
            d = y2 - y1
            v1 = np.clip(0.5 * ((y1 + y2) - _betaq(1.0 + (2.0 * y1) / d, rand, eta_c) * d), 0.0, 1.0)
            v2 = np.clip(0.5 * ((y1 + y2) + _betaq(1.0 + (2.0 * (1.0 - y2)) / d, rand, eta_c) * d), 0.0, 1.0)
        w = words(seed, g, np.arange(P), 3 + 4 * j)
        swap = mref.u53(w[:, 0], w[:, 1]) < 0.5
        a = np.where(sbx, np.where(swap, v2, v1), a)
        b = np.where(sbx, np.where(swap, v1, v2), b)
        bits = sbx * 1 + (sbx & swap) * 2
        for c, x in ((0, a), (1, b)):
            w = words(seed, g, np.arange(P), 4 + c + 4 * j)
            m = mref.u53(w[:, 0], w[:, 1]) < mutation
            out[2 * np.arange(P) + c, j] = np.where(m, mutate(x, mref.u53(w[:, 2], w[:, 3]), eta_m), x)
            bits = bits + m * (4 << c)
        dec[:, 3 + j] = bits
    return out, dec


def orient(y, status, sense):
    """Oriented objectives f [n][M] (larger is better) of y [M][n]: NaN rows where the status is set or a value is not
    finite."""
    f = (np.asarray(sense, dtype=np.float64)[:, None] * y).T.copy()
    bad = np.asarray(status, dtype=bool) | ~np.all(np.isfinite(y), axis=0)
    f[bad] = np.nan
    return f


def dominance(f):
    """D [n][n]: D[j, i] = point j dominates point i (NaN rows dominate nothing and are dominated by nothing)."""
    a, b = f[:, None, :], f[None, :, :]
    return np.all(a >= b, axis=2) & np.any(a > b, axis=2)


def ranks(f, target):
    """The rank kernel: dominator counts, then peeling until >= target points are ranked; infeasible points form the
    last rank when every feasible point is ranked first.  (rank [n] (UNRANKED for points not reached), fronts ranked,
    last rank, points ranked before the last rank)."""
    n = f.shape[0]
    ok = ~np.isnan(f[:, 0])
    D = dominance(f)
    count = D.sum(axis=0)
    rank = np.full(n, UNRANKED, dtype=np.int64)
    cur = np.flatnonzero(ok & (count == 0))
    rank[cur] = 0
    k, ranked = 0, cur.size
    while ranked < target and cur.size > 0:
        active = ok & (rank == UNRANKED)
        count = count - np.where(active, D[cur].sum(axis=0), 0)
        cur = np.flatnonzero(active & (count == 0))
        rank[cur] = k + 1
        ranked += cur.size
        k += 1
    if cur.size == 0 and ranked < target:
        rank[rank == UNRANKED] = k
        return rank, k + 1, k, ranked
    return rank, k + 1, k, ranked - cur.size


def crowding(f, rank):
    """The crowd kernel: per ranked feasible point and objective, the nearest values above and below it in its front's
    order by (f_m, index), the +inf ends, and (next - prev) / (max - min) summed in objective order; 0 elsewhere."""
    n, M = f.shape
    out = np.zeros(n)
    ok = ~np.isnan(f[:, 0]) & (rank != UNRANKED)
    for r in np.unique(rank[ok]):
        F = np.flatnonzero(ok & (rank == r))
        acc = np.zeros(F.size)
        for m in range(M):
            v = f[F, m]
            after = (v[None, :] > v[:, None]) | ((v[None, :] == v[:, None]) & (F[None, :] > F[:, None]))
            before = ~after & (F[None, :] != F[:, None])
            nxt = np.where(after, v[None, :], np.inf).min(axis=1)
            prv = np.where(before, v[None, :], -np.inf).max(axis=1)
            mx, mn = v.max(), v.min()
            with np.errstate(all="ignore"):
                term = np.where(mx == mn, 0.0, (nxt - prv) / (mx - mn))
            term = np.where(~after.any(axis=1) | ~before.any(axis=1), np.inf, term)
            acc = acc + term
        out[F] = acc
    return out


def survivors(rank, crowd, N):
    """The first N points in the order (rank asc, crowding desc, index asc), in ascending index."""
    order = np.lexsort((np.arange(rank.size), -crowd, rank))
    return np.sort(order[:N])


def survive(f, unit, sense, N):
    """One survival over the points f [n][M] with unit rows unit [n][K]: (population, objectives, rank, crowding of the
    N survivors, history row)."""
    rank, n_fronts, _, _ = ranks(f, N)
    crowd = crowding(f, rank)
    keep = survivors(rank, crowd, N)
    fs = f[keep]
    with np.errstate(all="ignore"):
        best = np.where(np.all(np.isnan(fs), axis=0), np.nan, np.nanmax(np.where(np.isnan(fs), -np.inf, fs), axis=0))
    hist = np.concatenate([[np.sum(rank[keep] == 0), n_fronts], np.asarray(sense) * best])
    return unit[keep], (np.asarray(sense)[None, :] * fs), rank[keep], crowd[keep], hist


def run(objective_fn, u0, n_gen, seed, sense, crossover=0.9, mutation=None, eta_c=15.0, eta_m=20.0, start=0):
    """The NSGA-II kernels' run over ``objective_fn`` (unit rows [n][K] -> (y [M][n], status [n] bool)) from the
    unit-cube population ``u0``.  Returns a dict with population, objectives, rank, crowding, history [G + 1][2 + M],
    n_failed and generation."""
    N, K = u0.shape
    mutation = 1.0 / K if mutation is None else mutation
    y, st = objective_fn(u0)
    f = orient(y, st, sense)
    n_failed = int(np.isnan(f[:, 0]).sum())
    pop, obj, rank, crowd, h = survive(f, np.array(u0, dtype=np.float64), sense, N)
    history = [h]
    for g in range(start, start + n_gen):
        kids, _ = offspring(pop, rank, crowd, g, seed, crossover, mutation, eta_c, eta_m)
        y, st = objective_fn(kids)
        fk = orient(y, st, sense)
        n_failed += int(np.isnan(fk[:, 0]).sum())
        fp = np.asarray(sense)[None, :] * obj
        pop, obj, rank, crowd, h = survive(np.concatenate([fp, fk]), np.concatenate([pop, kids]), sense, N)
        history.append(h)
    return dict(population=pop, objectives=obj, rank=rank, crowding=crowd, history=np.array(history),
                n_failed=n_failed, generation=start + n_gen)


def zdt(x, which=1):
    """ZDT1 / ZDT2 objectives (both minimised) of x [n][K] in the unit cube: y [2][n]."""
    g = 1.0 + 9.0 * x[:, 1:].sum(axis=1) / (x.shape[1] - 1)
    f1 = x[:, 0]
    f2 = g * (1.0 - np.sqrt(f1 / g)) if which == 1 else g * (1.0 - (f1 / g) ** 2)
    return np.stack([f1, f2])


def dtlz2(x, M=3):
    """DTLZ2 objectives (minimised) of x [n][K]: y [M][n]; the front is the unit sphere's positive orthant."""
    g = ((x[:, M - 1:] - 0.5) ** 2).sum(axis=1)
    th = x[:, :M - 1] * np.pi / 2
    out = []
    for i in range(M):
        v = 1.0 + g
        for j in range(M - 1 - i):
            v = v * np.cos(th[:, j])
        if i > 0:
            v = v * np.sin(th[:, M - 1 - i])
        out.append(v)
    return np.stack(out)


def igd(points, front):
    """Mean over the analytic front points ``front`` [P][M] of the distance to the nearest of ``points`` [n][M]."""
    d = np.sqrt(((front[:, None, :] - points[None, :, :]) ** 2).sum(axis=2))
    return float(d.min(axis=1).mean())
