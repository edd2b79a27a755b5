"""NumPy restatement of differential evolution (simplyp_b200/csrc/simplyp_de.cuh and the DE kernels): the Philox words,
the picks, the trials, the energies, the selection and the fixed-order reduction of de_reduce_kernel, driven by a
Python objective.  The oracle of the DE arithmetic in the tests; every floating-point operation is one IEEE operation
in the kernels' order, so the populations, energies and history agree bit for bit."""
import numpy as np

from tests import mcmc_reference as mref

BEST1BIN, RAND1BIN = "best1bin", "rand1bin"
DE_THREADS = 256


def words(seed, g, members, group):
    """The four words of group ``group`` of ``members`` (array) at generation g: counter (i, g lo, g hi, 4 + 256 q)."""
    m = np.asarray(members, dtype=np.uint64)
    ctr = np.stack([m, np.full_like(m, g & 0xFFFFFFFF), np.full_like(m, (g >> 32) & 0xFFFFFFFF),
                    np.full_like(m, 4 + 256 * group)], axis=1)
    return mref.philox4x32_10(ctr, [seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF])


def mulhi(w, n):
    return ((w.astype(np.uint64) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


def dither(seed, g, mutation):
    lo, hi = float(mutation[0]), float(mutation[1])
    w = words(seed, g, [0xFFFFFFFF], 0)
    return lo + (hi - lo) * float(mref.u53(w[:, 0], w[:, 1])[0])


def picks(N, K, g, seed, strategy):
    """(r [N][3] (column 2 = -1 for best1bin), fill [N]): distinct indices other than i, drawn from N - 1, N - 2,
    N - 3 and shifted past the ones already taken."""
    i = np.arange(N, dtype=np.int64)
    w = words(seed, g, i, 0)
    taken = [i]
    r = np.full((N, 3), -1, dtype=np.int64)
    for p in range(3 if strategy == RAND1BIN else 2):
        v = mulhi(w[:, p], N - 1 - p)
        for t in np.sort(np.stack(taken, axis=1), axis=1).T:
            v = v + (v >= t)
        r[:, p] = v
        taken.append(v)
    return r, mulhi(w[:, 3], K)


def trials(pop, best, g, seed, strategy, F, recombination):
    """Unit-cube trials [N][K] of every member at generation g (F: the generation's mutation factor)."""
    N, K = pop.shape
    r, fill = picks(N, K, g, seed, strategy)
    if strategy == RAND1BIN:
        xa, xb, xc = pop[r[:, 0]], pop[r[:, 1]], pop[r[:, 2]]
    else:
        xa, xb, xc = np.broadcast_to(pop[best], pop.shape), pop[r[:, 0]], pop[r[:, 1]]
    out = np.empty_like(pop)
    for j in range(K):
        w = words(seed, g, np.arange(N), 1 + j)
        cross = (mref.u53(w[:, 0], w[:, 1]) < recombination) | (fill == j)
        t = np.where(cross, xa[:, j] + F * (xb[:, j] - xc[:, j]), pop[:, j])
        out[:, j] = np.where((t > 1.0) | (t < 0.0), mref.u53(w[:, 2], w[:, 3]), t)
    return out


def bprime_outside(pop, best, g, seed, strategy, F):
    """How many mutant coordinates b'_j fall outside [0, 1] (crossover or not): redraw opportunities."""
    N, K = pop.shape
    r, _ = picks(N, K, g, seed, strategy)
    if strategy == RAND1BIN:
        b = pop[r[:, 0]] + F * (pop[r[:, 1]] - pop[r[:, 2]])
    else:
        b = pop[best] + F * (pop[r[:, 0]] - pop[r[:, 1]])
    return int(np.count_nonzero((b > 1.0) | (b < 0.0)))


def scale(u, bounds):
    lo, hi = bounds[:, 0], bounds[:, 1]
    v = 0.5 * (lo + hi) + (u - 0.5) * np.fabs(lo - hi)
    return np.where(v < lo, lo, np.where(v > hi, hi, v))


def energies(y, w, failed):
    """E = -sum_r w_r y_r [N] in row order; +inf for failed members, NaN and +inf."""
    acc = np.zeros(y.shape[1])
    for r in range(y.shape[0]):
        acc = acc + w[r] * y[r]
    e = -acc
    e[~(e < np.inf) | np.asarray(failed, dtype=bool)] = np.inf
    return e


def _tree(part):
    s = DE_THREADS // 2
    while s:
        part[:s] = part[:s] + part[s:2 * s]
        s //= 2
    return part[0]


def _strided_sum(x):
    part = np.zeros(DE_THREADS)
    for c in range(0, x.size, DE_THREADS):
        seg = x[c:c + DE_THREADS]
        part[:seg.size] = part[:seg.size] + seg
    return _tree(part)


def reduce(energy, flags):
    """de_reduce_kernel: (best, mean, std of the finite energies, number finite, replaced, failed)."""
    fin = np.abs(energy) < np.inf
    n_fin = int(fin.sum())
    mean = _strided_sum(np.where(fin, energy, 0.0)) / n_fin if n_fin else np.nan
    d = np.where(fin, energy - mean, 0.0) if n_fin else np.zeros_like(energy)
    sd = np.sqrt(_strided_sum(d * d) / n_fin) if n_fin else np.nan
    return (int(np.argmin(energy)), mean, sd, n_fin, int(np.sum(flags & 1)), int(np.sum((flags >> 1) & 1)))


def run(objective_fn, w, u0, bounds, n_gen, seed, strategy=BEST1BIN, mutation=(0.5, 1.0), recombination=0.7,
        tol=0.01, tol_abs=0.0, start=0):
    """The DE kernels' run: ``objective_fn`` (parameter rows [N][K] -> (y [R][N], failed [N] bool)), weights ``w``
    [R], unit-cube population ``u0``.  Returns a dict with population, energy, best, history [G][4], n_failed,
    generation, converged, converged_at."""
    pop = np.array(u0, dtype=np.float64)
    N = pop.shape[0]
    y, failed = objective_fn(scale(pop, bounds))
    energy = energies(y, w, failed)
    best, mean, sd, n_fin, acc, nf = reduce(energy, 2 * (energy == np.inf).astype(np.int64))
    history = [(-energy[best], -mean, sd, float(acc))]
    n_failed, g, converged, converged_at = nf, start, False, None
    for _ in range(n_gen):
        if converged:
            break
        F = dither(seed, g, mutation)
        trial = trials(pop, best, g, seed, strategy, F, recombination)
        y, failed = objective_fn(scale(trial, bounds))
        e_t = energies(y, w, failed)
        ok = e_t <= energy
        pop[ok] = trial[ok]
        energy[ok] = e_t[ok]
        best, mean, sd, n_fin, acc, nf = reduce(energy, ok.astype(np.int64) | 2 * (e_t == np.inf).astype(np.int64))
        history.append((-energy[best], -mean, sd, float(acc)))
        n_failed += nf
        g += 1
        if n_fin == N and sd <= tol_abs + tol * abs(mean):
            converged, converged_at = True, g
    return dict(population=pop, energy=energy, best=best, history=np.array(history), n_failed=n_failed,
                generation=g, converged=converged, converged_at=converged_at)


def rosenbrock(x):
    return np.sum(100.0 * (x[:, 1:] - x[:, :-1] ** 2) ** 2 + (1.0 - x[:, :-1]) ** 2, axis=1)


def sphere(x):
    return np.sum(x * x, axis=1)
