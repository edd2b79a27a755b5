"""NumPy restatement of the ensemble sampler (simplyp_b200/csrc/simplyp_mcmc.cuh): Philox4x32-10 and emcee's stretch
move with a uniform prior box, driven by a Python log-probability.  The oracle of the sampler's arithmetic in the
tests; every floating-point operation is one IEEE operation in the kernels' order, so proposals agree bit for bit."""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr [n][4], key [2] or [n][2] (uint32) -> [n][4] uint32 (Salmon et al. 2011, cuRAND's curand_Philox4x32_10)."""
    c = np.asarray(ctr, dtype=np.uint64).reshape(-1, 4)
    k = np.broadcast_to(np.asarray(key, dtype=np.uint64), (c.shape[0], 2))
    c0, c1, c2, c3 = (c[:, i].copy() for i in range(4))
    k0, k1 = k[:, 0].copy(), k[:, 1].copy()
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(W0)) & MASK
            k1 = (k1 + np.uint64(W1)) & MASK
        p0, p1 = M0 * c0, M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
    return np.stack([c0, c1, c2, c3], axis=1).astype(np.uint32)


def words(seed, t, w, block):
    """The four words of block ``block`` of walkers ``w`` (array) at iteration t."""
    w = np.asarray(w, dtype=np.uint64)
    ctr = np.stack([w, np.full_like(w, t & 0xFFFFFFFF), np.full_like(w, (t >> 32) & 0xFFFFFFFF),
                    np.full_like(w, block)], axis=1)
    return philox4x32_10(ctr, [seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF])


def u53(a, b):
    return ((a >> 5).astype(np.float64) * 67108864.0 + (b >> 6).astype(np.float64)) * (1.0 / 9007199254740992.0)


def propose(x, t, half, seed, lo, hi, a=2.0):
    """Proposals of the active half of walkers x [W][K]: (y [H][K], ln z [H], out_of_box [H] bool)."""
    W, K = x.shape
    H = W // 2
    w = np.arange(half * H, half * H + H)
    r = words(seed, t, w, 0)
    j = (1 - half) * H + ((r[:, 0].astype(np.uint64) * np.uint64(H)) >> np.uint64(32)).astype(np.int64)
    u = u53(r[:, 1], r[:, 2])
    s = (a - 1.0) * u + 1.0
    z = (s * s) / a
    xj, xk = x[j], x[w]
    y = xj - z[:, None] * (xj - xk)
    oob = ~np.all((y >= lo) & (y <= hi), axis=1)
    return y, np.log(z), oob


def accept(x, lp, accepted, y, log_z, lp_new, t, half, seed):
    """Metropolis-Hastings step of the active half, in place; returns the decisions [H] bool."""
    W, K = x.shape
    H = W // 2
    w = np.arange(half * H, half * H + H)
    r = words(seed, t, w, 1)
    log_u = np.log(u53(r[:, 0], r[:, 1]))
    with np.errstate(invalid="ignore"):
        diff = ((K - 1) * log_z + lp_new) - lp[w]
        ok = log_u < diff
    x[w[ok]] = y[ok]
    lp[w[ok]] = lp_new[ok]
    accepted[w[ok]] += 1
    return ok


def sample(lp_fn, x0, lo, hi, n_steps, seed, a=2.0, start=0, thin=1):
    """emcee's EnsembleSampler (StretchMove) over ``lp_fn`` ([n][K] -> [n]) with the box prior [lo, hi].
    Returns (chain [n_saved][W][K], chain_lp [n_saved][W], accepted [W], last walkers, last lp)."""
    x = np.array(x0, dtype=np.float64)
    lp = np.asarray(lp_fn(x), dtype=np.float64).copy()
    accepted = np.zeros(x.shape[0], dtype=np.int64)
    chain, chain_lp = [], []
    for t in range(start, start + n_steps):
        for half in (0, 1):
            y, log_z, oob = propose(x, t, half, seed, lo, hi, a)
            lp_new = np.asarray(lp_fn(y), dtype=np.float64).copy()
            lp_new[oob | np.isnan(lp_new)] = -np.inf
            accept(x, lp, accepted, y, log_z, lp_new, t, half, seed)
        if (t + 1) % thin == 0:
            chain.append(x.copy())
            chain_lp.append(lp.copy())
    K = x.shape[1]
    return (np.array(chain).reshape(-1, x.shape[0], K), np.array(chain_lp).reshape(-1, x.shape[0]), accepted, x, lp)


def gaussian_lp(mean, cov):
    """Log-density (up to a constant) of N(mean, cov) as a function [n][K] -> [n]."""
    prec = np.linalg.inv(cov)

    def lp(x):
        d = x - mean
        return -0.5 * np.einsum("ni,ij,nj->n", d, prec, d)
    return lp
