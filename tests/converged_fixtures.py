"""Parameter sets of the converged regime, for tests/test_converged_regime_*.py.

Random dense parameters (tests/util.random_params) never get near the edges a long fit reaches:
memberships exactly 0 or one-hot, omega = theta eta p far below eps, empty pr blocks, ratings the
model calls impossible (S_n = 0 or 0 < S_n < eps).  Two kinds of sets reach them here:

* planted problems: ratings drawn from a sharply structured model, many per id, then fitted for
  a long time (by the GPU engine in the GPU tests, by the oracle in the CPU tests);
* constructed sets: one-hot rows with the other entries 0, 1e-9, 1e-30, 1e-300 or subnormal, pr
  slabs with exact zeros and whole empty (k, l) blocks, and pr values that put S_n exactly on
  either side of the eps clamp.
"""
import numpy as np

from oracle import mmsbm_oracle as orc

EPS = orc.EPS
SUBNORMAL = 5e-320


def planted(seed, U, I, K, L, R, per_user, heavy_user=0, alpha=0.05):
    """int64 [N,3] rows from a sharp planted model (Dirichlet(alpha) memberships and pr); every user
    rates ``per_user`` items, user 0 ``heavy_user`` more (with repeats when that exceeds I)."""
    g = np.random.default_rng(seed)
    theta = g.dirichlet(np.full(K, alpha), U)
    eta = g.dirichlet(np.full(L, alpha), I)
    pr = g.dirichlet(np.full(R, alpha), (K, L))
    rows = []
    for u in range(U):
        n = per_user + (heavy_user if u == 0 else 0)
        items = g.choice(I, n, replace=n > I)
        p = np.einsum("k,nl,klr->nr", theta[u], eta[items], pr)
        p /= p.sum(axis=1, keepdims=True)
        r = (p.cumsum(axis=1) > g.random(n)[:, None]).argmax(axis=1)
        rows.append(np.stack([np.full(n, u), items, np.minimum(r, R - 1)], axis=1))
    rows = np.concatenate(rows).astype(np.int64)
    rows[:R, 2] = np.arange(R)                       # every level is used
    return rows


def start(rows, U, I, K, L, R, S, seed):
    """S seeded starting points, the reference's initialisation (oracle.seeded_init)."""
    fu, fi = orc.degree_factors(rows, K, L)
    fu = np.concatenate([fu, np.ones((U - fu.shape[0], K), np.int64)])
    fi = np.concatenate([fi, np.ones((I - fi.shape[0], L), np.int64)])
    out = [orc.seeded_init(seed + s, U, I, K, L, R, fu, fi) for s in range(S)]
    return tuple(np.stack(x) for x in zip(*out))


def oracle_fit(rows, theta, eta, pr, iterations):
    """The oracle's EM loop from one starting point (ids without a rating keep their row)."""
    U, K = theta.shape
    I, L = eta.shape
    fu = np.repeat(np.maximum(np.bincount(rows[:, 0], minlength=U), 1)[:, None], K, axis=1)
    fi = np.repeat(np.maximum(np.bincount(rows[:, 1], minlength=I), 1)[:, None], L, axis=1)
    for _ in range(iterations):
        theta, eta, pr = orc.em_iteration(rows, theta, eta, pr, fu, fi)
    return theta, eta, pr


def one_hot(g, n, k, fill):
    """[n, k] rows with one entry 1 and the others ``fill``."""
    x = np.full((n, k), float(fill))
    x[np.arange(n), g.integers(0, k, n)] = 1.0
    return x


def constructed_one_hot(seed=0, U=40, I=30, K=20, L=20, R=5, N=1000):
    """(rows, theta [S,U,K], eta [S,I,L], pr [S,K,L,R]): one run per fill value of the non-hot
    entries (0, 1e-9, 1e-30, 1e-300, subnormal), pr with whole empty (k, l) blocks and exact zeros
    inside slabs.  User 1 and item 2 have no rating, level R-1 has no row."""
    g = np.random.default_rng(seed)
    rows = np.stack([g.integers(0, U, N), g.integers(0, I, N), g.integers(0, R - 1, N)], axis=1)
    rows[:, 0][rows[:, 0] == 1] = 0
    rows[:, 1][rows[:, 1] == 2] = 3
    fills = [0.0, 1e-9, 1e-30, 1e-300, SUBNORMAL]
    th, et, p = [], [], []
    for s, fill in enumerate(fills):
        t = one_hot(g, U, K, fill)
        e = one_hot(g, I, L, fill)
        t /= t.sum(axis=1, keepdims=True)
        e /= e.sum(axis=1, keepdims=True)
        q = g.dirichlet(np.full(R, 0.3), (K, L))
        q[g.random((K, L, R)) < 0.3] = 0.0                     # exact zeros inside slabs
        q[g.random((K, L)) < 0.2] = 0.0                        # whole empty (k, l) blocks
        th.append(t), et.append(e), p.append(q)
    return rows.astype(np.int64), np.stack(th), np.stack(et), np.stack(p)


# pr values that put S_n = p[k,l,r] exactly on either side of the clamp (one-hot rows: S_n equals it)
BOUNDARY = [0.0, SUBNORMAL, 1e-300, np.nextafter(EPS, 0.0), EPS, np.nextafter(EPS, 1.0)]


def constructed_boundary(seed=1, U=48, I=36, K=8, L=8, R=4, N=600):
    """Exactly one-hot theta and eta (other entries 0): S_n = p[k_u, l_i, r_n].  Each (k, l) block of
    pr holds one of BOUNDARY at some level (the rest of the block renormalised), so ratings land on
    S = 0, subnormal, 1e-300 and the three floats around eps.  User b < 6 sits in row b of pr, whose
    blocks all hold BOUNDARY[b], and 10 of its ratings use the boundary level, so every value is hit.
    User U-1 and item I-1 have no rating.  One run."""
    g = np.random.default_rng(seed)
    ku, li = g.integers(0, K, U), g.integers(0, L, I)
    ku[:len(BOUNDARY)] = np.arange(len(BOUNDARY))   # users 0..5 sit in blocks of rows 0..5
    theta = np.zeros((U, K)); theta[np.arange(U), ku] = 1.0
    eta = np.zeros((I, L)); eta[np.arange(I), li] = 1.0
    pr = g.dirichlet(np.full(R, 0.5), (K, L))
    level = g.integers(0, R, (K, L))
    value = g.integers(0, len(BOUNDARY), (K, L))
    for b in range(len(BOUNDARY)):                   # users 0..5 land on every boundary value
        value[ku[b], :] = b
    for k in range(K):
        for l in range(L):
            rest = [r for r in range(R) if r != level[k, l]]
            pr[k, l, rest] *= (1.0 - BOUNDARY[value[k, l]]) / pr[k, l, rest].sum()
            pr[k, l, level[k, l]] = BOUNDARY[value[k, l]]
    rows = np.stack([g.integers(0, U - 1, N), g.integers(0, I - 1, N), g.integers(0, R, N)], axis=1)
    for b in range(len(BOUNDARY)):                   # 10 ratings of user b at its boundary level
        its = g.integers(0, I - 1, 10)
        rows[b * 10:(b + 1) * 10] = np.stack([np.full(10, b), its, level[ku[b], li[its]]], axis=1)
    return rows.astype(np.int64), theta[None], eta[None], pr[None]


def regime(rows, theta, eta, pr):
    """Shares that tell the converged regime from the easy one (theta/eta/pr of one run)."""
    w = orc.omegas(rows, theta, eta, pr)
    return {"theta_zero": float(np.mean(theta == 0.0)), "eta_zero": float(np.mean(eta == 0.0)),
            "omega_below_eps": float(np.mean(w < EPS)),
            "pr_zero": float(np.mean(pr == 0.0)),
            "pr_empty_block": float(np.mean(pr.sum(axis=2) == 0.0)),
            "theta_one_hot": float(np.mean(np.count_nonzero(theta > 1e-12, axis=1) == 1))}


def excess(got, want, rel, floor=0.0):
    """max over elements of |got - want| - rel |want| - floor (<= 0: within tolerance).  ``floor``
    is an absolute allowance for sums of products that underflow into subnormals, where float64
    itself keeps only the bits above 2**-1074 (see UNDERFLOW)."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    if not got.size:
        return -1.0
    return float(np.max(np.abs(got - want) - rel * np.abs(want) - floor))


# absolute error of one omega / max(S, eps) term whose product underflowed: at most 2**-1074 in
# omega, divided by at least eps = 2**-52
UNDERFLOW = 2.0 ** -1022
