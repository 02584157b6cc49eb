"""CPU reference of MMSBM fold-in, built from the oracle's own formulas (oracle/mmsbm_oracle.py):
each iteration is ``em_sums`` + ``scale_by_degree`` restricted to the rows of the new ids, with the
other side and pr fixed.  Test infrastructure, like the oracle."""
import numpy as np

from oracle import mmsbm_oracle as orc


def fold_in(rows, theta, eta, pr, iterations, side=0):
    """Rows of ids a fitted model has not seen.  ``side`` 0: ``theta`` holds the initial rows of the
    new users (``rows[:, 0]`` indexes them), ``eta`` and ``pr`` are fixed; ``side`` 1: ``eta`` holds
    the initial rows of the new items, ``theta`` and ``pr`` are fixed.  The degrees are those of
    ``rows``, divided out as max(deg, 1) like the reference's degree factors."""
    own = theta if side == 0 else eta
    deg = np.maximum(np.bincount(rows[:, side], minlength=own.shape[0]), 1).astype(np.int64)
    factors = np.repeat(deg[:, None], own.shape[1], axis=1)
    for _ in range(iterations):
        if side == 0:
            own = orc.scale_by_degree(orc.em_sums(rows, own, eta, pr)[0], factors)
        else:
            own = orc.scale_by_degree(orc.em_sums(rows, theta, own, pr)[1], factors)
    return own


def planted(seed, U, I, K, L, R, per_user):
    """Ratings drawn from a planted MMSBM: sparse-ish seeded theta [U,K], eta [I,L], pr [K,L,R];
    each user rates ``per_user`` distinct items, the rating drawn from sum_kl theta eta pr.
    Returns int [U*per_user, 3] rows in user order."""
    g = np.random.default_rng(seed)
    theta = g.dirichlet(np.full(K, 0.2), U)
    eta = g.dirichlet(np.full(L, 0.2), I)
    pr = g.dirichlet(np.full(R, 0.15), (K, L))
    rows = []
    for u in range(U):
        items = g.choice(I, per_user, replace=False)
        p = np.einsum("k,nl,klr->nr", theta[u], eta[items], pr)
        p /= p.sum(axis=1, keepdims=True)
        r = (p.cumsum(axis=1) > g.random(per_user)[:, None]).argmax(axis=1)
        rows.append(np.stack([np.full(per_user, u), items, r], axis=1))
    return np.concatenate(rows).astype(np.int64)
