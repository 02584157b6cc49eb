"""Exact evaluation of the reference's likelihood, of the observed-data log-likelihood and of the
EM sums, for the converged-regime tests.  Test infrastructure, like the oracle.

Every float64 input is a dyadic rational, so theta_k * eta_l * p_klr and S_n = sum_kl of them
are formed exactly as Python integers scaled by one power of two per rating.  Each quantity the
reference rounds only at the end is then rounded once from the exact value (int / int true
division is correctly rounded) and the per-rating terms are added with math.fsum.  No
np.longdouble (its width depends on the host) and no third-party package.

Cost: about 3 us per (rating, k, l) element; keep N*K*L per call below ~5e5.
"""
import math

import numpy as np

EPS = float(np.finfo(np.float64).eps)      # 2**-52, the reference's clamp (src/kernels_numpy.py:51)
_EPS_EXP = -52
assert EPS == 2.0 ** _EPS_EXP


def _split(x):
    """float64 array -> (integer mantissas as Python ints, exponents): x = m * 2**e exactly."""
    m, e = np.frexp(np.asarray(x, dtype=np.float64))
    return (m * 2.0 ** 53).astype(np.int64).tolist(), (e.astype(np.int64) - 53).tolist()


def _ratings(data, theta, eta, pr):
    """Per rating: (W [K*L] exact omegas as ints, scale exponent E) with omega_kl = W[kl] * 2**E,
    E <= -52 so that eps = 2**-52 is an integer at that scale too."""
    K, L = theta.shape[1], eta.shape[1]
    tm, te = _split(theta)
    em, ee = _split(eta)
    pm, pe = _split(np.moveaxis(pr, 2, 0).reshape(pr.shape[2], K * L))      # [R][K*L]
    for u, i, r in np.asarray(data, dtype=np.int64).tolist():
        tmu, teu, emi, eei, pmr, per = tm[u], te[u], em[i], ee[i], pm[r], pe[r]
        mant, expo = [], []
        for k in range(K):
            for l in range(L):
                kl = k * L + l
                mant.append(tmu[k] * emi[l] * pmr[kl])
                expo.append(teu[k] + eei[l] + per[kl])
        E = min([e for m, e in zip(mant, expo) if m] + [_EPS_EXP])
        yield [m << (e - E) if m else 0 for m, e in zip(mant, expo)], E


def likelihood(data, theta, eta, pr):
    """sum_n sum_kl w~ log(w~ / S~_n), w~ = max(omega, eps), S~ = max(S_n, eps): the reference's
    formula (src/expectation_maximization.py:157-167).  Each term is float(w~) *
    log1p(round((w~ - S~) / S~)) and is <= 0, so the fsum is within a few ulps of the exact value."""
    terms = []
    for W, E in _ratings(data, theta, eta, pr):
        one = 1 << -E                               # 1.0 at the rating's scale
        eps = 1 << (_EPS_EXP - E)
        S = max(sum(W), eps)
        for w in W:
            w = max(w, eps)
            terms.append((w / one) * math.log1p((w - S) / S))
    return math.fsum(terms)


def loglik(data, theta, eta, pr):
    """sum_n log max(S_n, eps) with S_n exact, rounded once before the logarithm."""
    terms = []
    for W, E in _ratings(data, theta, eta, pr):
        terms.append(math.log(max(sum(W), 1 << (_EPS_EXP - E)) / (1 << -E)))
    return math.fsum(terms)


def conditioning(data, theta, eta, pr):
    """sum_nkl w~ (|log w~| + |log S~_n|): the sum of the magnitudes of what the reference's formula
    adds, the scale of the rounding error any float64 evaluation of it carries."""
    terms = []
    for W, E in _ratings(data, theta, eta, pr):
        one = 1 << -E
        eps = 1 << (_EPS_EXP - E)
        lS = abs(math.log(max(sum(W), eps) / one))
        for w in W:
            w = max(w, eps) / one
            terms.append(w * (abs(math.log(w)) + lS))
    return math.fsum(terms)


def likelihood_tolerance(data, theta, eta, pr, exact=None):
    """What a float64 evaluation of the likelihood must meet: 1e-8 relative to the exact value
    plus 64 ulps of the conditioning sum."""
    exact = likelihood(data, theta, eta, pr) if exact is None else exact
    return 1e-8 * abs(exact) + 64 * 2.0 ** -53 * conditioning(data, theta, eta, pr)


def em_sums(data, theta, eta, pr):
    """(n_theta, n_eta, n_pr) of oracle.em_sums: inc = omega / max(S_n, eps) (omega unclamped),
    each per-rating contribution rounded once from the exact rational, added with fsum."""
    U, K = theta.shape
    I, L = eta.shape
    R = pr.shape[2]
    acc_t = [[[] for _ in range(K)] for _ in range(U)]
    acc_e = [[[] for _ in range(L)] for _ in range(I)]
    acc_p = [[[] for _ in range(R)] for _ in range(K * L)]
    for (u, i, r), (W, E) in zip(np.asarray(data, dtype=np.int64).tolist(), _ratings(data, theta, eta, pr)):
        S = max(sum(W), 1 << (_EPS_EXP - E))
        for k in range(K):
            acc_t[u][k].append(sum(W[k * L:(k + 1) * L]) / S)
        for l in range(L):
            acc_e[i][l].append(sum(W[l::L]) / S)
        for kl in range(K * L):
            acc_p[kl][r].append(W[kl] / S)
    nt = np.array([[math.fsum(c) for c in row] for row in acc_t]).reshape(U, K)
    ne = np.array([[math.fsum(c) for c in row] for row in acc_e]).reshape(I, L)
    npr = np.array([[math.fsum(c) for c in row] for row in acc_p]).reshape(K, L, R)
    return nt, ne, npr


def em_iteration(data, theta, eta, pr, fu, fi):
    """One EM step of the reference (oracle.em_iteration) on the exact sums of ``em_sums``: only the
    degree scaling and the pr normalisation round in float64.  Where the oracle's products
    underflow, a pr block whose exact sum is a few subnormals normalises to a distribution here,
    and to 0 in the oracle; later steps then depend on which one the model got."""
    from oracle import mmsbm_oracle as orc
    nt, ne, npr = em_sums(data, theta, eta, pr)
    return orc.scale_by_degree(nt, fu), orc.scale_by_degree(ne, fi), orc.normalize_pr(npr)
