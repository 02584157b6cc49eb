"""numpy reference of the convergence rule of MMSBM.fit(tol=...): the observed-data log-likelihood
EM increases and the per-run stopping rule applied to a trace of it."""
import numpy as np

from oracle import mmsbm_oracle as orc

EPS = np.finfo(float).eps


def loglik(data, theta, eta, pr, chunk=20000):
    """sum_n log max(sum_kl omega[n,k,l], eps) of one run (theta [U,K], eta [I,L], pr [K,L,R])."""
    total = 0.0
    for lo in range(0, len(data), chunk):
        s = orc.omegas(data[lo:lo + chunk], theta, eta, pr).sum(axis=(1, 2))
        total += float(np.sum(np.log(np.maximum(s, EPS))))
    return total


def stop_check(trace, tol):
    """Index j >= 1 of the first check with |l_j - l_{j-1}| <= tol * |l_j|, or None."""
    for j in range(1, len(trace)):
        if abs(trace[j] - trace[j - 1]) <= tol * abs(trace[j]):
            return j
    return None
