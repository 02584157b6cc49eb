"""CPU checks of the converged-regime yardsticks (tests/exact_reference.py,
tests/converged_fixtures.py): the exact reference agrees with the oracle where the oracle is
accurate, the oracle's EM sums agree with exact sums on the converged sets (so a GPU failure on
them is the kernel's), and the likelihood criterion of the GPU tests tells the factorised form's
dropped clamps from rounding."""
import numpy as np
import pytest

from oracle import mmsbm_oracle as orc
from tests import converged_fixtures as cf
from tests import exact_reference as ex
from tests.util import random_params, random_triples


def xlogx(x):
    safe = np.where(x > 0, x, 1.0)
    return np.where(x > 0, x * np.log(safe), 0.0)


def factorised_likelihood(rows, theta, eta, pr):
    """float64 algebra of lik_pass_kernel: sum_n T_n - S_n log max(S_n, eps) with
    T_n = sum_kl w log w expanded through log theta + log eta + log p (no clamp)."""
    u, i, r = rows.T
    p = np.moveaxis(pr, 2, 0)[r]
    W = np.einsum("nk,nkl->nl", theta[u], p)
    A = np.einsum("nk,nkl->nl", xlogx(theta[u]), p) + np.einsum("nk,nkl->nl", theta[u], xlogx(p))
    S = np.sum(W * eta[i], axis=1)
    T = np.sum(A * eta[i], axis=1) + np.sum(W * xlogx(eta[i]), axis=1)
    return float(np.sum(T - S * np.log(np.maximum(S, ex.EPS))))


def elementwise_likelihood(rows, theta, eta, pr):
    """float64 algebra of likelihood_kernel: per rating sum_kl w~ lw - log S~ * sum_kl w~, with
    lw = log eps for a clamped element and log theta + log eta + log p otherwise."""
    u, i, r = rows.T
    w = orc.omegas(rows, theta, eta, pr)
    with np.errstate(divide="ignore"):
        lw = np.log(theta[u])[:, :, None] + np.log(eta[i])[:, None, :] + np.log(np.moveaxis(pr, 2, 0)[r])
    small = w < ex.EPS
    wc = np.where(small, ex.EPS, w)
    lw = np.where(small, np.log(ex.EPS), lw)
    s1 = np.sum(wc * lw, axis=(1, 2))
    return float(np.sum(s1 - np.log(np.maximum(w.sum(axis=(1, 2)), ex.EPS)) * wc.sum(axis=(1, 2))))


@pytest.mark.parametrize("K,L,R,heavy", [(20, 20, 5, False), (7, 5, 4, True), (3, 32, 6, False)])
def test_exact_reference_matches_the_oracle_on_random_parameters(K, L, R, heavy):
    N, U, I = 1500, 80, 60
    rows = random_triples(5, N, U, I, R, heavy_tail=heavy)
    theta, eta, pr = random_params(6, U, I, K, L, R)
    for exact, oracle in ((ex.likelihood(rows, theta, eta, pr), orc.likelihood(rows, theta, eta, pr)),
                          (ex.loglik(rows, theta, eta, pr),
                           np.sum(np.log(np.maximum(orc.omegas(rows, theta, eta, pr).sum(axis=(1, 2)), ex.EPS))))):
        assert abs(exact - oracle) <= 1e-13 * abs(exact), (exact, oracle)


def oracle_fitted():
    """Planted sets fitted by the oracle's EM: K = L = 3 near-deterministic and K = L = 8."""
    out = []
    for (U, I, K, L, R, per, T) in ((100, 60, 3, 3, 4, 30, 1500), (50, 40, 8, 8, 5, 25, 600)):
        rows = cf.planted(7, U, I, K, L, R, per)
        th, et, pr = cf.start(rows, U, I, K, L, R, 1, seed=11)
        out.append((rows,) + cf.oracle_fit(rows, th[0], et[0], pr[0], T))
    return out


def sets():
    rows, th, et, pr = cf.constructed_one_hot()
    out = [(rows, th[s], et[s], pr[s]) for s in range(th.shape[0])]
    rows, th, et, pr = cf.constructed_boundary()
    return out + [(rows, th[0], et[0], pr[0])] + oracle_fitted()


def test_fixtures_are_in_the_converged_regime():
    for rows, th, et, pr in sets():
        got = cf.regime(rows, th, et, pr)
        assert got["omega_below_eps"] > 0.5 and got["pr_zero"] > 0.03, got
    rows, th, et, pr = cf.constructed_boundary()
    S = orc.omegas(rows, th[0], et[0], pr[0]).sum(axis=(1, 2))
    for b in cf.BOUNDARY:                              # every value around the clamp is hit exactly
        assert np.any(S == b), b


def test_oracle_em_sums_match_exact_sums():
    """<= 1e-14 per element, plus cf.UNDERFLOW per term where products underflow."""
    for rows, th, et, pr in sets():
        N, K, L = len(rows), th.shape[1], et.shape[1]
        for got, want, terms in zip(orc.em_sums(rows, th, et, pr), ex.em_sums(rows, th, et, pr), (N * L, N * K, N)):
            assert cf.excess(got, want, 1e-14, terms * cf.UNDERFLOW) <= 0.0


def test_likelihood_criterion_outcomes():
    """At one-hot K = L = 20 rows whose other entries are 1e-9, the oracle and the element-wise
    algebra meet the criterion and the factorised algebra (w log w for clamped elements) does not;
    on random parameters all three do."""
    g = np.random.default_rng(3)
    N, U, I, K, L, R = 1000, 60, 50, 20, 20, 5
    rows = random_triples(1, N, U, I, R)
    theta, eta, pr = random_params(2, U, I, K, L, R)
    hot = (cf.one_hot(g, U, K, 1e-9), cf.one_hot(g, I, L, 1e-9), pr)
    for params, fact_ok in (((theta, eta, pr), True), (hot, False)):
        exact = ex.likelihood(rows, *params)
        tol = ex.likelihood_tolerance(rows, *params, exact=exact)
        assert abs(orc.likelihood(rows, *params) - exact) <= tol
        assert abs(elementwise_likelihood(rows, *params) - exact) <= tol
        assert (abs(factorised_likelihood(rows, *params) - exact) <= tol) == fact_ok


def test_an_underflowing_pr_block_keeps_its_level_in_exact_sums():
    """A converged block pr[k, l] = [0, 1, 0, 0, 1e-323] whose level 1 has lost its rows: the exact
    n_pr of the block, 0.2 * 1e-323 / S_n, rounds to subnormals at level 4 and normalises to
    [0, 0, 0, 0, 1].  The oracle rounds (theta eta) p to 0 before it divides by S_n, and empties
    the block.  The GPU kernels factor
    p out of the sum and keep the level, like the exact step."""
    K = L = 2
    R = 5
    theta = np.array([[0.4, 0.6], [0.5, 0.5]])      # rating (0, 0, 4): theta eta p = 0.2 * 1e-323
    eta = np.array([[0.5, 0.5], [1.0, 0.0]])
    pr = np.full((K, L, R), 0.2)
    pr[0, 0] = [0.0, 1.0, 0.0, 0.0, 1e-323]
    rows = np.array([[0, 0, 4], [1, 1, 0], [1, 0, 2], [0, 1, 3]])
    fu, fi = orc.degree_factors(rows, K, L)
    exact = ex.em_iteration(rows, theta, eta, pr, fu, fi)[2]
    oracle = orc.em_iteration(rows, theta, eta, pr, fu, fi)[2]
    np.testing.assert_array_equal(exact[0, 0], [0.0, 0.0, 0.0, 0.0, 1.0])
    np.testing.assert_array_equal(oracle[0, 0], np.zeros(R))
    np.testing.assert_array_equal(exact[1], oracle[1])
