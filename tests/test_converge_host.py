"""Host side of MMSBM.fit(tol=...): the premise of the stopping rule (EM never lowers the
observed-data log-likelihood, checked with the oracle's EM) and the argument checks, which run
before any GPU work."""
import numpy as np
import pandas as pd
import pytest

import mmsbm_b200.mmsbm as mmsbm_mod
from oracle import mmsbm_oracle as orc
from tests import converge_reference as cref
from tests import fold_in_reference as fref


def test_oracle_em_never_lowers_loglik():
    K, L, R = 4, 3, 3
    rows = fref.planted(3, 60, 40, K, L, R, per_user=12)
    U, I = 60, 40
    fu, fi = orc.degree_factors(rows, K, L)
    _, kids = orc.child_seeds(7, 2)
    for kid in kids:
        theta, eta, pr = orc.seeded_init(kid, U, I, K, L, R, fu, fi)
        prev = cref.loglik(rows, theta, eta, pr)
        for _ in range(40):
            theta, eta, pr = orc.em_iteration(rows, theta, eta, pr, fu, fi)
            cur = cref.loglik(rows, theta, eta, pr)
            assert cur >= prev - 1e-12 * abs(prev), (cur, prev)
            prev = cur


def test_stop_check():
    assert cref.stop_check([-10.0, -5.0, -4.0, -3.999], 1e-3) == 3
    assert cref.stop_check([-10.0, -5.0, -4.0], 1e-6) is None
    assert cref.stop_check([-10.0, -10.0], 0.0) == 1
    assert cref.stop_check([-10.0], 1.0) is None


def frame():
    g = np.random.default_rng(0)
    return pd.DataFrame({"users": g.integers(0, 20, 200), "items": g.integers(0, 15, 200),
                         "ratings": g.integers(1, 4, 200)})


@pytest.mark.parametrize("tol, check_every", [(-1e-6, 10), (float("nan"), 10), (float("inf"), 10), ("1e-4", 10),
                                              (True, 10), (1e-4, 0), (1e-4, 1), (1e-4, 3), (1e-4, -2),
                                              (1e-4, 4.0), (None, 5)])
def test_bad_arguments_are_refused_before_gpu_work(tol, check_every):
    m = mmsbm_mod.MMSBM(2, 2, iterations=10, sampling=1, seed=0)
    with pytest.raises(ValueError):
        m.fit(frame(), silent=True, tol=tol, check_every=check_every)
    with pytest.raises(ValueError):
        m.cv_fit(frame(), folds=2, tol=tol, check_every=check_every)
    m.results = [{}]                       # refit checks its arguments right after "is it fitted"
    with pytest.raises(ValueError):
        m.refit(frame(), tol=tol, check_every=check_every)


def test_rating_sharded_tol_is_refused(monkeypatch):
    m = mmsbm_mod.MMSBM(2, 2, iterations=10, sampling=2, seed=0, shard="ratings")
    monkeypatch.setattr(mmsbm_mod, "dist_info", lambda: (0, 2))
    with pytest.raises(ValueError, match="shard='ratings'"):
        m.fit(frame(), silent=True, tol=1e-4)
    with pytest.raises(ValueError, match="shard='ratings'"):
        m.cv_fit(frame(), folds=2, tol=1e-4)
    m.results = [{}]
    with pytest.raises(ValueError, match="shard='ratings'"):
        m.refit(frame(), tol=1e-4)
    m.shard = "runs"
    m._check_convergence_args(1e-4, 10)    # runs sharded over ranks: accepted
