"""EM to convergence on the B200 (Engine.loglik, Engine.run_converge, fit / refit / cv_fit with tol).

The log-likelihood kernel is checked against numpy on the launch paths of tests/test_refit_gpu.py
(with ids that have no rating) and on every row-stride class of the shape envelope.  The loop is
checked against plain runs: a run that stops after t steps holds exactly the parameters of
``Engine.run(t)`` from the same start, and its trace holds exactly ``Engine.loglik`` after each
check's step count."""
import numpy as np
import pandas as pd
import pytest
from numpy.testing import assert_array_equal

from tests import converge_reference as cref
from tests import fold_in_reference as fref
from tests.test_refit_gpu import SHAPES, SIZES, frame, shape_id
from tests.test_shape_envelope_gpu import envelope_cases, problem
from tests.util import random_params, random_triples

pytestmark = pytest.mark.gpu

LOGLIK_TOL = 1e-12
MAX_IT, EVERY = 61, 4


def holed(shape, seed=31):
    """Rows of a refit-test shape without any rating of users 2 and U-1 and items 4 and I-1."""
    K, L, R, S, heavy = shape
    N, U, I = SIZES[heavy]
    rows = random_triples(seed, N, U, I, R, heavy_tail=heavy)
    keep = ~np.isin(rows[:, 0], [2, U - 1]) & ~np.isin(rows[:, 1], [4, I - 1])
    return rows[keep], U, I


def engine(rows, U, I, K, L, R, params):
    from mmsbm_b200.engine import Engine
    e = Engine(rows, U, I, R, K, L)
    e.set_params(*params)
    return e


def check_loglik(e, rows, params):
    got = e.loglik()
    for s in range(len(got)):
        want = cref.loglik(rows, params[0][s], params[1][s], params[2][s])
        assert abs(got[s] - want) <= LOGLIK_TOL * abs(want), (s, got[s], want)


@pytest.mark.parametrize("shape", SHAPES, ids=shape_id)
def test_loglik_matches_numpy(shape):
    K, L, R, S, _ = shape
    rows, U, I = holed(shape)
    params = random_params(5, U, I, K, L, R, S=S)
    e = engine(rows, U, I, K, L, R, params)
    check_loglik(e, rows, params)
    e.run(3)                                   # and at parameters EM produced (zero rows included)
    check_loglik(e, rows, e.get_params())


def one_per_stride():
    seen, out = set(), []
    for c in envelope_cases():
        ld = 4 * ((max(c[0], c[1]) + 3) // 4)
        if (ld, c[0] >= c[1]) not in seen:
            seen.add((ld, c[0] >= c[1]))
            out.append(c)
    return out


@pytest.mark.parametrize("case", one_per_stride(), ids=lambda c: "K%d_L%d_R%d_S%d" % c)
def test_loglik_envelope(case):
    K, L, R, S = case
    data, (U, I), params = problem(case)
    e = engine(data, U, I, K, L, R, params)
    check_loglik(e, data, params)


def plain_trace(rows, U, I, K, L, R, params):
    """Engine.loglik at steps 0, 4, ..., 60, 61 of plain runs."""
    e = engine(rows, U, I, K, L, R, params)
    out, done = [e.loglik()], 0
    while done < MAX_IT:
        step = min(EVERY, MAX_IT - done)
        e.run(step)
        done += step
        out.append(e.loglik())
    return np.stack(out, axis=1)               # [S, checks + 1]


def spread_tol(plain):
    """A tol (one of the relative changes of the plain trace) at which the runs stop after as many
    different step counts as possible, and after a late one for a single run.  A run that stops at
    the last check and one that never stops both end after MAX_IT steps: they count as one."""
    rel = np.abs(np.diff(plain, axis=1)) / np.abs(plain[:, 1:])

    def stops(tol):
        return [cref.stop_check(t, tol) or len(t) - 1 for t in plain]

    return float(max(np.unique(rel), key=lambda tol: (len(set(stops(tol))), min(stops(tol)))))


@pytest.mark.parametrize("shape", SHAPES, ids=shape_id)
def test_runs_stop_like_plain_runs(shape):
    K, L, R, S, _ = shape
    rows, U, I = holed(shape)
    params = random_params(9, U, I, K, L, R, S=S)
    plain = plain_trace(rows, U, I, K, L, R, params)
    tol = spread_tol(plain)
    e = engine(rows, U, I, K, L, R, params)
    iters, conv, trace = e.run_converge(MAX_IT, tol, EVERY)
    got = e.get_params()
    assert trace.shape == (S, plain.shape[1])
    stops = set()
    for s in range(S):
        j = cref.stop_check(plain[s], tol)
        t = MAX_IT if j is None else min(j * EVERY, MAX_IT)
        stops.add(t)
        assert conv[s] == (j is not None) and iters[s] == t, (s, j, iters[s], conv[s])
        last = len(plain[s]) - 1 if j is None else j
        assert_array_equal(trace[s, :last + 1], plain[s, :last + 1])
        assert np.isnan(trace[s, last + 1:]).all()
        ref = engine(rows, U, I, K, L, R, params)
        ref.run(t)
        want = ref.get_params()
        for k, name in enumerate(("theta", "eta", "pr")):
            assert_array_equal(got[k][s], want[k][s], err_msg=f"run {s} {name} after {t} steps")
    assert S == 1 or len(stops) > 1, stops


@pytest.mark.parametrize("shape", SHAPES, ids=shape_id)
def test_tol_zero_runs_to_max_and_repeats(shape):
    K, L, R, S, _ = shape
    rows, U, I = holed(shape)
    params = random_params(13, U, I, K, L, R, S=S)
    e = engine(rows, U, I, K, L, R, params)
    iters, conv, trace = e.run_converge(MAX_IT, 0.0, EVERY)
    assert (iters == MAX_IT).all() and not conv.any()
    ref = engine(rows, U, I, K, L, R, params)
    ref.run(MAX_IT)
    for got, want in zip(e.get_params(), ref.get_params()):
        assert_array_equal(got, want)
    tol = float(np.nanmedian(np.abs(np.diff(trace, axis=1)) / np.abs(trace[:, 1:])))
    outs = []
    for _ in range(2):
        x = engine(rows, U, I, K, L, R, params)
        outs.append(x.run_converge(MAX_IT, tol, EVERY) + x.get_params())
    for a, b in zip(*outs):
        assert_array_equal(a, b)


def test_planted_trace_never_decreases():
    from mmsbm_b200.engine import Engine
    K, L, R, S = 20, 20, 5, 8
    rows = fref.planted(4, 600, 400, K, L, R, per_user=40)
    e = Engine(rows, 600, 400, R, K, L)
    e.set_params(*random_params(2, 600, 400, K, L, R, S=S))
    iters, conv, trace = e.run_converge(200, 0.0, 10)
    for s in range(S):
        t = trace[s][~np.isnan(trace[s])]      # tol = 0 stops a run only where l repeats exactly
        assert len(t) == -(-iters[s] // 10) + 1
        d = np.diff(t)
        assert (d >= -1e-12 * np.abs(t[1:])).all(), (s, d.min())


def df(seed=3):
    rows = fref.planted(seed, 300, 200, 6, 6, 5, per_user=25)
    return frame(rows)


def check_keys(results, max_it, check_every=10):
    for r in results:
        assert isinstance(r["iterations"], int) and isinstance(r["converged"], bool)
        assert 1 <= r["iterations"] <= max_it
        assert r["converged"] or r["iterations"] == max_it
        lik = r["loglik"]
        assert not np.isnan(lik).any()
        assert len(lik) == -(-r["iterations"] // check_every) + 1
        assert np.isfinite(r["likelihood"])


def test_fit_refit_cv_fit_keys_and_save_load(tmp_path):
    from mmsbm_b200 import MMSBM
    data = df()
    m = MMSBM(6, 6, iterations=300, sampling=3, seed=1)
    m.fit(data, silent=True, tol=1e-3)
    check_keys(m.results, 300)
    assert any(r["converged"] for r in m.results)
    test = data.sample(400, random_state=0)
    before = m.predict(test)
    path = str(tmp_path / "m.npz")
    m.save(path)
    assert_array_equal(MMSBM.load(path).predict(test), before)
    m.refit(data, iterations=100, tol=1e-6, check_every=6)
    check_keys(m.results, 100, 6)
    plain = MMSBM(6, 6, iterations=300, sampling=3, seed=1)
    plain.fit(data, silent=True)
    assert not ({"iterations", "converged", "loglik"} & set(plain.results[0]))
    c = MMSBM(6, 6, iterations=200, sampling=2, seed=1)
    acc = c.cv_fit(data, folds=2, tol=1e-4)
    assert len(acc) == 2
    check_keys(c.results, 200)


def test_debug_logs_checks():
    import logging
    from mmsbm_b200 import MMSBM
    m = MMSBM(6, 6, iterations=40, sampling=1, seed=1, debug=True)
    seen = []
    sink = logging.Handler(logging.DEBUG)
    sink.emit = lambda record: seen.append(record.getMessage())
    m.logger.addHandler(sink)
    m.logger.setLevel(logging.DEBUG)
    try:
        m.fit(df(), silent=True, tol=0.0)
    finally:
        m.logger.removeHandler(sink)
    assert sum("Log-likelihood at run 0" in x for x in seen) == 5


def test_every_new_kernel_variant_is_launched():
    """The log-likelihood pass of every lane-group size (1..8 lanes, rows of 4..32 doubles and the
    sliced wide rows) and the three kernels of the loop are launched by the envelope sweep above and
    one run_converge call."""
    import re
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for case in one_per_stride():
            K, L, R, S = case
            data, (U, I), params = problem(case)
            engine(data, U, I, K, L, R, params).loglik()
        rows, U, I = holed(SHAPES[2])
        engine(rows, U, I, 20, 20, 5, random_params(1, U, I, 20, 20, 5, S=2)).run_converge(8, 1e-3, 4)
        torch.cuda.synchronize()
    launched = {re.sub(r"\((?:int|bool)\)|\s", "", ev.key).split("(")[0].split("::")[-1]
                for ev in prof.key_averages()}
    want = ["loglik_pass_kernel<%d>" % g for g in range(1, 9)] + \
        ["converge_init_kernel", "converge_latch_kernel", "converge_copy_kernel"]
    missing = [k for k in want if not any(n.startswith(k) for n in launched)]
    assert not missing, (missing, sorted(launched))

