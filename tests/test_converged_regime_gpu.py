"""The kernels at the parameters a converged fit reaches (tests/converged_fixtures.py), on every
launch path of the EM step: one EM step, the launch strategies, both likelihood forms, the
observed-data log-likelihood, fold-in, refit and prediction, against the oracle (EM sums, fold-in,
prediction) and against the exact reference (likelihood, log-likelihood).  Needs a B200.

Per-element comparisons allow, besides the relative tolerance, UNDERFLOW per term of the sum:
products that fall into the subnormal range keep only the bits above 2**-1074 in any float64
evaluation, the oracle's included."""
import functools

import numpy as np
import pytest

from oracle import mmsbm_oracle as orc
from tests import converged_fixtures as cf
from tests import exact_reference as ex
from tests import fold_in_reference as fref

pytestmark = pytest.mark.gpu

PARAM_TOL = 1e-10
LOGLIK_TOL = 1e-12

# name: (U, I, K, L, R, S, ratings per user, extra ratings of user 0, EM steps), the launch path
FITTED = {
    "coop_k3": (120, 80, 3, 3, 4, 1, 40, 0, 3000),        # one run, 4-double rows: em_small_kernel
    "k20_s8": (60, 40, 20, 20, 5, 8, 20, 0, 1000),        # six-run and pair groups
    "pieces_k6": (40, 2500, 6, 6, 5, 2, 15, 2600, 1000),  # user 0 > 2048 ratings: pieces and fix-up
    "wide_k40": (20, 17, 40, 36, 5, 2, 17, 0, 1000),      # K, L > 32: small_gemm_kernel, CH >= 2
    "k32_r31": (24, 20, 32, 32, 31, 2, 20, 0, 1000),      # one run per warp at the pair limit
}
# onehot_k16_l32_r25: the factorised likelihood's operand tables just fit (16 R ldk ldl = 200 KB), the
# element-wise kernel's do not, so the runs it takes over read their tables from global memory
CONSTRUCTED = ("onehot_k20", "onehot_k16_l32_r25", "boundary_k8")
ALL = tuple(FITTED) + CONSTRUCTED

# the regime each fitted set must stay in (its first run; the first fit measured 0.80 - 0.96 of the
# memberships of one side exactly 0, 0.84 - 0.998 of omega below eps and 0.53 - 0.97 of pr exactly 0).
# No fit empties a whole (k, l) block of pr: onehot_k20 does.
REGIME_MIN = {"membership_zero": 0.2, "omega_below_eps": 0.8, "pr_zero": 0.4}


@functools.lru_cache(maxsize=None)
def problem(name):
    """(rows, U, I, R, K, L, theta [S,U,K], eta [S,I,L], pr [S,K,L,R])."""
    from mmsbm_b200.engine import Engine
    if name.startswith("onehot"):
        rows, th, et, pr = cf.constructed_one_hot() if name == "onehot_k20" else \
            cf.constructed_one_hot(seed=2, U=30, I=24, K=16, L=32, R=25, N=500)
        return (rows, th.shape[1], et.shape[1], pr.shape[3], th.shape[2], et.shape[2], th, et, pr)
    if name == "boundary_k8":
        rows, th, et, pr = cf.constructed_boundary()
        return (rows, th.shape[1], et.shape[1], pr.shape[3], th.shape[2], et.shape[2], th, et, pr)
    U, I, K, L, R, S, per, heavy, T = FITTED[name]
    rows = cf.planted(7, U, I, K, L, R, per, heavy)
    e = Engine(rows, U, I, R, K, L)
    e.set_params(*cf.start(rows, U, I, K, L, R, S, seed=11))
    e.run(T)
    return (rows, U, I, R, K, L) + e.get_params()


def engine(name):
    from mmsbm_b200.engine import Engine
    rows, U, I, R, K, L, th, et, pr = problem(name)
    e = Engine(rows, U, I, R, K, L)
    e.set_params(th, et, pr)
    return e


def runs(name):
    """The runs checked against the exact reference (first and last: it costs ~3 us per element)."""
    S = problem(name)[6].shape[0]
    return sorted({0, S - 1})


@pytest.mark.parametrize("name", tuple(FITTED))
def test_fitted_sets_are_in_the_converged_regime(name):
    rows, U, I, R, K, L, th, et, pr = problem(name)
    got = cf.regime(rows, th[0], et[0], pr[0])
    got["membership_zero"] = max(got["theta_zero"], got["eta_zero"])
    print(name, {k: round(v, 3) for k, v in got.items()})
    for k, v in REGIME_MIN.items():
        assert got[k] >= v, (k, got[k])
    assert np.all(np.isfinite(th)) and np.all(np.isfinite(et)) and np.all(np.isfinite(pr))


# ------------------------------------------------------------------- one EM step
def check_step(got, want, rel, terms, zero=None, scale=1.0):
    """Within rel (plus UNDERFLOW per term, times ``scale`` where a sum was divided by a small
    total), finite, and exactly 0 where no term is nonzero (``zero``, default: where ``want`` is 0).
    Where the oracle's 0 is an underflow the kernel may hold a subnormal: the floor covers it."""
    got = np.asarray(got)
    assert np.all(np.isfinite(got))
    floor = terms * cf.UNDERFLOW * scale
    assert cf.excess(got, want, rel, floor) <= 0.0, cf.excess(got, want, rel, floor)
    assert np.all(got[want == 0.0 if zero is None else zero] == 0.0)


def support(rows, theta, eta, pr):
    """Where the EM sums have no nonzero term at all (they must be exactly 0 on the GPU too)."""
    one = (theta != 0).astype(float), (eta != 0).astype(float), (pr != 0).astype(float)
    return tuple(x == 0.0 for x in orc.em_sums(rows, *one))


def pr_scale(npr, terms):
    """1 / block total of unnormalised pr sums: normalising divides their underflow error by it.  A
    block whose total is itself within the underflow floor normalises to anything (inf)."""
    tot = npr.sum(axis=2, keepdims=True)
    with np.errstate(divide="ignore"):
        return np.where(tot <= terms * cf.UNDERFLOW, np.inf, 1.0 / np.minimum(tot, 1.0))


@pytest.mark.parametrize("name", ALL)
def test_one_em_step(name):
    from mmsbm_b200 import _lib
    rows, U, I, R, K, L, th, et, pr = problem(name)
    N, S = len(rows), th.shape[0]
    e = engine(name)
    rt, re_, rp = (x.cpu().numpy() for x in e.step_raw(_lib.RAW_THETA | _lib.RAW_ETA_PR))
    e = engine(name)
    e.run(1)
    gt, ge, gp = e.get_params()
    fu = np.repeat(np.maximum(np.bincount(rows[:, 0], minlength=U), 1)[:, None], K, axis=1)
    fi = np.repeat(np.maximum(np.bincount(rows[:, 1], minlength=I), 1)[:, None], L, axis=1)
    for s in range(S):
        nt, ne, npr = orc.em_sums(rows, th[s], et[s], pr[s])
        zt, ze, zp = support(rows, th[s], et[s], pr[s])
        check_step(rt[s][:, :K], nt, PARAM_TOL, N * L, zt)
        check_step(re_[s][:, :L], ne, PARAM_TOL, N * K, ze)
        check_step(rp[s], npr, PARAM_TOL, N, zp)
        t1, e1, p1 = orc.em_iteration(rows, th[s], et[s], pr[s], fu, fi)
        check_step(gt[s], t1, PARAM_TOL, N * L, zt)
        check_step(ge[s], e1, PARAM_TOL, N * K, ze)
        check_step(gp[s], p1, PARAM_TOL, N, zp, pr_scale(npr, N))
        assert np.all(gp[s][zp.all(axis=2)] == 0.0)                # empty blocks normalise to 0
    # the oracle is the yardstick here: it agrees with exact sums on this set (run 0) far inside
    # PARAM_TOL (its sequential sums over a 2600-rating user are ~4e-14 off)
    xt, xe, xp = ex.em_sums(rows, th[0], et[0], pr[0])
    nt, ne, npr = orc.em_sums(rows, th[0], et[0], pr[0])
    for a, b, terms in ((nt, xt, N * L), (ne, xe, N * K), (npr, xp, N)):
        assert cf.excess(a, b, 1e-13, terms * cf.UNDERFLOW) <= 0.0


# ------------------------------------------------------------------- launch strategies
STRATEGIES = (("graph", {"MMSBM_NO_OVERLAP": "1"}), ("overlap", {"MMSBM_FORCE_OVERLAP": "1"}),
              ("queue", {"MMSBM_NO_GRAPH": "1", "MMSBM_NO_OVERLAP": "1", "MMSBM_DYN": "1"}),
              ("queue+overlap", {"MMSBM_FORCE_OVERLAP": "1", "MMSBM_DYN": "1"}))
KNOBS = ("MMSBM_NO_GRAPH", "MMSBM_NO_OVERLAP", "MMSBM_FORCE_OVERLAP", "MMSBM_DYN", "MMSBM_COOP")


@pytest.mark.parametrize("name", ALL)
def test_launch_strategies(name, monkeypatch):
    """MMSBM_NO_GRAPH / MMSBM_FORCE_OVERLAP / MMSBM_DYN give the same bits as plain launches;
    the multi-kernel path (MMSBM_COOP=0) agrees with the cooperative one to 1e-11."""
    rows = problem(name)[0]
    outs = {}
    for label, env in (("plain", {"MMSBM_NO_GRAPH": "1", "MMSBM_NO_OVERLAP": "1", "MMSBM_DYN": "0"}),) \
            + STRATEGIES + (("coop0", {"MMSBM_COOP": "0"}),):
        for k in KNOBS:
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        e = engine(name)
        e.run(9)
        outs[label] = e.get_params()
    for label, _ in STRATEGIES:
        for a, b in zip(outs["plain"], outs[label]):
            np.testing.assert_array_equal(a, b, err_msg=label)
    N = len(rows)
    for a, b in zip(outs["plain"], outs["coop0"]):
        assert cf.excess(b, a, 1e-11, N * cf.UNDERFLOW) <= 0.0
        assert np.array_equal(a == 0.0, b == 0.0)


def test_sharded_engine_with_one_rank_is_bit_identical():
    from mmsbm_b200.parallel import ShardedEngine
    rows, U, I, R, K, L, th, et, pr = problem("k20_s8")
    a = engine("k20_s8")
    a.run(5)
    b = ShardedEngine(rows, U, I, R, K, L)
    b.set_params(th, et, pr)
    b.run(3)
    b.run(2)
    for x, y in zip(a.get_params(), b.get_params()):
        np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(a.likelihood(), b.likelihood())
    b.close()


# ------------------------------------------------------------------- likelihood and log-likelihood
@pytest.mark.parametrize("name", ALL)
def test_likelihood_both_forms_against_exact(name, monkeypatch):
    """|got - exact| <= 1e-8 |exact| + 64 ulps of sum |terms| (exact_reference.likelihood_tolerance),
    for the default (factorised, element-wise where its clamp bound does not hold) and the
    element-wise form, with the full and the smallest workspace."""
    import torch
    from mmsbm_b200 import _lib
    rows, U, I, R, K, L, th, et, pr = problem(name)
    N, S = len(rows), th.shape[0]
    e = engine(name)
    fast = e.likelihood()
    need = _lib.C.c_size_t(0)
    _lib.check(e.lib.mmsbm_likelihood_min_workspace_bytes(N, U, I, R, K, L, S, _lib.C.byref(need)), "min ws")
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    out = torch.empty(S, dtype=torch.float64, device="cuda")
    _lib.check(e.lib.mmsbm_likelihood(e.useg.data_ptr(), e.uadj.data_ptr(), e.usched.data_ptr(), N, U, I, R, K, L, S,
                                      e.theta.data_ptr(), e.eta.data_ptr(), e.pr.data_ptr(), out.data_ptr(),
                                      ws.data_ptr(), need.value, torch.cuda.current_stream().cuda_stream), "lik")
    np.testing.assert_array_equal(out.cpu().numpy(), fast)
    monkeypatch.setenv("MMSBM_LIK_ELEMENTWISE", "1")
    slow = e.likelihood()
    monkeypatch.delenv("MMSBM_LIK_ELEMENTWISE")
    for s in runs(name):
        exact = ex.likelihood(rows, th[s], et[s], pr[s])
        tol = ex.likelihood_tolerance(rows, th[s], et[s], pr[s], exact)
        print(f"{name} run {s}: exact {exact:.12e} factorised {fast[s] - exact:+.3e} "
              f"element-wise {slow[s] - exact:+.3e} tolerance {tol:.3e}")
        assert abs(slow[s] - exact) <= tol
        assert abs(fast[s] - exact) <= tol


@pytest.mark.parametrize("name", ALL)
def test_loglik_against_exact(name):
    rows, U, I, R, K, L, th, et, pr = problem(name)
    """LOGLIK_TOL relative, plus 64 ulps per rating: a fit that predicts every rating with certainty
    has S_n = 1 up to rounding and a log-likelihood of about 0."""
    got = engine(name).loglik()
    for s in runs(name):
        want = ex.loglik(rows, th[s], et[s], pr[s])
        assert abs(got[s] - want) <= LOGLIK_TOL * abs(want) + 64 * 2.0 ** -53 * len(rows), (s, got[s], want)


# k20_s8 still moves after 1000 steps; wide_k40 has a log-likelihood of ~1e-14 (see above), which a
# relative tolerance does not settle
@pytest.mark.parametrize("name", ("coop_k3", "pieces_k6", "k32_r31"))
def test_converge_from_a_fitted_set_stops_at_the_first_check(name):
    e = engine(name)
    iters, conv, trace = e.run_converge(200, tol=1e-6, check_every=10)
    print(name, iters, trace[:, :3])
    assert np.all(iters == 10) and np.all(conv)


# ------------------------------------------------------------------- fold-in
def start_sums(rows, side, init, fixed, pr):
    """S_n of every new row at the fold-in start (the new ids' ``init`` rows)."""
    if side == 0:
        return np.einsum("nk,nl,kln->n", init[rows[:, 0]], fixed[rows[:, 1]], pr[:, :, rows[:, 2]])
    return np.einsum("nk,nl,kln->n", fixed[rows[:, 0]], init[rows[:, 1]], pr[:, :, rows[:, 2]])


@pytest.mark.parametrize("side", [0, 1])
def test_fold_in_against_reference(side):
    """New users (side 0) / items (side 1) against converged eta / theta and pr, with one id per path
    of fold_in.cu: a warp (<= 192 rows of 8 doubles), a CTA (<= 1536) and pieces.  Side 0 draws the
    rows at random: the converged model calls many of them impossible.  Side 1 starts the new items
    one-hot, so a row's S_n is sum_k theta_uk p_klr of the hot group l: its rows are picked from
    (user, level) pairs where that is 0, below eps and above it, in turn.  Both sides have rows with
    S = 0 and with 0 < S < eps."""
    rows, U, I, R, K, L, th, et, pr = problem("pieces_k6")
    e = engine("pieces_k6")
    S = th.shape[0]
    g = np.random.default_rng(5 + side)
    degrees = [1, 3, 150, 700, 2000]
    own = np.repeat(np.arange(len(degrees)), degrees)
    width = K if side == 0 else L
    if side == 0:
        new = np.stack([own, g.integers(0, I, len(own)), g.integers(0, R, len(own))], axis=1)
        init = g.random((S, len(degrees), width)) / np.asarray(degrees)[None, :, None]
    else:
        hot = g.integers(0, L, len(degrees))
        init = np.zeros((S, len(degrees), L))
        init[:, np.arange(len(degrees)), hot] = 1.0
        x = np.einsum("uk,klr->ulr", th[0], pr[0])                 # S of a one-hot item in group l
        cols = []
        for a, deg in enumerate(degrees):
            xa = x[:, hot[a], :]
            kinds = [np.argwhere(xa == 0.0), np.argwhere((xa > 0) & (xa < cf.EPS)), np.argwhere(xa >= cf.EPS)]
            kinds = [k for k in kinds if len(k)]
            pick = [kinds[j % len(kinds)][g.integers(0, len(kinds[j % len(kinds)]))] for j in range(deg)]
            cols.append(np.array([[u, a, r] for u, r in pick]))
        new = np.concatenate(cols)
    new = new.astype(np.int64)
    s0 = start_sums(new, side, init[0], et[0] if side == 0 else th[0], pr[0])
    print(f"side {side}: {np.sum(s0 == 0)} rows with S = 0, {np.sum((s0 > 0) & (s0 < cf.EPS))} below eps")
    assert np.sum(s0 == 0) > 0 and np.sum((s0 > 0) & (s0 < cf.EPS)) > 0
    for T in (1, 10):
        got = e.fold_in(side, new, init, T)
        for s in range(S):
            want = fref.fold_in(new, init[s], et[s], pr[s], T, 0) if side == 0 \
                else fref.fold_in(new, th[s], init[s], pr[s], T, 1)
            check_step(got[s], want, PARAM_TOL, T * len(new) * width)


# ------------------------------------------------------------------- refit
@pytest.mark.parametrize("K,L,R,S,U,I,per", [(3, 3, 4, 1, 120, 80, 40), (20, 20, 5, 2, 60, 40, 20)])
def test_refit_from_a_converged_model(K, L, R, S, U, I, per):
    """MMSBM.refit from a model fitted for 1000 steps on planted data, on a set with new ids whose rows
    the model calls impossible, against 10 EM steps from the documented start.

    The steps are taken on exact sums (exact_reference.em_iteration), not by the oracle: at the
    K = L = 20 start a pr block holds [0, 1, 0, 0, 1e-323] and level 1 loses its rows.  The oracle
    rounds (theta eta) p to 0 for that block and empties it; the exact sum is a subnormal at level 4,
    which normalises to [0, 0, 0, 0, 1], and so does the kernel (it factors p out of the sum).  The
    models differ from the second step on, by ~1e-1 on O(1) entries.  Against the exact steps the
    kernel is within 1e-9 (the same association in numpy: ~2e-14 after 10 steps)."""
    from mmsbm_b200 import MMSBM
    from tests.test_refit_gpu import changed_set, documented_start, frame, snapshot
    steps = 10
    rows = cf.planted(3, U, I, K, L, R, per)
    m = MMSBM(K, L, iterations=1000, sampling=S, seed=4)
    m.fit(frame(rows), silent=True)
    pre = snapshot(m.results)
    df, enc, labels = changed_set(rows, U, I, R, seed=6)
    assert m.refit(df, iterations=steps, seed=9) == labels
    U2, I2 = U + 7, I + 5
    fu = np.repeat(np.maximum(np.bincount(enc[:, 0], minlength=U2), 1)[:, None], K, axis=1)
    fi = np.repeat(np.maximum(np.bincount(enc[:, 1], minlength=I2), 1)[:, None], L, axis=1)
    absent_u, absent_i = np.setdiff1d(np.arange(U2), enc[:, 0]), np.setdiff1d(np.arange(I2), enc[:, 1])
    clamped = 0
    for s, (th, et, pr) in enumerate(documented_start(pre, enc, U, I, K, L, seed=9)):
        S0 = orc.omegas(enc, th, et, pr).sum(axis=(1, 2))
        print(f"run {s}: {np.sum(S0 == 0)} rows with S = 0, {np.sum((S0 > 0) & (S0 < cf.EPS))} below eps")
        clamped += int(np.sum(S0 < cf.EPS))
        t, e_, p = th, et, pr
        nz = (th, et, pr)                                  # entries any arithmetic can make nonzero
        for _ in range(steps):
            zt, ze, zp = support(enc, *nz)
            nz = (~zt, ~ze, ~zp)
            npr = ex.em_sums(enc, t, e_, p)[2]
            t, e_, p = ex.em_iteration(enc, t, e_, p, fu, fi)
        zt[absent_u], ze[absent_i] = False, False
        t[absent_u], e_[absent_i] = th[absent_u], et[absent_i]
        got = m.results[s]
        N = len(enc)
        check_step(got["theta"], t, 1e-9, steps * N * L, zt)
        check_step(got["eta"], e_, 1e-9, steps * N * K, ze)
        check_step(got["pr"], p, 1e-9, steps * N, zp, pr_scale(npr, steps * N))
        exact = ex.likelihood(enc, t, e_, p)
        assert abs(got["likelihood"] - exact) <= ex.likelihood_tolerance(enc, t, e_, p, exact)
    assert clamped > 0                                     # the eps clamp is on the path


# ------------------------------------------------------------------- prediction
@pytest.mark.parametrize("name", ALL)
def test_prod_dist_and_argmax(name):
    """prod_dist against the oracle (1e-12 per element); rows the oracle sums to exactly 0 are exactly
    0 (predict_stats drops rows by that test); the argmax is the oracle's wherever the top two levels
    differ by more than 1e-12 relative.  k32_r31 takes the variant that reads pr from global memory."""
    from mmsbm_b200.engine import predict_stats
    rows, U, I, R, K, L, th, et, pr = problem(name)
    g = np.random.default_rng(2)
    test = np.concatenate([rows, np.stack([g.integers(0, U, 2000), g.integers(0, I, 2000),
                                           g.integers(0, R, 2000)], axis=1)])
    rat = engine(name).prod_dist_device(test).cpu().numpy()
    for s in range(th.shape[0]):
        want = orc.rating_distribution(test, th[s], et[s], pr[s])
        assert np.all(np.isfinite(rat[s]))
        assert cf.excess(rat[s], want, 1e-12, K * L * cf.UNDERFLOW * cf.EPS) <= 0.0
        empty = want.sum(axis=1) == 0.0
        assert np.all(rat[s][empty] == 0.0)
        top = np.sort(want, axis=1)[:, -2:]
        clear = (top[:, 1] - top[:, 0]) > 1e-12 * top[:, 1]
        print(f"{name} run {s}: {empty.sum()} all-zero rows, {np.sum(~clear)} near-ties")
        np.testing.assert_array_equal(np.argmax(rat[s], axis=1)[clear], np.argmax(want, axis=1)[clear])
        stats, pred = predict_stats(rat[s], test[:, 2], want_pred=True)
        assert stats[0]["s2"] >= 0 and pred.shape == (1, len(test))
