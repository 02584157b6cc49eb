"""MMSBM.refit on the B200: continuation of a fit is bit-exact, a refit on a changed rating set
(dropped ids, new ids, an empty rating level) matches the oracle's EM from the documented start,
restored and folded-in models refit, and a refit with more data predicts at least as well.

Refit sets are the first input from MMSBM in which some ids have no rating at all, among them the
last codes, so the oracle test runs on every launch path of the EM kernels: the cooperative
one-launch path, the multi-kernel path with segments cut into pieces, pair and six-run groups and
more than 32 groups."""
import numpy as np
import pandas as pd
import pytest
from numpy.testing import assert_array_equal

from oracle import mmsbm_oracle as orc
from tests import fold_in_reference as fref
from tests.util import random_triples, rel_err

pytestmark = pytest.mark.gpu

PARAM_TOL = 1e-9          # tests/test_em_gpu.py after several iterations (1e-10 for one)
LIK_TOL = 1e-8

# (K, L, R, S, heavy-tailed ids)
SHAPES = [(6, 5, 5, 1, False),        # cooperative one-launch path (em_small.cu)
          (20, 20, 5, 8, True),       # multi-kernel path, six-run and pair groups, long segments
          (20, 20, 5, 2, True),       # pair groups
          (20, 20, 5, 6, False),      # six-run groups
          (40, 36, 5, 2, False)]      # more than 32 groups
SIZES = {False: (4000, 150, 90), True: (24000, 500, 240)}     # N, U, I


def shape_id(s):
    return "K%d_L%d_R%d_S%d%s" % (s[:4] + ("_heavy" if s[4] else "",))


def frame(rows):
    """String labels whose sorted order is the numeric order, so label k has code k."""
    return pd.DataFrame({"users": ["u%05d" % u for u in rows[:, 0]],
                         "items": ["i%05d" % i for i in rows[:, 1]], "ratings": rows[:, 2] + 1})


def snapshot(results):
    return [{k: np.array(v, copy=True) for k, v in r.items()} for r in results]


# ------------------------------------------------------------------- 1. continuation is exact
@pytest.mark.parametrize("shape", SHAPES, ids=shape_id)
def test_continuation_is_exact(shape):
    """fit(a iterations) + refit(same data, b) == fit(a + b): the refit starts from the fitted
    parameters bit for bit and the EM step carries no other state.  a = 9 and b = 6 cross the
    two-iteration graph replay of the small-problem path with an odd count."""
    from mmsbm_b200 import MMSBM
    K, L, R, S, heavy = shape
    N, U, I = SIZES[heavy]
    df = frame(random_triples(21, N, U, I, R, heavy_tail=heavy))
    a = MMSBM(K, L, iterations=9, sampling=S, seed=11)
    a.fit(df, silent=True)
    added = a.refit(df, iterations=6)
    assert added == {"users": [], "items": []}
    assert a.iterations == 9
    b = MMSBM(K, L, iterations=15, sampling=S, seed=11)
    b.fit(df, silent=True)
    for x, y in zip(a.results, b.results):
        for key in ("theta", "eta", "pr"):
            assert_array_equal(x[key], y[key], err_msg=key)
        assert_array_equal(x["likelihood"], y["likelihood"])
    test = df.sample(600, random_state=2)
    assert_array_equal(a.predict(test), b.predict(test))


# ------------------------------------------------------------------- 2. against the oracle
def changed_set(rows, U, I, R, seed):
    """(frame, encoded rows, labels) of a refit set: 80 % of ``rows`` without any row of users
    3 and U-1, items 5 and I-1 and rating level 1, plus rows of 7 new users with known items, 5 new
    items with known users and 6 rows of a new user with a new item.  New users are "v..", new
    items "j.."; their codes follow the known ones in label order."""
    g = np.random.default_rng(seed)
    keep = (g.random(len(rows)) < 0.8) & ~np.isin(rows[:, 0], [3, U - 1]) & ~np.isin(rows[:, 1], [5, I - 1]) \
        & (rows[:, 2] != 1)
    levels = np.array([r for r in range(R) if r != 1])
    known_u = np.setdiff1d(np.arange(U), [3, U - 1])
    known_i = np.setdiff1d(np.arange(I), [5, I - 1])
    parts, labels = [rows[keep]], {"users": ["v%05d" % k for k in range(7)], "items": ["j%05d" % k for k in range(5)]}
    nu_rows = np.repeat(np.arange(7), [1, 2, 3, 10, 25, 4, 1])
    parts.append(np.stack([U + nu_rows, g.choice(known_i, len(nu_rows)), g.choice(levels, len(nu_rows))], 1))
    ni_rows = np.repeat(np.arange(5), [2, 6, 1, 12, 3])
    parts.append(np.stack([g.choice(known_u, len(ni_rows)), I + ni_rows, g.choice(levels, len(ni_rows))], 1))
    parts.append(np.stack([U + g.integers(0, 7, 6), I + g.integers(0, 5, 6), g.choice(levels, 6)], 1))
    enc = np.concatenate(parts).astype(np.int64)
    enc = enc[g.permutation(len(enc))]
    users = np.array(["u%05d" % u if u < U else labels["users"][u - U] for u in enc[:, 0]], dtype=object)
    items = np.array(["i%05d" % i if i < I else labels["items"][i - I] for i in enc[:, 1]], dtype=object)
    df = pd.DataFrame({"users": users, "items": items, "ratings": enc[:, 2] + 1})
    return df, enc, labels


def documented_start(pre, enc, U, I, K, L, seed):
    """theta0 / eta0 / pr0 of every run by the rule of MMSBM.refit."""
    U2, I2 = int(enc[:, 0].max()) + 1, int(enc[:, 1].max()) + 1
    du = np.maximum(np.bincount(enc[:, 0], minlength=U2), 1)[U:, None]
    di = np.maximum(np.bincount(enc[:, 1], minlength=I2), 1)[I:, None]
    out = []
    for res, child in zip(pre, np.random.SeedSequence(seed).spawn(len(pre))):
        rng = np.random.default_rng(child)
        th = np.concatenate([res["theta"], rng.random((U2 - U, K)) / du])
        et = np.concatenate([res["eta"], rng.random((I2 - I, L)) / di])
        out.append((th, et, res["pr"]))
    return out


@pytest.mark.parametrize("shape", SHAPES, ids=shape_id)
def test_against_oracle(shape):
    from mmsbm_b200 import MMSBM
    K, L, R, S, heavy = shape
    N, U, I = SIZES[heavy]
    rows = random_triples(31, N, U, I, R, heavy_tail=heavy)
    m = MMSBM(K, L, iterations=5, sampling=S, seed=4)
    m.fit(frame(rows), silent=True)
    pre = snapshot(m.results)
    df, enc, labels = changed_set(rows, U, I, R, seed=6)
    added = m.refit(df, iterations=10, seed=9)
    assert added == labels
    U2, I2 = U + 7, I + 5
    assert m.p == U2 - 1 and m.m == I2 - 1 and m._dims['n_ratings'] == R
    assert_array_equal(m.train, enc)

    fu = np.repeat(np.maximum(np.bincount(enc[:, 0], minlength=U2), 1)[:, None], K, axis=1)
    fi = np.repeat(np.maximum(np.bincount(enc[:, 1], minlength=I2), 1)[:, None], L, axis=1)
    absent_u, absent_i = np.setdiff1d(np.arange(U), enc[:, 0]), np.setdiff1d(np.arange(I), enc[:, 1])
    assert {3, U - 1} <= set(absent_u.tolist()) and {5, I - 1} <= set(absent_i.tolist())
    for s, (th, et, pr) in enumerate(documented_start(pre, enc, U, I, K, L, seed=9)):
        if heavy and s not in (0, S - 1):              # the oracle is slow at this size: two runs
            continue
        t, e, p = th, et, pr
        for _ in range(10):
            t, e, p = orc.em_iteration(enc, t, e, p, fu, fi)
        t[absent_u], e[absent_i] = th[absent_u], et[absent_i]
        got = m.results[s]
        assert got["theta"].shape == (U2, K) and got["eta"].shape == (I2, L)
        worst = max(rel_err(got["theta"], t), rel_err(got["eta"], e), rel_err(got["pr"], p))
        assert worst < PARAM_TOL, (s, worst)
        want = orc.likelihood(enc, t, e, p)
        assert abs(got["likelihood"] - want) <= LIK_TOL * abs(want), (s, got["likelihood"], want)
        # ids without a row keep their bits; the empty level's slab is zero
        assert_array_equal(got["theta"][absent_u], pre[s]["theta"][absent_u])
        assert_array_equal(got["eta"][absent_i], pre[s]["eta"][absent_i])
        assert np.all(got["pr"][:, :, 1] == 0.0)

    # the engine keeps the new index and the restored rows for predict / likelihood
    th_d, et_d, pr_d = m._engine.get_params()
    for s in range(S):
        assert_array_equal(th_d[s], m.results[s]["theta"])
        assert_array_equal(et_d[s], m.results[s]["eta"])
        assert_array_equal(pr_d[s], m.results[s]["pr"])
    assert_array_equal(m._engine.likelihood(), [r["likelihood"] for r in m.results])
    # decoded indices: the known labels in code order, then the new ones
    m.predict(df.iloc[:300])
    assert list(m.theta.index) == ["u%05d" % u for u in range(U)] + labels["users"]
    assert list(m.eta.index) == ["i%05d" % i for i in range(I)] + labels["items"]


def test_refit_refuses_an_empty_set():
    from mmsbm_b200 import MMSBM
    rows = random_triples(3, 500, 40, 20, 3)
    m = MMSBM(3, 3, iterations=3, sampling=1, seed=1)
    m.fit(frame(rows), silent=True)
    bad = frame(rows[:10]).assign(ratings=99)
    with pytest.raises(ValueError, match="no row"):
        m.refit(bad)
    with pytest.raises(AssertionError, match="fit the model"):
        MMSBM(3, 3).refit(frame(rows))


# ------------------------------------------------------------------- 3. restored and folded-in models
def test_restored_models(tmp_path):
    from mmsbm_b200 import MMSBM
    K, L, R, S = 6, 5, 5, 3
    N, U, I = SIZES[False]
    rows = random_triples(41, N, U, I, R)
    m = MMSBM(K, L, iterations=8, sampling=S, seed=2)
    m.fit(frame(rows), silent=True)
    m.save(str(tmp_path / "fitted.npz"))
    df, enc, labels = changed_set(rows, U, I, R, seed=8)

    loaded = MMSBM.load(str(tmp_path / "fitted.npz"))
    assert loaded.refit(df, iterations=7, seed=3) == m.refit(df, iterations=7, seed=3)
    for x, y in zip(m.results, loaded.results):
        for key in ("theta", "eta", "pr", "likelihood"):
            assert_array_equal(x[key], y[key], err_msg=key)
    assert loaded.data_handler.return_dicts() == m.data_handler.return_dicts()
    test = df.iloc[:400]
    assert_array_equal(loaded.predict(test), m.predict(test))
    loaded.save(str(tmp_path / "refitted.npz"))
    again = MMSBM.load(str(tmp_path / "refitted.npz"))
    assert_array_equal(again.predict(test), m.predict(test))

    # a second refit continues the first: refit(4) + refit(5) == refit(9) from the same model
    one = MMSBM.load(str(tmp_path / "fitted.npz"))
    two = MMSBM.load(str(tmp_path / "fitted.npz"))
    assert one.refit(df, iterations=4, seed=3) == labels
    assert one.refit(df, iterations=5, seed=3) == {"users": [], "items": []}
    two.refit(df, iterations=9, seed=3)
    for x, y in zip(one.results, two.results):
        for key in ("theta", "eta", "pr", "likelihood"):
            assert_array_equal(x[key], y[key], err_msg=key)


def test_zero_iterations_is_the_documented_start(tmp_path):
    from mmsbm_b200 import MMSBM
    K, L, R, S = 6, 5, 5, 2
    N, U, I = SIZES[False]
    rows = random_triples(43, N, U, I, R)
    m = MMSBM(K, L, iterations=6, sampling=S, seed=5)
    m.fit(frame(rows), silent=True)
    pre = snapshot(m.results)
    df, enc, _ = changed_set(rows, U, I, R, seed=10)
    m.refit(df, iterations=0, seed=12)
    for s, (th, et, pr) in enumerate(documented_start(pre, enc, U, I, K, L, seed=12)):
        assert_array_equal(m.results[s]["theta"], th)
        assert_array_equal(m.results[s]["eta"], et)
        assert_array_equal(m.results[s]["pr"], pr)
        assert abs(m.results[s]["likelihood"] - orc.likelihood(enc, th, et, pr)) <= LIK_TOL * abs(
            m.results[s]["likelihood"])


def test_after_fold_in():
    """Ids added by fold_in are known to refit: it adds only the others and starts the folded-in
    ids from their fold-in rows."""
    from mmsbm_b200 import MMSBM
    K, L, R, S = 6, 5, 5, 2
    N, U, I = SIZES[False]
    rows = random_triples(47, N, U, I, R)
    m = MMSBM(K, L, iterations=6, sampling=S, seed=5)
    m.fit(frame(rows), silent=True)
    df, enc, labels = changed_set(rows, U, I, R, seed=14)
    folded = m.fold_in(df[df["users"].str.startswith("v") & df["items"].str.startswith("i")], iterations=5)
    assert folded == {"users": labels["users"], "items": []}
    pre = snapshot(m.results)
    added = m.refit(df, iterations=0)
    assert added == {"users": [], "items": labels["items"]}
    for s in range(S):
        assert_array_equal(m.results[s]["theta"], pre[s]["theta"])
        assert_array_equal(m.results[s]["eta"][:I], pre[s]["eta"])
    m.refit(df, iterations=5)
    assert m._engine.likelihood().shape == (S,)
    assert m.predict(df.iloc[:200]).shape == (200, R)


# ------------------------------------------------------------------- 4. quality
def test_refit_with_more_data_predicts_at_least_as_well():
    """Planted model (tests/fold_in_reference.planted): 10 % of the ratings are held out for
    testing.  The first fit sees 90 % of the rest: the later 10 % are most of the ratings of the
    first 125 users, who arrive with only a few.  The refit on all of it must predict the held-out
    ratings at least as well as the model before it; the planted parameters themselves are printed
    as the ceiling."""
    from mmsbm_b200 import MMSBM
    U, I, K, L, R, per = 1000, 150, 4, 4, 5, 40
    rows = fref.planted(13, U, I, K, L, R, per)
    g = np.random.default_rng(0)
    held = g.random(len(rows)) < 0.1
    later = ~held & (rows[:, 0] < 125) & (g.random(len(rows)) < 0.8)
    first = rows[~held & ~later]
    assert abs(len(first) / (~held).sum() - 0.9) < 0.01
    # test rows of ids the first fit knows, so that both models are scored on the same rows
    tr = rows[held & np.isin(rows[:, 0], first[:, 0]) & np.isin(rows[:, 1], first[:, 1])]
    test = frame(tr)
    m = MMSBM(K, L, iterations=100, sampling=2, seed=7)
    m.fit(frame(first), silent=True)
    m.predict(test)
    before = m.score(silent=True)["stats"]["accuracy"]
    m.refit(frame(rows[~held]), iterations=100)
    m.predict(test)
    after = m.score(silent=True)["stats"]["accuracy"]
    pg = np.random.default_rng(13)                    # the planted parameters: planted()'s first draws
    theta, eta = pg.dirichlet(np.full(K, 0.2), U), pg.dirichlet(np.full(L, 0.2), I)
    pr = pg.dirichlet(np.full(R, 0.15), (K, L))
    planted = np.mean(np.argmax(orc.rating_distribution(tr, theta, eta, pr), axis=1) == tr[:, 2])
    print(f"held-out accuracy: before {before:.4f}, after {after:.4f}, planted {planted:.4f} on {len(tr)} ratings")
    assert len(m.test) == len(tr)
    assert after >= before, (before, after)
