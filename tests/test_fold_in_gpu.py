"""Fold-in on the B200: Engine.fold_in (csrc/fold_in.cu) against the CPU reference, against the EM
step it restricts, and MMSBM.fold_in end to end (known ids untouched, new ids served, restored
models, cold-start quality)."""
import numpy as np
import pandas as pd
import pytest

from oracle import mmsbm_oracle as orc
from tests import fold_in_reference as fref
from tests.util import random_params, random_triples, rel_err

pytestmark = pytest.mark.gpu

SHAPES = [(10, 10, 5, 3), (20, 20, 5, 8), (7, 5, 4, 1), (3, 32, 6, 2), (33, 9, 5, 1), (40, 36, 5, 2),
          # whole-warp rows of 4 and 8 doubles per lane (fold_in_kernel<32, 4> and <32, 8>)
          (100, 5, 10, 2), (256, 3, 4, 1)]


def caps(width):
    """Rows per warp slice and per CTA of fold_in_kernel (kFoldSliceBytes = 12 KB, 8 warps)."""
    ld = (width + 3) // 4 * 4
    cap_w = 12 * 1024 // (ld * 8)
    return cap_w, 8 * cap_w


def make_case(shape, side, degrees, seed=0):
    """Engine over a random training set with S random runs, plus fold-in rows of new ids with the
    given degrees (neighbours uniform over the known ids, levels 0..R-2: the last level has no rows)
    and seeded initial rows [S, n_new, width]."""
    from mmsbm_b200.engine import Engine
    K, L, R, S = shape
    U, I = 70, 50
    data = random_triples(seed, 2000, U, I, R)
    theta, eta, pr = random_params(seed + 1, U, I, K, L, R, S)
    eng = Engine(data, U, I, R, K, L)
    eng.set_params(theta, eta, pr)
    g = np.random.default_rng(seed + 2)
    n_other = I if side == 0 else U
    own = np.repeat(np.arange(len(degrees)), degrees)
    other = g.integers(0, n_other, len(own))
    level = g.integers(0, max(R - 1, 1), len(own))
    perm = g.permutation(len(own))                       # rows of different ids interleaved
    own, other, level = own[perm], other[perm], level[perm]
    rows = np.stack([own, other, level] if side == 0 else [other, own, level], axis=1).astype(np.int64)
    width = K if side == 0 else L
    init = g.random((S, len(degrees), width)) / np.maximum(np.asarray(degrees), 1)[None, :, None]
    return eng, (theta, eta, pr), rows, init


def degrees_for(kind, width, seed=0):
    g = np.random.default_rng(seed)
    if kind == "uniform":
        return [1] + g.integers(2, 30, 40).tolist()
    cap_w, cap_c = caps(width)
    # heavy tail: one id beyond a CTA's shared memory (cut into pieces), one just beyond, the
    # boundaries of the warp and CTA paths, short ids and a degree-1 id
    return [2 * cap_c + 37, cap_c + 1, cap_c, cap_w + 1, cap_w, 17, 1, 3, 250, 2]


def reference(params, rows, init, iterations, side):
    theta, eta, pr = params
    out = []
    for s in range(init.shape[0]):
        if side == 0:
            out.append(fref.fold_in(rows, init[s], eta[s], pr[s], iterations, side=0))
        else:
            out.append(fref.fold_in(rows, theta[s], init[s], pr[s], iterations, side=1))
    return np.stack(out)


@pytest.mark.parametrize("kind", ["uniform", "heavy"])
@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "K%d_L%d_R%d_S%d" % s)
def test_kernel_matches_reference(shape, side, kind):
    K, L, R, S = shape
    degrees = degrees_for(kind, K if side == 0 else L)
    eng, params, rows, init = make_case(shape, side, degrees)
    for it in (1, 10):
        got = eng.fold_in(side, rows, init, it)
        want = reference(params, rows, init, it, side)
        assert got.shape == want.shape
        assert rel_err(got, want) < 1e-10, (it, rel_err(got, want))


@pytest.mark.parametrize("side", [0, 1])
def test_kernel_matches_reference_400_iterations(side):
    shape = (10, 10, 5, 3)
    eng, params, rows, init = make_case(shape, side, degrees_for("uniform", 10), seed=4)
    got = eng.fold_in(side, rows, init, 400)
    want = reference(params, rows, init, 400, side)
    assert rel_err(got, want) < 1e-8, rel_err(got, want)


def test_kernel_400_iterations_long_segments():
    shape = (20, 20, 5, 2)
    eng, params, rows, init = make_case(shape, 0, degrees_for("heavy", 20), seed=5)
    got = eng.fold_in(0, rows, init, 400)
    want = reference(params, rows, init, 400, 0)
    assert rel_err(got, want) < 1e-8, rel_err(got, want)


@pytest.mark.parametrize("side", [0, 1])
@pytest.mark.parametrize("shape", [(10, 10, 5, 3), (33, 9, 5, 2)], ids=lambda s: "K%d_L%d_R%d_S%d" % s)
def test_one_iteration_is_the_em_step(shape, side):
    """Fold-in of training ids from their current rows, on their own rows, is their row of one
    Engine.run step from the same state."""
    from mmsbm_b200.engine import Engine
    K, L, R, S = shape
    U, I = 90, 60
    data = random_triples(8, 6000, U, I, R, heavy_tail=True)
    theta, eta, pr = random_params(9, U, I, K, L, R, S)
    eng = Engine(data, U, I, R, K, L)
    eng.set_params(theta, eta, pr)
    ids = np.array([0, 1, 2, 7, 30, 55])
    rows = data[np.isin(data[:, side], ids)].copy()
    rows[:, side] = np.searchsorted(ids, rows[:, side])
    init = (theta if side == 0 else eta)[:, ids]
    got = eng.fold_in(side, rows, init, 1)
    eng.run(1)
    th1, et1, _ = eng.get_params()
    want = (th1 if side == 0 else et1)[:, ids]
    assert rel_err(got, want) < 1e-13, rel_err(got, want)


def test_reproducible():
    eng, _, rows, init = make_case((20, 20, 5, 8), 0, degrees_for("heavy", 20), seed=3)
    a = eng.fold_in(0, rows, init, 25)
    b = eng.fold_in(0, rows, init, 25)
    assert np.array_equal(a, b)


# ------------------------------------------------------------------------ MMSBM.fold_in
def frames(seed=1, U=120, I=60, R=5, n=5000, held_users=12, held_items=6):
    """(train, fold-in rows, later rows of the held-out users): string ids, some users and items
    held out of training."""
    g = np.random.default_rng(seed)
    data = random_triples(seed, n, U, I, R)
    df = pd.DataFrame({"users": ["u%d" % u for u in data[:, 0]], "items": ["i%d" % i for i in data[:, 1]],
                       "ratings": data[:, 2] + 1})
    hu = set(g.choice(U, held_users, replace=False).tolist())
    hi = set(g.choice(I, held_items, replace=False).tolist())
    new_u, new_i = np.isin(data[:, 0], list(hu)), np.isin(data[:, 1], list(hi))
    train = df[~new_u & ~new_i]
    cold = df[new_u ^ new_i]
    first = cold.sample(frac=0.6, random_state=seed)
    return train, first, cold.drop(first.index)


def fitted(seed=2, sampling=3, iterations=30, K=6, L=5):
    from mmsbm_b200 import MMSBM
    train, first, later = frames()
    m = MMSBM(K, L, iterations=iterations, sampling=sampling, seed=seed)
    m.fit(train)
    return m, train, first, later


def test_known_ids_untouched_and_new_ids_served():
    m, train, first, later = fitted()
    known = train.sample(400, random_state=0)
    before = m.predict(known).copy()
    pre = [{k: np.array(v) for k, v in r.items()} for r in m.results]
    added = m.fold_in(first, iterations=20, seed=4)
    assert added["users"] == sorted(added["users"]) and added["users"] and added["items"]
    assert np.array_equal(m.predict(known), before)
    for r, p in zip(m.results, pre):
        assert np.array_equal(r["theta"][:len(p["theta"])], p["theta"])
        assert np.array_equal(r["eta"][:len(p["eta"])], p["eta"])
        assert np.array_equal(r["pr"], p["pr"])

    # oracle: the same plan and initial rows, the reference fold-in of every run
    from mmsbm_b200.data_handler import DataHandler
    dh = DataHandler()
    dh.obs_dict, dh.items_dict, dh.ratings_dict = (
        {k: v for k, v in d.items() if v < n} for d, n in
        zip(m.data_handler.return_dicts(), (len(pre[0]["theta"]), len(pre[0]["eta"]), 10 ** 9)))
    plan = dh.plan_fold_in(first)
    assert plan["users"] == added["users"] and plan["items"] == added["items"]
    nu, ni = len(plan["users"]), len(plan["items"])
    du = np.maximum(np.bincount(plan["user_rows"][:, 0], minlength=nu), 1)[:, None]
    di = np.maximum(np.bincount(plan["item_rows"][:, 1], minlength=ni), 1)[:, None]
    test = m.data_handler.format_test_data(later)
    new = (test[:, 0] >= len(pre[0]["theta"])) | (test[:, 1] >= len(pre[0]["eta"]))
    assert new.all() and len(test) > 50
    rats = []
    for s, child in enumerate(np.random.SeedSequence(4).spawn(len(pre))):
        rng = np.random.default_rng(child)
        tu, ti = rng.random((nu, m.user_groups)) / du, rng.random((ni, m.item_groups)) / di
        th = fref.fold_in(plan["user_rows"], tu, pre[s]["eta"], pre[s]["pr"], 20, 0)
        et = fref.fold_in(plan["item_rows"], pre[s]["theta"], ti, pre[s]["pr"], 20, 1)
        assert rel_err(m.results[s]["theta"][-nu:], th) < 1e-10
        assert rel_err(m.results[s]["eta"][-ni:], et) < 1e-10
        rats.append(orc.rating_distribution(test, np.concatenate([pre[s]["theta"], th]),
                                            np.concatenate([pre[s]["eta"], et]), pre[s]["pr"]))
    got = m.predict(later)
    assert np.array_equal(np.argmax(got, axis=1), np.argmax(np.mean(rats, axis=0), axis=1))


def test_restored_models(tmp_path):
    from mmsbm_b200 import MMSBM
    m, train, first, later = fitted()
    m.save(str(tmp_path / "fitted.npz"))
    loaded = MMSBM.load(str(tmp_path / "fitted.npz"))
    a = m.fold_in(first, iterations=15)
    b = loaded.fold_in(first, iterations=15)
    assert a == b
    for x, y in zip(m.results, loaded.results):
        assert np.array_equal(x["theta"], y["theta"]) and np.array_equal(x["eta"], y["eta"])
    m.save(str(tmp_path / "folded.npz"))
    again = MMSBM.load(str(tmp_path / "folded.npz"))
    assert again.data_handler.return_dicts() == m.data_handler.return_dicts()
    for x, y in zip(m.results, again.results):
        assert np.array_equal(x["theta"], y["theta"]) and np.array_equal(x["eta"], y["eta"])
    assert np.array_equal(again.predict(later), m.predict(later))


def test_cold_start_quality():
    """Users held out of training entirely: folding in half of their ratings must predict the other
    half better than uniform theta rows.  The numpy reference of this exact pipeline (same encoding,
    seeds and iterations) gives accuracy 0.525 with fold-in against 0.4475 with uniform rows on
    these 1200 held-out ratings; the threshold keeps a margin of 0.05."""
    from mmsbm_b200 import MMSBM
    U, I, K, L, R, per = 300, 120, 4, 4, 5, 40
    rows = fref.planted(7, U, I, K, L, R, per)
    held = rows[:, 0] >= 240
    frame = pd.DataFrame({"users": rows[:, 0], "items": rows[:, 1], "ratings": rows[:, 2] + 1})
    hrows = frame[held]
    first = hrows.groupby("users").head(per // 2)
    rest = hrows.drop(first.index)
    m = MMSBM(K, L, iterations=100, sampling=1, seed=5)
    m.fit(frame[~held])
    n_known = len(m.results[0]["theta"])
    added = m.fold_in(first)
    assert len(added["users"]) == 60 and added["items"] == []
    m.predict(rest)
    acc = m.score(silent=True)["stats"]["accuracy"]
    test = m.test
    res = m.results[0]
    uniform = np.concatenate([res["theta"][:n_known], np.full((60, K), 1.0 / K)])
    acc_u = orc.prediction_stats(orc.rating_distribution(test, uniform, res["eta"], res["pr"]),
                                 test[:, 2], list(range(R)))["accuracy"]
    assert len(test) == 1200
    assert acc >= acc_u + 0.05, (acc, acc_u)
