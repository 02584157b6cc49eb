"""CPU tests of fold-in: the reference restricted to new rows against the oracle's EM step, and the
host planning of MMSBM.fold_in (encoding, dropped / ignored rows, warnings).  No GPU needed."""
import contextlib
import logging

import numpy as np
import pandas as pd
import pytest

from mmsbm_b200.data_handler import DataHandler
from oracle import mmsbm_oracle as orc
from tests import fold_in_reference as fref
from tests.util import dtype_frames, random_triples


# ------------------------------------------------------------------ reference vs the EM step
@pytest.mark.parametrize("side", [0, 1])
def test_reference_fold_in_is_the_em_step_restricted(side):
    """One fold-in iteration of a subset of training ids, started from their current rows and given
    all their training rows, is bit for bit their rows of orc.em_iteration: np.add.at adds in row
    order and omega is per row, so both compute the same floating-point operations."""
    U, I, R, K, L = 60, 40, 5, 6, 4
    data = random_triples(3, 3000, U, I, R)
    fu, fi = orc.degree_factors(data, K, L)
    theta, eta, pr = orc.seeded_init(np.random.SeedSequence(11), U, I, K, L, R, fu, fi)
    th1, et1, _ = orc.em_iteration(data, theta, eta, pr, fu, fi)
    ids = np.array([0, 5, 17, 33, 34, 39])
    sel = np.isin(data[:, side], ids)
    rows = data[sel].copy()
    rows[:, side] = np.searchsorted(ids, rows[:, side])
    if side == 0:
        got = fref.fold_in(rows, theta[ids], eta, pr, 1, side=0)
        want = th1[ids]
    else:
        got = fref.fold_in(rows, theta, eta[ids], pr, 1, side=1)
        want = et1[ids]
    assert np.array_equal(got, want)


# ------------------------------------------------------------------ host planning
@contextlib.contextmanager
def captured_warnings():
    """The "MMSBM" logger does not propagate; its handlers are swapped for a sink for the call."""
    class Sink(logging.Handler):
        def __init__(self):
            super().__init__(logging.WARNING)
            self.messages = []

        def emit(self, record):
            self.messages.append(record.getMessage())

    log = logging.getLogger("MMSBM")
    saved = log.handlers[:], log.propagate, log.level
    sink = Sink()
    for h in saved[0]:
        log.removeHandler(h)
    log.addHandler(sink)
    log.propagate = False
    log.setLevel(logging.WARNING)
    try:
        yield sink.messages
    finally:
        log.removeHandler(sink)
        for h in saved[0]:
            log.addHandler(h)
        log.propagate, log.level = saved[1], saved[2]


def _strs(frame, c):
    return [str(x) for x in frame.iloc[:, c].tolist()]


def _expected(dh, fold):
    """What plan_fold_in must return, by a plain per-row walk over the str()-ed cells."""
    obs, items, rats = dh.obs_dict, dh.items_dict, dh.ratings_dict
    kept, counts = [], {"rating": 0, "both_new": 0, "both_known": 0}
    for u, i, r in zip(_strs(fold, 0), _strs(fold, 1), _strs(fold, 2)):
        if r not in rats:
            counts["rating"] += 1
        elif u not in obs and i not in items:
            counts["both_new"] += 1
        elif u in obs and i in items:
            counts["both_known"] += 1
        else:
            kept.append((u, i, r))
    new_u = sorted({u for u, i, r in kept if u not in obs})
    new_i = sorted({i for u, i, r in kept if i not in items})
    user_rows = [(new_u.index(u), items[i], rats[r]) for u, i, r in kept if u not in obs]
    item_rows = [(obs[u], new_i.index(i), rats[r]) for u, i, r in kept if i not in items]
    return new_u, new_i, np.array(user_rows, dtype=np.int64).reshape(-1, 3), \
        np.array(item_rows, dtype=np.int64).reshape(-1, 3), counts


def _split(d):
    """(train, fold-in frame): some users, items and one rating value are held out of training;
    the fold-in frame holds every held-out row plus a few rows of known users and items."""
    su, si, sr = _strs(d, 0), _strs(d, 1), _strs(d, 2)
    hu = set(sorted(set(su))[1::3][:4])
    hi = set(sorted(set(si))[2::5][:5])
    hr = {sorted(set(sr))[-1]} if len(set(sr)) > 2 else set()
    held = np.array([u in hu or i in hi or r in hr for u, i, r in zip(su, si, sr)])
    return d[~held], pd.concat([d[held], d[~held].iloc[:4]])


@pytest.mark.parametrize("case", list(dtype_frames()))
def test_plan_fold_in(case):
    d, _ = dtype_frames()[case]
    train, fold = _split(d)
    dh = DataHandler()
    dh.format_train_data(train)
    before = [dict(t) for t in dh.return_dicts()]
    new_u, new_i, user_rows, item_rows, counts = _expected(dh, fold)
    with captured_warnings() as msgs:
        plan = dh.plan_fold_in(fold)
    assert [dict(t) for t in dh.return_dicts()] == before          # planning changes nothing
    assert plan["users"] == new_u and plan["items"] == new_i
    assert np.array_equal(plan["user_rows"], user_rows)
    assert np.array_equal(plan["item_rows"], item_rows)
    assert sum("ratings" in m and "remove" in m for m in msgs) == (counts["rating"] > 0)
    assert sum("neither was in the train set" in m for m in msgs) == (counts["both_new"] > 0)
    assert sum("fit again to use them" in m for m in msgs) == (counts["both_known"] > 0)
    assert len(msgs) == sum(v > 0 for v in counts.values())
    if counts["both_new"]:
        assert f"those {counts['both_new']} rows" in next(m for m in msgs if "neither" in m)
    assert counts["both_known"] >= 4 and (new_u or new_i)

    # the new ids get the codes after the existing ones, in sorted(set(str)) order
    dh.add_fold_in_ids(plan["users"], plan["items"])
    obs, items = dh.obs_dict, dh.items_dict
    assert all(obs[k] == v for k, v in before[0].items()) and all(items[k] == v for k, v in before[1].items())
    assert [obs[u] for u in new_u] == list(range(len(before[0]), len(before[0]) + len(new_u)))
    assert [items[i] for i in new_i] == list(range(len(before[1]), len(before[1]) + len(new_i)))
    assert dh.ratings_dict == before[2]

    # a second call sees them as known (rows whose both ids were new may now be usable)
    new_u2, new_i2, user_rows2, item_rows2, _ = _expected(dh, fold)
    with captured_warnings():
        again = dh.plan_fold_in(fold)
    assert not set(again["users"]) & set(new_u) and not set(again["items"]) & set(new_i)
    assert again["users"] == new_u2 and again["items"] == new_i2
    assert np.array_equal(again["user_rows"], user_rows2) and np.array_equal(again["item_rows"], item_rows2)
    if not counts["both_new"]:
        assert again["users"] == [] and again["items"] == []


def test_plan_fold_in_messages_and_empty_frame():
    dh = DataHandler()
    dh.format_train_data(pd.DataFrame({"users": [1, 2, 3], "items": ["a", "b", "a"], "ratings": [1, 2, 1]}))
    fold = pd.DataFrame({"users": [9, 1, 8, 2, 1, 7], "items": ["a", "z", "y", "b", "a", "a"],
                         "ratings": [1, 2, 1, 5, 2, 2]})
    with captured_warnings() as msgs:
        plan = dh.plan_fold_in(fold)
    assert msgs == [
        "The ratings 5 are in the fold-in set but weren't in the train set so I'll remove them.",
        "The users 8 are in the fold-in set with items y and neither was in the train set so I'll remove "
        "those 1 rows.",
        "The users 1 and items a of 1 fold-in rows were in the train set so I'll ignore those rows: "
        "fit again to use them.",
    ]
    assert plan["users"] == ["7", "9"] and plan["items"] == ["z"]
    assert plan["user_rows"].tolist() == [[1, 0, 0], [0, 0, 1]]
    assert plan["item_rows"].tolist() == [[0, 0, 1]]
    with captured_warnings() as msgs:
        empty = dh.plan_fold_in(fold.iloc[:0])
    assert msgs == [] and empty["users"] == [] and empty["items"] == []
