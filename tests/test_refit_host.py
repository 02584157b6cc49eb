"""CPU tests of the host planning of MMSBM.refit (DataHandler.plan_refit): encoding against the
fitted dictionaries, new ids ranked and appended, both-new rows kept, unseen ratings dropped with a
warning, an empty result refused.  No GPU needed."""
import numpy as np
import pandas as pd
import pytest

from mmsbm_b200.data_handler import DataHandler
from tests.test_fold_in_host import _split, _strs, captured_warnings
from tests.util import dtype_frames


def _expected(dh, frame):
    """What plan_refit must return, by a plain per-row walk over the str()-ed cells."""
    obs, items, rats = dh.obs_dict, dh.items_dict, dh.ratings_dict
    kept = [(u, i, r) for u, i, r in zip(_strs(frame, 0), _strs(frame, 1), _strs(frame, 2)) if r in rats]
    new_u = sorted({u for u, _, _ in kept if u not in obs})
    new_i = sorted({i for _, i, _ in kept if i not in items})
    code_u = dict(obs, **{u: len(obs) + k for k, u in enumerate(new_u)})
    code_i = dict(items, **{i: len(items) + k for k, i in enumerate(new_i)})
    rows = np.array([(code_u[u], code_i[i], rats[r]) for u, i, r in kept], dtype=np.int64).reshape(-1, 3)
    dropped = sum(r not in rats for r in _strs(frame, 2))
    both_new = sum(u not in obs and i not in items for u, i, _ in kept)
    return new_u, new_i, rows, dropped, both_new


@pytest.mark.parametrize("case", list(dtype_frames()))
def test_plan_refit(case):
    d, _ = dtype_frames()[case]
    train, extra = _split(d)
    dh = DataHandler()
    dh.format_train_data(train)
    before = [dict(t) for t in dh.return_dicts()]
    frame = pd.concat([train, extra])                        # old rows plus the new ones
    new_u, new_i, rows, dropped, both_new = _expected(dh, frame)
    with captured_warnings() as msgs:
        plan = dh.plan_refit(frame)
    assert [dict(t) for t in dh.return_dicts()] == before      # planning changes nothing
    assert plan["users"] == new_u and plan["items"] == new_i
    assert np.array_equal(plan["rows"], rows)
    assert new_u or new_i
    # the known rows keep their training codes, in frame order
    assert np.array_equal(plan["rows"][:len(train)], dh.parse_test_data(DataHandler._to_object_str(train)))
    assert len(msgs) == (dropped > 0)
    if dropped:
        assert "are in the refit set but weren't in the train set so I'll remove them" in msgs[0]
    # rows whose user and item are both new are kept
    assert ((plan["rows"][:, 0] >= len(before[0])) & (plan["rows"][:, 1] >= len(before[1]))).sum() == both_new


def test_plan_refit_messages_and_empty():
    dh = DataHandler()
    dh.format_train_data(pd.DataFrame({"users": [1, 2, 3], "items": ["a", "b", "a"], "ratings": [1, 2, 1]}))
    frame = pd.DataFrame({"users": [9, 1, 8, 2, 1, 10], "items": ["a", "z", "y", "b", "a", "a"],
                          "ratings": [1, 2, 1, 5, 2, 2]})
    with captured_warnings() as msgs:
        plan = dh.plan_refit(frame)
    assert msgs == ["The ratings 5 are in the refit set but weren't in the train set so I'll remove them."]
    # users: known "1" "2" "3" -> 0 1 2; new "10" "8" "9" (string order) -> 3 4 5; items: new "y" "z" -> 2 3
    assert plan["users"] == ["10", "8", "9"] and plan["items"] == ["y", "z"]
    assert plan["rows"].tolist() == [[5, 0, 0], [0, 3, 1], [4, 2, 0], [0, 0, 1], [3, 0, 1]]
    with pytest.raises(ValueError, match="no row"):
        dh.plan_refit(frame.iloc[:0])
    with captured_warnings() as msgs, pytest.raises(ValueError, match="no row"):
        dh.plan_refit(frame.iloc[3:4])
    assert len(msgs) == 1
    with pytest.raises(ValueError, match="three columns"):
        dh.plan_refit(frame.iloc[:, :2])


@pytest.mark.parametrize("case", ["int", "str", "mixed"])
def test_plan_refit_after_add_fold_in_ids(case):
    """Ids recorded by add_fold_in_ids (fold-in, or an earlier refit) are known: they keep their
    codes, and only ids new to the extended dictionaries are appended."""
    d, _ = dtype_frames()[case]
    train, extra = _split(d)
    dh = DataHandler()
    dh.format_train_data(train)
    with captured_warnings():
        first = dh.plan_refit(extra)
    dh.add_fold_in_ids(first["users"], first["items"])
    extended = [dict(t) for t in dh.return_dicts()]
    with captured_warnings():
        again = dh.plan_refit(pd.concat([train, extra]))
    assert again["users"] == [] and again["items"] == []
    new_u, new_i, rows, _, _ = _expected(dh, pd.concat([train, extra]))
    assert new_u == [] and new_i == [] and np.array_equal(again["rows"], rows)
    assert [dict(t) for t in dh.return_dicts()] == extended

    # a frame with ids new to the extended dictionaries: codes after the extended ones
    more = train.iloc[:5].copy()
    more[more.columns[0]] = pd.Series(["zz-new-%d" % k for k in range(5)], index=more.index, dtype=object)
    with captured_warnings():
        plan = dh.plan_refit(pd.concat([train, more]))
    assert plan["users"] == sorted("zz-new-%d" % k for k in range(5))
    assert plan["rows"][len(train):, 0].tolist() == [len(extended[0]) + k for k in range(5)]
