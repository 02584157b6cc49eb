"""String-rank encoding of (user, item, rating) columns.

Same observable behaviour as the reference's DataHandler (src/data_handler.py:10-144):
every cell is ``str()``-ed, ids are ranked by ``sorted(set(strings))`` (lexicographic:
'10' < '2'), train rows are encoded to an int64 ``[N,3]`` array, test rows whose
user / item / rating was not seen in training are dropped with a warning, and fitted
parameters are decoded back to the original labels.

Fast path (SURVEY.md section 8 f2): a column is first factorised on its RAW values (one hash
pass, ``pd.factorize``), ``str()`` then runs once per DISTINCT value, the distinct strings are
ranked, and the codes are mapped through that small table -- O(N) numpy work plus O(D log D)
python work instead of N python-level ``str`` / dict operations.  It is taken only where it
is provably identical to ``sorted(set(str(x) for x in column.tolist()))``: integer, bool and
float dtypes (floats factorised on their bit patterns, so -0.0 / 0.0 stay distinct like
their strings; distinct raw values with equal strings are merged by the string table) and
object columns that hold only ``str``.  Anything else (mixed objects, nullable / datetime
dtypes, frames that do not have exactly three columns) takes the per-cell path.
"""
import logging

import numpy as np
import pandas as pd

from .helpers import _invert_dict


def _stringify(col):
    """Per-cell ``str(x)`` of a pandas column as an object ndarray
    (src/data_handler.py:27-32, via ``.tolist()`` so numpy scalars print as python ones)."""
    values = col.tolist()
    kind = col.dtype.kind if hasattr(col.dtype, "kind") else "O"
    if kind in "iub" and len(values) > 64:
        arr = col.to_numpy()
        uniq, inv = np.unique(arr, return_inverse=True)
        table = np.array([str(v) for v in uniq.tolist()], dtype=object)
        return table[inv]
    return np.array([str(x) for x in values], dtype=object)


def _distinct_strings(col):
    """``(codes, strings)`` of a pandas column: ``strings[codes[n]] == str(col.tolist()[n])`` for
    every row.  ``strings`` may hold duplicates (two raw values that print alike); callers go
    through a string-keyed table, which merges them."""
    arr = col.to_numpy()
    kind = arr.dtype.kind
    if kind in "iub":
        codes, uniq = pd.factorize(arr)
        return codes, [str(v) for v in uniq.tolist()]
    if kind == "f" and arr.dtype.itemsize in (4, 8):
        bits = np.ascontiguousarray(arr).view(np.int32 if arr.dtype.itemsize == 4 else np.int64)
        codes, ubits = pd.factorize(bits)
        return codes, [str(v) for v in ubits.view(arr.dtype).tolist()]
    if kind == "O" and len(arr) and pd.api.types.infer_dtype(arr, skipna=False) == "string":
        codes, uniq = pd.factorize(arr)
        return codes, [str(v) for v in uniq.tolist()]
    values = np.array([str(x) for x in col.tolist()], dtype=object)      # per-cell path
    if not len(values):
        return np.zeros(0, dtype=np.int64), []
    codes, uniq = pd.factorize(values)
    return codes, uniq.tolist()


def _distinct_strings_all(cols):
    """``_distinct_strings`` of several columns; the hash passes run in threads for long columns
    (pandas' factorize releases the GIL)."""
    if len(cols) > 1 and len(cols[0]) >= 100_000:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(len(cols)) as ex:
            return list(ex.map(_distinct_strings, cols))
    return [_distinct_strings(c) for c in cols]


def _rank_table(strings):
    """{string: rank in sorted(set(strings))} (src/data_handler.py:39-44)."""
    return {s: k for k, s in enumerate(sorted(set(strings.tolist())))}


def _listed(values):
    return ", ".join(sorted(set(str(a) for a in values)))


def _encode(strings, table):
    uniq, inv = np.unique(strings.astype(str), return_inverse=True) if len(strings) > 64 \
        else (None, None)
    if uniq is None:
        return np.array([table[s] for s in strings.tolist()], dtype=np.int64)
    codes = np.array([table[s] for s in uniq.tolist()], dtype=np.int64)
    return codes[inv]


class DataHandler:
    obs_dict = None
    items_dict = None
    ratings_dict = None

    def __init__(self):
        pass

    @staticmethod
    def _get_data(path_):
        return pd.read_csv(path_, sep=None, usecols=[0, 1, 2], engine="python")

    @staticmethod
    def _check_data(df):
        assert df.isnull().sum().sum() == 0, "Data contains missing values. Aborting."

    @staticmethod
    def _to_object_str(data):
        out = data.copy()
        for col in out.columns:
            out[col] = pd.Series(_stringify(out[col]), index=out.index, dtype=object)
        return out

    @staticmethod
    def _create_values_dict(x):
        return _rank_table(np.asarray([str(a) for a in x], dtype=object))

    @staticmethod
    def _rename_values(x, dict_):
        return [dict_[str(a)] for a in x]

    def parse_train_data(self, df):
        cols = [df.iloc[:, c].to_numpy(dtype=object) for c in range(3)]
        self.obs_dict, self.items_dict, self.ratings_dict = (_rank_table(c) for c in cols)
        out = np.empty((len(df), 3), dtype=np.int64)
        for c, table in enumerate((self.obs_dict, self.items_dict, self.ratings_dict)):
            out[:, c] = _encode(cols[c], table)
        return out

    def parse_test_data(self, df):
        out = np.empty((len(df), 3), dtype=np.int64)
        for c, table in enumerate((self.obs_dict, self.items_dict, self.ratings_dict)):
            out[:, c] = _encode(df.iloc[:, c].to_numpy(dtype=object), table)
        return out

    @staticmethod
    def return_original_indices(x, dict_):
        inv = _invert_dict(dict_)
        return [inv[a] for a in x]

    def return_theta_indices(self, theta):
        theta = pd.DataFrame(theta)
        theta.index = self.return_original_indices(theta.index, self.obs_dict)
        return theta

    def return_eta_indices(self, eta):
        eta = pd.DataFrame(eta)
        eta.index = self.return_original_indices(eta.index, self.items_dict)
        return eta

    def return_pr_indices(self, pr):
        inv = _invert_dict(self.ratings_dict)
        return {inv[a]: pd.DataFrame(pr[:, :, a]) for a in range(pr.shape[2])}

    def format_train_data(self, data):
        if data.shape[1] != 3:                   # the reference's behaviour for odd frames, cell by cell
            data = self._to_object_str(data)
            self._check_data(data)
            return self.parse_train_data(data)
        # (_check_data runs on the stringified frame in the reference, src/data_handler.py:103-105,
        #  where no cell is null any more: it cannot fire, so there is nothing to check here)
        out = np.empty((len(data), 3), dtype=np.int64)
        tables = []
        for c, (codes, strings) in enumerate(_distinct_strings_all([data.iloc[:, c] for c in range(3)])):
            table = {s: k for k, s in enumerate(sorted(set(strings)))}
            lut = np.array([table[s] for s in strings], dtype=np.int64)
            out[:, c] = lut[codes] if len(codes) else 0
            tables.append(table)
        self.obs_dict, self.items_dict, self.ratings_dict = tables
        return out

    def _check_test_in_train(self, data):
        """Column by column (users, items, ratings -- looked up BY NAME like the
        reference, src/data_handler.py:112-127): warn about the unseen values among the
        rows still present and drop those rows."""
        logger = logging.getLogger("MMSBM")
        for column, table in (("users", self.obs_dict), ("items", self.items_dict),
                              ("ratings", self.ratings_dict)):
            present = set(str(a) for a in data.loc[:, column])
            unseen = present.difference(table.keys())
            if len(unseen):
                logger.warning(
                    f"The {column} {', '.join(str(a) for a in unseen)} are in the test set but weren't in "
                    f"the train set so I'll remove them.")
                data = data[~data.loc[:, column].isin(unseen)]
        return data

    def format_test_data(self, data):
        if list(data.columns) != ["users", "items", "ratings"]:
            # the reference looks the columns up by name (KeyError otherwise) and encodes by position
            data = self._to_object_str(data)
            self._check_data(data)
            data = self._check_test_in_train(data)
            return self.parse_test_data(data)
        logger = logging.getLogger("MMSBM")
        alive = np.ones(len(data), dtype=bool)
        enc = np.empty((len(data), 3), dtype=np.int64)
        parts = _distinct_strings_all([data[c] for c in ("users", "items", "ratings")])
        for c, (column, table) in enumerate((("users", self.obs_dict), ("items", self.items_dict),
                                             ("ratings", self.ratings_dict))):
            codes, strings = parts[c]
            lut = np.array([table.get(s, -1) for s in strings], dtype=np.int64)
            present = np.zeros(len(strings), dtype=bool)
            present[codes[alive]] = True                      # distinct values among the rows still there
            unseen = set(s for s, p, k in zip(strings, present, lut) if p and k < 0)
            if len(unseen):
                logger.warning(
                    f"The {column} {', '.join(str(a) for a in unseen)} are in the test set but weren't in "
                    f"the train set so I'll remove them.")
                bad = np.array([s in unseen for s in strings], dtype=bool)
                alive &= ~bad[codes]
            enc[:, c] = lut[codes] if len(codes) else 0
        return enc[alive]

    def _encode_known(self, data, what):
        """Rows of ``data`` (read by position, cells ``str()``-ed) encoded against the fitted
        dictionaries, shared by ``plan_fold_in`` and ``plan_refit``.  Returns (codes, labels, alive):
        the int code per column (-1 where the value is unknown), the ``str`` label per column, and
        the rows whose rating value is known (the others are dropped with a warning)."""
        if data.shape[1] < 3:
            raise ValueError(f"{what} data needs three columns: users, items, ratings")
        parts = _distinct_strings_all([data.iloc[:, c] for c in range(3)])
        codes = []
        for (col, strings), table in zip(parts, (self.obs_dict, self.items_dict, self.ratings_dict)):
            lut = np.array([table.get(s, -1) for s in strings], dtype=np.int64)
            codes.append(lut[col] if len(col) else np.zeros(0, dtype=np.int64))
        labels = [np.array(strings, dtype=object)[col] if len(col) else np.zeros(0, dtype=object)
                  for col, strings in parts]
        alive = codes[2] >= 0
        if not alive.all():
            logging.getLogger("MMSBM").warning(
                f"The ratings {_listed(labels[2][~alive])} are in the {what} set but weren't in the "
                f"train set so I'll remove them.")
        return codes, labels, alive

    @staticmethod
    def _rank_new(labels):
        """(new labels ranked by ``sorted(set(str))``, the rank of every row's label)."""
        new = sorted(set(labels.tolist()))
        rank = {s: k for k, s in enumerate(new)}
        return new, np.array([rank[s] for s in labels.tolist()], dtype=np.int64)

    def plan_fold_in(self, data):
        """Host side of ``MMSBM.fold_in``: encode the rows of ``data`` (read by position, cells
        ``str()``-ed) against the fitted dictionaries and split them into the two fold-in sets.
        Nothing is changed; ``add_fold_in_ids`` records the new ids once they have parameters.

        Rows with a rating value unseen in training, and rows whose user and item are both new, are
        dropped; rows whose user and item are both known are ignored; each with a warning.  New
        users (items) get the codes after the existing ones, ranked among themselves by
        ``sorted(set(str))``.  Returns {"users", "items": new labels in code order,
        "user_rows": int [n,3] (new user - first new code, item, rating),
        "item_rows": int [m,3] (user, new item - first new code, rating)}."""
        logger = logging.getLogger("MMSBM")
        codes, labels, alive = self._encode_known(data, "fold-in")
        cu, ci, cr = codes
        both_new = alive & (cu < 0) & (ci < 0)
        if both_new.any():
            logger.warning(f"The users {_listed(labels[0][both_new])} are in the fold-in set with items "
                           f"{_listed(labels[1][both_new])} and neither was in the train set so I'll remove "
                           f"those {int(both_new.sum())} rows.")
            alive &= ~both_new
        both_known = alive & (cu >= 0) & (ci >= 0)
        if both_known.any():
            logger.warning(f"The users {_listed(labels[0][both_known])} and items {_listed(labels[1][both_known])} "
                           f"of {int(both_known.sum())} fold-in rows were in the train set so I'll ignore "
                           f"those rows: fit again to use them.")
            alive &= ~both_known
        out = {}
        for name, c, table, own, rows_name in (("users", 0, self.obs_dict, cu, "user_rows"),
                                              ("items", 1, self.items_dict, ci, "item_rows")):
            sel = alive & (own < 0)
            new, rank = self._rank_new(labels[c][sel])
            rows = np.stack([cu[sel], ci[sel], cr[sel]], axis=1).astype(np.int64).reshape(-1, 3)
            rows[:, c] = rank
            out[name], out[rows_name] = new, rows
        return out

    def plan_refit(self, data):
        """Host side of ``MMSBM.refit``: encode the rows of ``data`` (read by position, cells
        ``str()``-ed) against the fitted dictionaries.  Nothing is changed; ``add_fold_in_ids``
        records the new ids.

        Known ids keep their codes; new users (items) get the codes after the existing ones, ranked
        among themselves by ``sorted(set(str))``, as in ``plan_fold_in``.  Rows whose user and item
        are both new are kept.  Rows with a rating value unseen in training are dropped with a
        warning; if none is left this raises ``ValueError``.  Returns {"users", "items": new labels
        in code order, "rows": int [N,3] (user, item, rating) in the order of ``data``}."""
        codes, labels, alive = self._encode_known(data, "refit")
        if not alive.any():
            raise ValueError("refit data holds no row with a rating value the model knows")
        out = {}
        for name, c, table in (("users", 0, self.obs_dict), ("items", 1, self.items_dict)):
            sel = alive & (codes[c] < 0)
            out[name], rank = self._rank_new(labels[c][sel])
            codes[c][sel] = len(table) + rank
        out["rows"] = np.stack([c[alive] for c in codes], axis=1).astype(np.int64)
        return out

    def add_fold_in_ids(self, users, items):
        """Give the new labels of ``plan_fold_in`` / ``plan_refit`` their codes after the existing
        ones."""
        for table, new in ((self.obs_dict, users), (self.items_dict, items)):
            base = len(table)
            for k, s in enumerate(new):
                table[s] = base + k

    def return_dicts(self):
        return self.obs_dict, self.items_dict, self.ratings_dict
