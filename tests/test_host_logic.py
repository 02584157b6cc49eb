"""CPU tests of the host-side logic: encoding, fold construction, sharding helpers,
the C-ABI library's exported symbols.  No GPU needed, no compute call made."""
import ctypes
import json
import logging
import os
import re

import numpy as np
import pandas as pd
import pytest

from mmsbm_b200 import _lib
from mmsbm_b200.data_handler import DataHandler
from mmsbm_b200.helpers import get_n_per_group, structure_folds
from mmsbm_b200.parallel import shard_runs, user_partition
from oracle import mmsbm_oracle as orc
from tests.util import mock_data

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------ C ABI
def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "mmsbm_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(mmsbm_[a-z_0-9]+)\s*\(", header)))
    assert declared, "no declarations found"
    assert os.path.exists(_lib.LIB_PATH), "run `python -m mmsbm_b200.build` first"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert sorted(_lib.EXPORTS) == declared
    assert lib.mmsbm_abi_version() == 4


def test_no_cpu_fallback_without_device():
    """Without a GPU the backend must raise ImportError (the reference's own signal,
    src/backend.py:23-28), never compute on the CPU.  Checked in a child process that sees no
    device (CUDA_VISIBLE_DEVICES empty), so that it runs on a GPU machine too."""
    import subprocess
    import sys
    code = ("import pytest\n"
            "from mmsbm_b200.backend import load_backend\n"
            "for name in ('auto', 'b200', 'numpy'):\n"
            "    with pytest.raises(ImportError):\n"
            "        load_backend(name)\n"
            "print('no fallback')\n")
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and res.stdout.strip() == "no fallback", res.stdout[-2000:] + res.stderr[-2000:]


def test_product_code_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing shipped may import, link or call it."""
    offenders = []
    for top in ("mmsbm_b200", "include"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    for ln in open(os.path.join(dirpath, f)).read().splitlines():
                        if "oracle" in ln and re.match(r"\s*(import|from|#include)\b", ln):
                            offenders.append((f, ln.strip()))
    src = open(os.path.join(ROOT, "kernels_b200.py")).read()
    assert "oracle" not in src and not offenders, offenders


# ---------------------------------------------------------------- encoding
def test_encoding_matches_reference_golden(golden_dir):
    enc = json.load(open(os.path.join(golden_dir, "encoding.json")))
    df = pd.DataFrame({"users": [1, 10, 2, 100, 11, 10], "items": ["b", "a", "B", "10", "9", "a"],
                       "ratings": [5.0, 1.0, 3.5, 10.0, 2.0, 1.0]})
    dh = DataHandler()
    out = dh.format_train_data(df)
    assert out.dtype == np.int64 and out.tolist() == enc["train_out"]
    assert [dh.obs_dict, dh.items_dict, dh.ratings_dict] == enc["dicts"]
    tdf = pd.DataFrame({"users": [10, 7, 2, 100, 1], "items": ["a", "a", "zz", "9", "B"],
                        "ratings": [1.0, 5.0, 3.5, 4.0, 10.0]})
    assert dh.format_test_data(tdf).tolist() == enc["test_out"]


def test_encoding_warnings(golden_dir):
    """Every warning of the "MMSBM" logger.  That logger does not propagate (logger.setup_logger), so
    pytest attaches its own capture handlers to it; forcing propagation would count each record
    twice.  The warnings are caught by a sink that is the only handler on the logger for the call."""
    enc = json.load(open(os.path.join(golden_dir, "encoding.json")))
    dh = DataHandler()
    dh.format_train_data(pd.DataFrame({"users": [1, 10, 2, 100, 11, 10],
                                       "items": ["b", "a", "B", "10", "9", "a"],
                                       "ratings": [5.0, 1.0, 3.5, 10.0, 2.0, 1.0]}))

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
        dh.format_test_data(pd.DataFrame({"users": [10, 7, 2, 100, 1], "items": ["a", "a", "zz", "9", "B"],
                                          "ratings": [1.0, 5.0, 3.5, 4.0, 10.0]}))
    finally:
        log.removeHandler(sink)
        for h in saved[0]:
            log.addHandler(h)
        log.propagate, log.level = saved[1], saved[2]
    assert sink.messages == enc["test_warnings"]


def test_encoding_fixture_and_large_int_path(golden_dir):
    g = np.load(os.path.join(golden_dir, "fixture.npz"))
    meta = json.load(open(os.path.join(golden_dir, "fixture.json")))
    dh = DataHandler()
    np.testing.assert_array_equal(dh.format_train_data(mock_data(1)), g["train"])
    assert dh.obs_dict == meta["obs_dict"] and dh.ratings_dict == meta["ratings_dict"]
    np.testing.assert_array_equal(dh.format_test_data(mock_data(2)), g["test"])
    # the per-distinct-value fast path (>64 rows, integer dtype) against the oracle's per-cell str()
    rng = np.random.default_rng(5)
    df = pd.DataFrame({"users": rng.integers(0, 300, 5000), "items": rng.integers(0, 120, 5000).astype(str),
                       "ratings": rng.integers(1, 11, 5000)})
    out = DataHandler().format_train_data(df)
    ref, _ = orc.encode_train(df["users"].tolist(), df["items"].tolist(), df["ratings"].tolist())
    np.testing.assert_array_equal(out, ref)


def test_stringdtype_columns():
    s = pd.StringDtype()
    df = pd.DataFrame({"users": pd.Series(["u1", "u2", "u1", "u3"], dtype=s),
                       "items": pd.Series(["i1", "i2", "i1", "i3"], dtype=s),
                       "ratings": pd.Series(["1", "2", "3", "1"], dtype=s)})
    dh = DataHandler()
    out = dh.format_train_data(df)
    assert out.shape == (4, 3) and np.issubdtype(out.dtype, np.integer)
    assert dh.format_test_data(df).shape == (4, 3)


def test_decoding_round_trip():
    dh = DataHandler()
    dh.format_train_data(mock_data(1))
    th = dh.return_theta_indices(np.zeros((5, 2)))
    assert list(th.index) == [f"user{k}" for k in range(5)]
    assert set(dh.return_pr_indices(np.zeros((2, 2, 5))).keys()) == {"1", "2", "3", "4", "5"}


# ------------------------------------------------------------------- folds
def test_fold_helpers():
    df = mock_data(1)
    assert structure_folds(df, 2) == 5
    with pytest.raises(AssertionError):
        structure_folds(df, 11)
    rng = np.random.default_rng(0)
    small = df.iloc[:3]
    got = get_n_per_group(small, n=5, rng=rng)          # shrinks to the group size
    assert sorted(got) == [0, 1, 2]
    # a failed over-sized request consumes no random numbers in numpy's Generator.choice
    a, b = np.random.default_rng(9), np.random.default_rng(9)
    with pytest.raises(ValueError):
        a.choice(np.arange(3), 5, replace=False)
    assert a.random() == b.random()


# ---------------------------------------------------------------- sharding
def test_shard_runs_and_user_partition():
    for world in (1, 2, 3, 8):
        got = sorted(s for r in range(world) for s in shard_runs(8, r, world))
        assert got == list(range(8))
    deg = np.array([5, 1, 1, 1, 8, 2, 2, 10, 1, 1])
    for world in (1, 2, 4, 8):
        b = user_partition(deg, world)
        assert b[0] == 0 and b[-1] == len(deg) and np.all(np.diff(b) >= 0) and len(b) == world + 1
    b = user_partition(deg, 2)
    left = deg[:b[1]].sum()
    assert abs(left - deg.sum() / 2) <= deg.max()


@pytest.mark.parametrize("case", ["int", "float", "str", "bool", "mixed", "dates", "nan"])
def test_encoding_fast_path_matches_reference_for_every_dtype(golden_dir, case):
    """The factorise-first encoding (data_handler._distinct_strings) against outputs of the real
    reference DataHandler (tests/golden/make_golden_encoding.py) and against the per-cell path."""
    from tests.util import dtype_frames
    g = np.load(os.path.join(golden_dir, "encoding_dtypes.npz"))
    dicts = json.load(open(os.path.join(golden_dir, "encoding_dtypes.json")))[case]
    train, test = dtype_frames()[case]
    dh = DataHandler()
    np.testing.assert_array_equal(dh.format_train_data(train.copy()), g[case + "_train"])
    assert [[list(kv) for kv in d.items()] for d in dh.return_dicts()] == dicts      # same keys, same order
    np.testing.assert_array_equal(dh.format_test_data(test.copy()), g[case + "_test"])
    slow = DataHandler()
    np.testing.assert_array_equal(slow.parse_train_data(slow._to_object_str(train.copy())), g[case + "_train"])
    assert slow.return_dicts() == dh.return_dicts()


@pytest.mark.parametrize("case", ["fixture", "ints", "strs", "shuffled_index", "str_index", "floats"])
def test_fold_construction_matches_reference(golden_dir, case):
    """MMSBM._make_folds (numpy fast path and the pandas path) against the folds the real
    reference's cv_fit builds (tests/golden/make_golden_folds.py): same held-out labels in the
    same order, same train rows, and the generator left in the same state."""
    import hashlib
    from mmsbm_b200.mmsbm import MMSBM
    from tests.util import fold_frames
    want = json.load(open(os.path.join(golden_dir, "folds.json")))[case]
    frame, folds = fold_frames()[case]
    for fast in (True, False):
        m = MMSBM(2, 2, iterations=1, seed=7)
        if not fast:
            m._make_folds_fast = lambda *a: None
        pairs = m._make_folds(frame, folds)
        if fast:
            assert MMSBM._make_folds_fast(MMSBM(2, 2, seed=7), frame, folds, structure_folds(frame, folds)) is not None
        assert [[str(a) for a in te.index] for _, te in pairs] == want["test"]
        assert [hashlib.sha1(",".join(str(a) for a in tr.index).encode()).hexdigest() for tr, _ in pairs] \
            == want["train_sha1"]
        assert float(m.rng.random()) == want["next_random"]


def test_encoding_threaded_hash_passes_match_serial():
    """Columns of >= 100k rows are factorised in threads (data_handler._distinct_strings_all)."""
    from mmsbm_b200 import data_handler as dhm
    rng = np.random.default_rng(11)
    n = 120_000
    df = pd.DataFrame({"users": rng.integers(0, 5000, n), "items": ["i%d" % x for x in rng.integers(0, 900, n)],
                       "ratings": rng.choice([0.5, 1.0, 2.5, 4.0], n)})
    fast = DataHandler()
    out = fast.format_train_data(df)
    cols = [df.iloc[:, c] for c in range(3)]
    for (codes, strings), col in zip(dhm._distinct_strings_all(cols), cols):
        c2, s2 = dhm._distinct_strings(col)
        np.testing.assert_array_equal(codes, c2)
        assert strings == s2
    slow = DataHandler()
    np.testing.assert_array_equal(slow.parse_train_data(slow._to_object_str(df.iloc[:20000].copy())),
                                  DataHandler().format_train_data(df.iloc[:20000]))
    assert out.shape == (n, 3) and out[:, 0].max() == len(fast.obs_dict) - 1


@pytest.mark.parametrize("backend", ["numba", "numpy"])
def test_bench_reference_arm_runs_without_a_gpu(backend):
    """`bench.py --impl reference` is the CPU arm of the bench contract: one JSON line, the same
    metric / unit / config keys as the GPU arm, impl = reference, no device work."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "ml100k",
                          "--cpu-rows", "3000", "--steps", "1", "--warmup", "1", "--cpu-backend", backend],
                         capture_output=True, text=True, timeout=300, cwd=root)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "rating-updates/sec" and line["value"] > 0
    assert line["unit"] == "rating-updates/s" and line["higher_is_better"] is True
    assert line["config"]["workload"] == "ml100k" and line["gpu_launches"] == 0
    # the unmodified reference when baseline/_ref is installed (oracle/install_reference.py), else the port
    have_ref = os.path.exists(os.path.join(root, "baseline", "_ref", "kernels_numpy.py"))
    assert line["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert line["cpu_baseline"]["backend"] == backend
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}


def test_bench_algorithmic_bytes_match_the_survey_table():
    """bench.b_alg is SURVEY.md section 8d's B_alg = 8(K+L) + 16/S + 16(K U + L I)/N; the table there
    lists 180.2 / 163.6 / 324.6 / 530.5 bytes per rating-update for the four shapes."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    want = {"ml100k": 180.2, "ml1m": 163.6, "ml20m": 324.6, "netflix": 530.5}
    for name, want_b in want.items():
        U, I, N, K, L, S = bench.WORKLOADS[name]
        assert abs(bench.b_alg(U, I, N, K, L, S) - want_b) < 0.06, name


def test_committed_roofline_fractions_are_physical_and_reproducible():
    """Every fraction of the roofline block of a committed bench line can be recomputed from files
    under profiles/ -- the ncu metrics CSV named in the line (re-parsed here), the peaks file, the
    line's own times -- and none exceeds 1."""
    import glob
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("ncu_record", os.path.join(root, "profiles", "ncu_record.py"))
    ncu_record = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ncu_record)
    peaks = json.load(open(os.path.join(root, "profiles", "peaks.json")))
    seen = 0
    for path in sorted(glob.glob(os.path.join(root, "profiles", "r2_v1[5-9]_bench_*.json"))):
        line = json.loads(open(path).read().strip().splitlines()[-1])
        roof = line.get("roofline")
        if not roof or line.get("n_gpus") != 1 or line.get("impl") == "reference":
            continue
        g = roof["gather"]
        seg_ms = roof["kernel_ms"]["by_user"] + roof["kernel_ms"]["by_item"]
        assert g["peak_gbs"] == peaks["gather_gbs"]
        assert abs(g["achieved_gbs"] - g["bytes_per_iteration"] / (seg_ms * 1e-3) / 1e9) < 1e-6 * g["achieved_gbs"]
        assert 0.0 < g["frac"] <= 1.0
        if roof["frac"] is None:
            continue                                         # cooperative path: no bandwidth fraction claimed
        src = os.path.join(root, roof["ncu_record"])
        assert os.path.exists(src), f"{path} names {roof['ncu_record']}, which is not committed"
        rec = ncu_record.extract(src)
        want = rec["dram_bytes_per_iteration"] / (line["ms_per_iteration"] * 1e-3) / 1e9
        assert abs(roof["achieved"] - want) < 1e-6 * want
        assert abs(roof["frac"] - want / roof["peak"]) < 1e-9
        assert 0.0 < roof["frac"] <= 1.0
        assert abs(roof["traffic"] - rec["segment_pass_dram_bytes"]) < 1e-6 * roof["traffic"]
        assert roof["traffic"] <= rec["dram_bytes_per_iteration"]
        seen += 1
    assert seen >= 3


def test_unsupported_shapes_are_refused_before_any_gpu_work(tmp_path, monkeypatch):
    """The kernels' shape envelope (INTEGRATION.md, 'Supported shapes') is checked up front with the
    limit spelled out, instead of failing deep inside the fit."""
    monkeypatch.chdir(tmp_path)                               # the logger writes mmsbm.log
    from mmsbm_b200.mmsbm import MMSBM
    MMSBM(20, 20)._check_shape(5)
    MMSBM(256, 3)._check_shape(4)                             # wide rows: ratings x groups <= 1024
    MMSBM(32, 32)._check_shape(31)
    for K, L, R in ((257, 2, 5), (2, 300, 5), (10, 10, 32), (64, 8, 17), (8, 200, 6)):
        with pytest.raises(ValueError, match="mmsbm_b200"):
            MMSBM(K, L)._check_shape(R)
