"""INTEGRATION.md level 1, for real: the UNMODIFIED reference (baseline/_ref, installed by
oracle/install_reference.py) runs ITS OWN ``MMSBM`` with ``backend="b200"``: its loader
(src/backend.py:16-22) imports this repo's ``kernels_b200`` plugin, its spawn pool
(src/mmsbm.py:182-185) pickles the model into worker processes, and its loop
(src/mmsbm.py:243-250) calls the plugin's ``update_coefficients`` every iteration.  The
reference's own known answers must come out (tests/test_mmsbm.py:53-81 of the reference).

Runs in a subprocess because the reference's flat module names (``mmsbm``, ``helpers``,
``logger`` ...) must not leak into this test session.

Without baseline/_ref (a plain checkout) the same driving is restated in RESTATED: the
reference's plugin import by module name, its spawn pool with one run per worker, its per-run
loop (seeded init, update_coefficients + the three host normalisations, the likelihood from
compute_omegas), its best-run choice and the statistics of the mean prediction matrix.  Both
drivers are held to the same known answers."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")

SCRIPT = r'''
import json, os, sys
root, ref = sys.argv[1], sys.argv[2]
sys.path.insert(0, ref)            # the reference's flat modules: mmsbm, backend, ...
sys.path.insert(1, root)           # kernels_b200.py (the plugin) and the mmsbm_b200 package
import numpy as np, pandas as pd
os.chdir(sys.argv[3])

def mock_data(seed, n=100):        # the reference's fixture, tests/test_mmsbm.py:12-22
    rng = np.random.default_rng(seed)
    return pd.DataFrame({
        "users": [f"user{rng.choice(list(range(5)))}" for _ in range(n)],
        "items": [f"item{rng.choice(list(range(10)))}" for _ in range(n)],
        "ratings": [rng.choice(list(range(1, 6))) for _ in range(n)]})

if __name__ == "__main__":
    import mmsbm as ref_mmsbm
    assert os.path.dirname(os.path.abspath(ref_mmsbm.__file__)) == os.path.abspath(ref)
    from mmsbm_b200 import _lib
    out = {}
    for sampling in (1, 3):
        m = ref_mmsbm.MMSBM(2, 2, iterations=10, sampling=sampling, seed=1, backend="b200")
        m.fit(mock_data(1), silent=True)              # through the reference's spawn pool
        assert m.em._backend == "b200"
        m.predict(mock_data(2))
        s = m.score(silent=True)["stats"]
        out[str(sampling)] = {k: float(v) for k, v in s.items()}
        out[str(sampling)]["theta0"] = float(m.theta.sum(axis=0).iloc[0])
        out[str(sampling)]["psum"] = float(m.prediction_matrix.sum())
    # the reference's own loop in THIS process: the plugin's index cache must hit after call one
    m = ref_mmsbm.MMSBM(2, 2, iterations=10, seed=1, backend="b200")
    m.data_handler = __import__("data_handler").DataHandler()
    train = m.data_handler.format_train_data(mock_data(1))
    m._prepare_objects(train)
    import ctypes
    lib = _lib.load()
    h0, m0 = ctypes.c_int64(), ctypes.c_int64()
    lib.mmsbm_index_cache_stats(ctypes.byref(h0), ctypes.byref(m0))
    res = m.run_one_sampling(train, m.child_states[0], 0)
    h1, m1 = ctypes.c_int64(), ctypes.c_int64()
    lib.mmsbm_index_cache_stats(ctypes.byref(h1), ctypes.byref(m1))
    out["cache"] = {"hits": h1.value - h0.value, "misses": m1.value - m0.value}
    out["inproc_likelihood"] = float(res["likelihood"])
    print("RESULT " + json.dumps(out))
'''

RESTATED = r'''
import ctypes, importlib, json, multiprocessing as mp, os, sys
root = sys.argv[1]
sys.path.insert(0, root)           # kernels_b200.py (the plugin), mmsbm_b200, oracle, tests
import numpy as np
from oracle import mmsbm_oracle as orc
from tests.util import mock_data   # the reference's fixture, tests/test_mmsbm.py:12-22

K = L = 2
ITERATIONS = 10
EPS = np.finfo(np.float64).eps


def likelihood(plugin, data, theta, eta, pr):
    """src/expectation_maximization.py:157-167, omegas from the backend."""
    w = plugin.compute_omegas(data, theta, eta, pr)
    ws, ts = np.maximum(w, EPS), np.maximum(w.sum(axis=(1, 2)), EPS)
    return float(np.sum(ws * np.log(ws) - ws * np.log(ts[:, None, None])))


def run_one_sampling(args):
    """src/mmsbm.py:187-269: seeded init, the EM loop through the backend, the likelihood."""
    train, child = args
    plugin = importlib.import_module("kernels_b200")   # what load_backend("b200") imports
    R = len(np.unique(train[:, 2]))
    fu, fi = orc.degree_factors(train, K, L)
    rng = np.random.default_rng(child)
    theta = rng.random((fu.shape[0], K)) / fu
    eta = rng.random((fi.shape[0], L)) / fi
    pr = orc.normalize_pr(rng.random((K, L, R)))
    for _ in range(ITERATIONS):
        n_theta, n_eta, n_pr = plugin.update_coefficients(train, theta, eta, pr)
        theta, eta, pr = n_theta / fu, n_eta / fi, orc.normalize_pr(n_pr)
    return {"likelihood": likelihood(plugin, train, theta, eta, pr), "theta": theta, "eta": eta, "pr": pr}


if __name__ == "__main__":
    os.chdir(sys.argv[2])
    from mmsbm_b200 import DataHandler, _lib
    plugin = importlib.import_module("kernels_b200")
    out = {}
    for sampling in (1, 3):
        dh = DataHandler()
        train = dh.format_train_data(mock_data(1))
        children = np.random.default_rng(1).bit_generator._seed_seq.spawn(sampling)
        with mp.get_context("spawn").Pool(processes=sampling) as pool:   # src/mmsbm.py:182-185
            results = pool.map(run_one_sampling, [(train, c) for c in children])
        test = dh.format_test_data(mock_data(2))
        levels = list(np.unique(train[:, 2]))
        rats = [plugin.prod_dist(test, r["theta"], r["eta"], r["pr"]) for r in results]
        best = orc.choose_best(rats, test[:, 2], levels)
        matrix = np.mean(rats, axis=0)
        stats = orc.prediction_stats(matrix, test[:, 2], levels)
        stats["likelihood"] = results[best]["likelihood"]
        out[str(sampling)] = {k: float(v) for k, v in stats.items()}
        out[str(sampling)]["theta0"] = float(results[best]["theta"].sum(axis=0)[0])
        out[str(sampling)]["psum"] = float(matrix.sum())
    # the loop in THIS process: the plugin's index cache must hit after call one
    train = DataHandler().format_train_data(mock_data(1))
    lib = _lib.load()
    h0, m0 = ctypes.c_int64(), ctypes.c_int64()
    lib.mmsbm_index_cache_stats(ctypes.byref(h0), ctypes.byref(m0))
    res = run_one_sampling((train, np.random.default_rng(1).bit_generator._seed_seq.spawn(1)[0]))
    h1, m1 = ctypes.c_int64(), ctypes.c_int64()
    lib.mmsbm_index_cache_stats(ctypes.byref(h1), ctypes.byref(m1))
    out["cache"] = {"hits": h1.value - h0.value, "misses": m1.value - m0.value}
    out["inproc_likelihood"] = res["likelihood"]
    print("RESULT " + json.dumps(out))
'''


def test_reference_mmsbm_runs_on_the_b200_plugin(tmp_path):
    script = tmp_path / "drive_reference.py"
    if os.path.exists(os.path.join(REF, "mmsbm.py")):
        script.write_text(SCRIPT)
        args = [ROOT, REF, str(tmp_path)]
    else:
        script.write_text(RESTATED)
        args = [ROOT, str(tmp_path)]
    res = subprocess.run([sys.executable, str(script)] + args, capture_output=True, text=True,
                         timeout=900, cwd=str(tmp_path))
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    line = [ln for ln in res.stdout.splitlines() if ln.startswith("RESULT ")][-1]
    out = json.loads(line[len("RESULT "):])
    one = out["1"]
    # the reference's known answers for its fixture (SURVEY.md section 4, measured with its numpy backend)
    assert one["accuracy"] == pytest.approx(0.13, abs=1e-12)
    assert one["one_off_accuracy"] == pytest.approx(0.55, abs=1e-12)
    assert one["mae"] == pytest.approx(0.78, abs=1e-12)
    assert one["s2"] == 153
    assert one["s2pond"] == pytest.approx(129.4766730930339, rel=1e-9)
    assert one["likelihood"] == pytest.approx(-13.773187406968459, rel=1e-8)
    assert one["theta0"] == pytest.approx(2.1112326760042786, rel=1e-9)
    assert one["psum"] == pytest.approx(100.0, rel=1e-9)
    # sampling=3 through the pool: three worker processes; the reference picks run 1 (likelihood
    # -17.739...) and scores the mean prediction matrix (tests/golden/sampling3.npz, made by the
    # reference's numpy backend)
    three = out["3"]
    assert three["accuracy"] == pytest.approx(0.10, abs=1e-12) and three["s2"] == 164
    assert three["likelihood"] == pytest.approx(-17.73915051, rel=1e-8)
    assert three["s2pond"] == pytest.approx(126.599259, rel=1e-7)
    # 10 update_coefficients calls on one array: one index build, then nine hits (the reference's
    # compute_likelihood goes through compute_omegas, which needs no index)
    assert out["cache"]["misses"] == 1 and out["cache"]["hits"] == 9
    assert out["inproc_likelihood"] == pytest.approx(-13.773187406968459, rel=1e-8)
