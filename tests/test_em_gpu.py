"""Parity of the CUDA path with the oracle and the reference's golden vectors.
Everything here calls through the C ABI (host-pointer entry points via the plugin
module, device-pointer entry points via Engine).  Needs a B200.

Tolerances (BASELINE.json north_star): integer / index work bit-exact; theta, eta, pr
<= 1e-10 relative per element after one iteration from identical inputs; likelihood
<= 1e-8 relative; same best run.  The CUDA path reassociates the sums (em_step.cu
header), so agreement is ~1e-14, far inside the budget; the tests assert the budget and
print the observed error.
"""
import json
import os

import numpy as np
import pytest

from oracle import mmsbm_oracle as orc
from tests.util import mock_data, random_params, random_triples, rel_err

pytestmark = pytest.mark.gpu

PARAM_TOL = 1e-10
LIK_TOL = 1e-8


@pytest.fixture(scope="module")
def kb():
    from mmsbm_b200 import kernels_b200
    return kernels_b200


def _gold(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


# ----------------------------------------------------------------- plugin (b1) level
def test_toy_backends_like_the_reference_test(kb, golden_dir):
    """tests/test_backends.py:7-60 of the reference, with 'b200' as the alternative backend."""
    g = _gold(golden_dir, "toy_backends.npz")
    for tag in ("omega", "prod"):
        args = [g[f"{tag}_{k}"] for k in ("data", "theta", "eta", "pr")]
        out = kb.compute_omegas(*args)
        assert np.allclose(out, g[f"{tag}_omegas_numpy"], atol=1e-8)
        np.testing.assert_array_equal(out, g[f"{tag}_omegas_numpy"])     # same product order: bit-exact
        dist = kb.prod_dist(*args)
        assert np.allclose(dist, g[f"{tag}_prod_numpy"], atol=1e-8)
        assert rel_err(dist, g[f"{tag}_prod_numpy"]) < 1e-13
        nt, ne, npr = kb.update_coefficients(*args)
        assert rel_err(nt, g[f"{tag}_ntheta"]) < PARAM_TOL
        assert rel_err(ne, g[f"{tag}_neta"]) < PARAM_TOL
        assert rel_err(npr, g[f"{tag}_npr"]) < PARAM_TOL


@pytest.mark.parametrize("name,tags", [("medium.npz", [""]), ("wide.npz", ["k20_", "l32_", "odd_"])])
def test_update_coefficients_against_reference_golden(kb, golden_dir, name, tags):
    g = _gold(golden_dir, name)
    for t in tags:
        data, theta, eta, pr = (g[t + k] for k in ("data", "theta", "eta", "pr"))
        nt, ne, npr = kb.update_coefficients(data, theta, eta, pr)
        errs = (rel_err(nt, g[t + "ntheta"]), rel_err(ne, g[t + "neta"]), rel_err(npr, g[t + "npr"]))
        print(name, t, "rel err n_theta/n_eta/n_pr", errs)
        assert max(errs) < PARAM_TOL
        lik = kb.likelihood(data, theta, eta, pr)
        assert abs(lik - g[t + "likelihood"]) <= LIK_TOL * abs(g[t + "likelihood"])
        assert abs(lik - g[t + "likelihood"]) <= 1e-12 * abs(g[t + "likelihood"])
        assert rel_err(kb.prod_dist(data[:257], theta, eta, pr), g[t + "prod"]) < 1e-12
        om = kb.compute_omegas(data[:300], theta, eta, pr)
        np.testing.assert_array_equal(om, orc.omegas(data[:300], theta, eta, pr))


def test_empty_rating_level_and_zero_rows(kb):
    """A level with no rows keeps a zero slab (src/kernels_numpy.py:74-77); an all-zero
    theta row gives sum_omega = 0 -> divided by eps, contributing exactly zero."""
    data = np.array([[0, 0, 0], [1, 1, 2], [1, 0, 2], [2, 1, 0]], dtype=np.int64)
    g = np.random.default_rng(3)
    theta, eta, pr = g.random((3, 3)), g.random((2, 2)), g.random((3, 2, 3))
    theta[2] = 0.0
    nt, ne, npr = kb.update_coefficients(data, theta, eta, pr)
    rt, re_, rpr = orc.em_sums(data, theta, eta, pr)
    assert np.all(npr[:, :, 1] == 0) and np.all(nt[2] == 0)
    assert rel_err(nt, rt) < PARAM_TOL and rel_err(ne, re_) < PARAM_TOL and rel_err(npr, rpr) < PARAM_TOL


def test_bad_ids_raise(kb):
    from mmsbm_b200._lib import MmsbmError
    theta, eta, pr = random_params(0, 3, 3, 2, 2, 2)
    with pytest.raises(MmsbmError):
        kb.update_coefficients(np.array([[0, 5, 0]], dtype=np.int64), theta, eta, pr)
    with pytest.raises(MmsbmError):
        kb.update_coefficients(np.array([[0, 0, 2]], dtype=np.int64), theta, eta, pr)


# ------------------------------------------------------------------ index structure (a8)
@pytest.mark.parametrize("shape", [(100, 5, 10, 5), (1, 1, 1, 1), (5000, 300, 7, 3), (70000, 2000, 900, 5),
                                   (300000, 50, 40000, 11)])
@pytest.mark.parametrize("heavy", [False, True])
def test_index_build_bit_exact(shape, heavy):
    from mmsbm_b200.engine import Engine
    N, U, I, R = shape
    data = random_triples(17, N, U, I, R, heavy_tail=heavy)
    e = Engine(data, U, I, R, 2, 2)
    for col, seg, adj, perm, deg, n_ids in ((0, e.useg, e.uadj, e.uperm, e.udeg, U),
                                            (1, e.iseg, e.iadj, e.iperm, e.ideg, I)):
        rseg, rperm = orc.bucket_order(data[:, col], data[:, 2], n_ids, R)
        np.testing.assert_array_equal(seg.cpu().numpy()[:n_ids * R + 1], rseg)
        np.testing.assert_array_equal(perm.cpu().numpy()[:N], rperm)
        np.testing.assert_array_equal(adj.cpu().numpy()[:N], data[rperm, 1 - col].astype(np.int32))
        np.testing.assert_array_equal(deg.cpu().numpy()[:n_ids], np.bincount(data[:, col], minlength=n_ids))


def test_index_lists_match_reference_lists(golden_dir):
    """MMSBM._user_indices/_item_indices/_rating_indices == the reference's np.where lists."""
    from mmsbm_b200 import MMSBM
    g = _gold(golden_dir, "fixture.npz")
    mm = MMSBM(2, 2, iterations=1, seed=1)
    mm._prepare_objects(g["train"])
    for key, got in (("user", mm._user_indices), ("item", mm._item_indices), ("rating", mm._rating_indices)):
        want = np.split(g[f"{key}_index_concat"], np.cumsum(g[f"{key}_index_len"])[:-1])
        assert len(got) == len(want)
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(mm._normalization_factors["user"], g["norm_user"])
    np.testing.assert_array_equal(mm._normalization_factors["item"], g["norm_item"])


# ------------------------------------------------------------- device engine (a2-a5, a7)
def test_fixture_one_and_ten_iterations(golden_dir):
    from mmsbm_b200.engine import Engine
    g = _gold(golden_dir, "fixture.npz")
    e = Engine(g["train"], 5, 10, 5, 2, 2)
    e.set_params(g["theta0"], g["eta0"], g["pr0"])
    e.run(1)
    th, et, pr = e.get_params()
    errs = (rel_err(th[0], g["theta1"]), rel_err(et[0], g["eta1"]), rel_err(pr[0], g["pr1"]))
    print("fixture, 1 iteration:", errs)
    assert max(errs) < PARAM_TOL
    assert abs(e.likelihood()[0] - g["likelihood1"]) <= LIK_TOL * abs(g["likelihood1"])
    e.run(9)
    th, et, pr = e.get_params()
    errs = (rel_err(th[0], g["theta10"]), rel_err(et[0], g["eta10"]), rel_err(pr[0], g["pr10"]))
    print("fixture, 10 iterations:", errs)
    assert max(errs) < 1e-9
    lik = e.likelihood()[0]
    assert abs(lik - g["likelihood10"]) <= LIK_TOL * abs(g["likelihood10"])


@pytest.mark.parametrize("K,L,R,S", [(10, 10, 5, 3), (20, 20, 5, 2), (7, 5, 4, 1), (3, 32, 6, 2), (33, 9, 5, 1),
                                     (1, 1, 2, 1), (64, 48, 5, 1), (130, 70, 3, 1), (12, 28, 10, 2), (20, 20, 5, 5),
                                     (20, 20, 5, 8), (7, 18, 4, 7), (20, 19, 3, 13),
                                     # the BASELINE.json shapes the kernels specialise on: Netflix
                                     # (K=L=32, one run: 8-lane rows on both sides), ML-1M (K=L=10, eight
                                     # runs: pairs of 3-lane rows), ML-100K (K=L=10, one run)
                                     (32, 32, 5, 1), (10, 10, 5, 8), (10, 10, 5, 1),
                                     # rows of 16 and 24 doubles (4- and 6-lane groups, alone and in pairs)
                                     (16, 16, 7, 2), (24, 22, 6, 3)])
@pytest.mark.parametrize("heavy", [False, True])
def test_batched_runs_one_iteration_vs_oracle(K, L, R, S, heavy):
    from mmsbm_b200.engine import Engine
    N, U, I = 60000, 700, 450
    data = random_triples(23, N, U, I, R, heavy_tail=heavy)
    theta, eta, pr = random_params(29, U, I, K, L, R, S=S)
    e = Engine(data, U, I, R, K, L)
    e.set_params(theta, eta, pr)
    e.run(1)
    th, et, prn = e.get_params()
    lik = e.likelihood()
    fu, fi = orc.degree_factors(data, K, L)
    worst = 0.0
    for s in range(S):
        rt, re_, rp = orc.em_iteration(data, theta[s], eta[s], pr[s], fu, fi, chunk=20000)
        worst = max(worst, rel_err(th[s], rt), rel_err(et[s], re_), rel_err(prn[s], rp))
        want = sum(orc.likelihood(data[lo:lo + 20000], rt, re_, rp) for lo in range(0, N, 20000))
        # 1e-8 relative (north_star); the absolute floor covers the degenerate K=L=1 case where
        # the reference's value is exactly 0 and only rounding noise (~1e-16 per element) is left
        assert abs(lik[s] - want) <= LIK_TOL * abs(want) + 1e-15 * N * K * L
        # size-independent invariants of one EM step
        np.testing.assert_allclose(th[s].sum(axis=1), 1.0, rtol=1e-12)
        np.testing.assert_allclose(et[s].sum(axis=1), 1.0, rtol=1e-12)
        np.testing.assert_allclose(prn[s].sum(axis=2), 1.0, rtol=1e-12)
    print(f"K={K} L={L} R={R} S={S} heavy={heavy}: worst rel err {worst:.3e}")
    assert worst < PARAM_TOL


def test_one_giant_segment_and_many_empty_levels():
    """A user holding most of the ratings (one warp walks a 40k-row segment) and rating levels
    that almost never occur (empty (segment, level) groups everywhere)."""
    from mmsbm_b200.engine import Engine
    g = np.random.default_rng(61)
    N, U, I, K, L, R = 50000, 300, 2000, 10, 10, 9
    data = random_triples(67, N, U, I, R)
    data[U:45000, 0] = 7                                    # user 7 owns ~90 % of the rows
    data[R:, 2] = g.choice(R, size=N - R, p=[0.45, 0.45, 0.04, 0.03, 0.01, 0.01, 0.005, 0.004, 0.001])
    theta, eta, pr = random_params(71, U, I, K, L, R, S=2)
    e = Engine(data, U, I, R, K, L)
    e.set_params(theta, eta, pr)
    e.run(1)
    th, et, prn = e.get_params()
    fu, fi = orc.degree_factors(data, K, L)
    for s in range(2):
        rt, re_, rp = orc.em_iteration(data, theta[s], eta[s], pr[s], fu, fi)
        assert max(rel_err(th[s], rt), rel_err(et[s], re_), rel_err(prn[s], rp)) < PARAM_TOL


@pytest.mark.parametrize("N,U,I,R,K,L", [(1, 1, 1, 1, 1, 1), (40, 1, 7, 1, 3, 2), (40, 6, 1, 3, 2, 4),
                                         (500, 30, 20, 1, 5, 5), (64, 64, 64, 2, 2, 2)])
def test_degenerate_shapes(N, U, I, R, K, L):
    """One user, one item, one rating level, one row: every loop bound of the kernels at its edge."""
    from mmsbm_b200.engine import Engine
    data = random_triples(97, max(N, U, I, R), U, I, R)[:max(N, U, I, R)]
    theta, eta, pr = random_params(101, U, I, K, L, R, S=2)
    e = Engine(data, U, I, R, K, L)
    e.set_params(theta, eta, pr)
    e.run(2)
    th, et, prn = e.get_params()
    lik = e.likelihood()
    fu, fi = orc.degree_factors(data, K, L)
    for s in range(2):
        t_, e_, p_ = theta[s], eta[s], pr[s]
        for _ in range(2):
            t_, e_, p_ = orc.em_iteration(data, t_, e_, p_, fu, fi)
        assert max(rel_err(th[s], t_), rel_err(et[s], e_), rel_err(prn[s], p_)) < 1e-9
        want = orc.likelihood(data, t_, e_, p_)
        assert abs(lik[s] - want) <= LIK_TOL * abs(want) + 1e-15 * len(data) * K * L
    rat = e.prod_dist_device(data).cpu().numpy()
    for s in range(2):
        assert rel_err(rat[s], orc.rating_distribution(data, th[s], et[s], prn[s])) < 1e-12


def test_unsupported_shapes_fail_loudly():
    from mmsbm_b200._lib import MmsbmError
    from mmsbm_b200.engine import Engine
    data = random_triples(73, 2000, 30, 20, 40)
    theta, eta, pr = random_params(79, 30, 20, 3, 3, 40, S=1)
    e = Engine(data, 30, 20, 40, 3, 3)
    e.set_params(theta, eta, pr)
    with pytest.raises(MmsbmError):                          # R > 31 rating levels
        e.run(1)
    with pytest.raises(ValueError):
        Engine(np.array([[0, 0, 0], [5, 0, 0]]), 3, 2, 2, 2, 2)   # user id out of range


def test_debug_mode_and_dropped_test_rows(tmp_path, monkeypatch, caplog):
    """debug=True logs the likelihood every 50 iterations (src/mmsbm.py:252-254); test rows with
    ids unseen in training are dropped with the reference's warning."""
    import logging
    import pandas as pd
    monkeypatch.chdir(tmp_path)
    from mmsbm_b200 import MMSBM
    mm = MMSBM(2, 2, iterations=60, sampling=2, seed=4, debug=True)
    mm.fit(mock_data(1), silent=True)
    assert len(mm.results) == 2 and all(np.isfinite(r["likelihood"]) for r in mm.results)
    test = pd.concat([mock_data(2, n=20), pd.DataFrame({"users": ["ghost"], "items": ["item1"], "ratings": [3]})])
    monkeypatch.setattr(logging.getLogger("MMSBM"), "propagate", True)
    with caplog.at_level(logging.WARNING, logger="MMSBM"):
        pred = mm.predict(test)
    assert pred.shape == (20, 5)
    assert any("ghost" in r.getMessage() for r in caplog.records)


def test_raw_sums_flags_and_finalize():
    """RAW flags give the unnormalised numerators; finalize = the post-all-reduce epilogue."""
    from mmsbm_b200 import _lib
    from mmsbm_b200.engine import Engine
    N, U, I, K, L, R = 20000, 300, 200, 6, 9, 5
    data = random_triples(31, N, U, I, R)
    theta, eta, pr = random_params(37, U, I, K, L, R, S=2)
    e = Engine(data, U, I, R, K, L)
    e.set_params(theta, eta, pr)
    th, et, prn = (t.clone() for t in e.step_raw(_lib.RAW_THETA | _lib.RAW_ETA_PR))
    for s in range(2):
        rt, re_, rp = orc.em_sums(data, theta[s], eta[s], pr[s])
        assert rel_err(th[s].cpu().numpy()[:, :K], rt) < PARAM_TOL
        assert rel_err(et[s].cpu().numpy()[:, :L], re_) < PARAM_TOL
        assert rel_err(prn[s].cpu().numpy(), rp) < PARAM_TOL
        assert abs(rp.sum() - N) < 1e-6                       # every rating distributes mass 1
    e.finalize(et, prn)
    fu, fi = orc.degree_factors(data, K, L)
    for s in range(2):
        _, re_, rp = orc.em_iteration(data, theta[s], eta[s], pr[s], fu, fi)
        assert rel_err(et[s].cpu().numpy()[:, :L], re_) < PARAM_TOL
        assert rel_err(prn[s].cpu().numpy(), rp) < PARAM_TOL


def test_reproducible_bits():
    """Fixed summation order: two runs of the same step give identical bits."""
    from mmsbm_b200.engine import Engine
    data = random_triples(41, 50000, 400, 300, 5, heavy_tail=True)
    theta, eta, pr = random_params(43, 400, 300, 10, 10, 5, S=2)
    outs = []
    for _ in range(2):
        e = Engine(data, 400, 300, 5, 10, 10)
        e.set_params(theta, eta, pr)
        e.run(3)
        outs.append(e.get_params() + (e.likelihood(),))
    for a, b in zip(*outs):
        np.testing.assert_array_equal(a, b)


def test_launch_strategies_give_identical_bits(monkeypatch):
    """mmsbm_em_run has three launch strategies -- plain launches, CUDA-graph replay of iteration
    pairs (small problems) and a second stream for the off-critical-path kernels (large ones).
    They run the same kernels on the same data, so the results must be bit-identical."""
    from mmsbm_b200.engine import Engine
    data = random_triples(83, 80000, 900, 500, 5, heavy_tail=True)
    theta, eta, pr = random_params(89, 900, 500, 12, 9, 5, S=3)
    outs = {}
    for name, env in (("plain", {"MMSBM_NO_GRAPH": "1", "MMSBM_NO_OVERLAP": "1", "MMSBM_DYN": "0"}),
                      ("graph", {"MMSBM_NO_OVERLAP": "1"}),
                      ("overlap", {"MMSBM_FORCE_OVERLAP": "1"}),
                      # launch-wide piece queue (persistent CTAs), plain and inside the CUDA graph
                      ("queue", {"MMSBM_NO_GRAPH": "1", "MMSBM_NO_OVERLAP": "1", "MMSBM_DYN": "1"}),
                      ("queue+graph", {"MMSBM_NO_OVERLAP": "1", "MMSBM_DYN": "1"}),
                      ("queue+overlap", {"MMSBM_FORCE_OVERLAP": "1", "MMSBM_DYN": "1"})):
        for k in ("MMSBM_NO_GRAPH", "MMSBM_NO_OVERLAP", "MMSBM_FORCE_OVERLAP", "MMSBM_DYN"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        e = Engine(data, 900, 500, 5, 12, 9)
        e.set_params(theta, eta, pr)
        e.run(11)
        outs[name] = e.get_params() + (e.likelihood(),)
    for name in ("graph", "overlap", "queue", "queue+graph", "queue+overlap"):
        for a, b in zip(outs["plain"], outs[name]):
            np.testing.assert_array_equal(a, b, err_msg=name)


def test_likelihood_paths_agree(monkeypatch):
    """The factorised likelihood (O(K+L) per rating) against the element-wise kernel (the
    reference's per-element clamp, K*L visits) and the oracle; the run batching that adapts to
    the workspace size must not change a bit."""
    import torch
    from mmsbm_b200 import _lib
    from mmsbm_b200.engine import Engine
    for (K, L, R, S, heavy) in ((20, 20, 5, 3, True), (10, 7, 4, 2, False), (32, 32, 5, 1, False)):
        N, U, I = 50000, 600, 400
        data = random_triples(101, N, U, I, R, heavy_tail=heavy)
        theta, eta, pr = random_params(103, U, I, K, L, R, S=S)
        theta[:, 5, 0] = 0.0                                   # exact zeros: x log x := 0
        pr[:, 0, 0, 0] = 1e-300                                # an element far below eps
        e = Engine(data, U, I, R, K, L)
        e.set_params(theta, eta, pr)
        fast = e.likelihood()
        monkeypatch.setenv("MMSBM_LIK_ELEMENTWISE", "1")
        slow = e.likelihood()
        monkeypatch.delenv("MMSBM_LIK_ELEMENTWISE")
        for s in range(S):
            want = sum(orc.likelihood(data[lo:lo + 10000], theta[s], eta[s], pr[s]) for lo in range(0, N, 10000))
            assert abs(slow[s] - want) <= 1e-11 * abs(want)
            assert abs(fast[s] - want) <= 1e-10 * abs(want)    # spec: 1e-8
        # smallest accepted workspace (one run per batch) gives the same bits as the full one
        need = _lib.C.c_size_t(0)
        lib = e.lib
        _lib.check(lib.mmsbm_likelihood_min_workspace_bytes(N, U, I, R, K, L, S, _lib.C.byref(need)), "min ws")
        ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
        out = torch.empty(S, dtype=torch.float64, device="cuda")
        _lib.check(lib.mmsbm_likelihood(e.useg.data_ptr(), e.uadj.data_ptr(), e.usched.data_ptr(), N, U, I, R, K, L, S,
                                        e.theta.data_ptr(), e.eta.data_ptr(), e.pr.data_ptr(), out.data_ptr(),
                                        ws.data_ptr(), need.value, torch.cuda.current_stream().cuda_stream), "lik")
        np.testing.assert_array_equal(out.cpu().numpy(), fast)
        small = torch.empty(1024, dtype=torch.uint8, device="cuda")
        rc = lib.mmsbm_likelihood(e.useg.data_ptr(), e.uadj.data_ptr(), e.usched.data_ptr(), N, U, I, R, K, L, S,
                                  e.theta.data_ptr(), e.eta.data_ptr(), e.pr.data_ptr(), out.data_ptr(),
                                  small.data_ptr(), 1024, torch.cuda.current_stream().cuda_stream)
        assert rc != 0                                          # too small: an error, not a wrong answer


# ------------------------------------------------------------------- predict / stats (a6, a10)
def test_predict_stats_vs_oracle():
    from mmsbm_b200.engine import predict_stats
    g = np.random.default_rng(47)
    M, R, S = 5000, 5, 3
    rat = g.random((S, M, R))
    rat /= rat.sum(axis=2, keepdims=True)
    rat[0, :50] = 0.0                       # rows without prediction are dropped
    rat[1, 100:120] = 0.2                   # exact ties -> first maximum
    rat[2, 200, :] = [0, 0.5, 0, 0.5, 0]    # E[r] = 2 exactly; also a tie
    rat[2, 201, :] = [0.5, 0.5, 0, 0, 0]    # E[r] = 0.5 -> rounds half to even (0)
    real = g.integers(0, R, M)
    stats, pred = predict_stats(rat, real, want_pred=True)
    for s in range(S):
        want = orc.prediction_stats(rat[s], real, list(range(R)))
        np.testing.assert_array_equal(pred[s], np.argmax(rat[s], axis=1))      # bit-exact predictions
        for k in ("accuracy", "one_off_accuracy", "mae"):
            assert stats[s][k] == want[k], k
        assert int(stats[s]["s2"]) == int(want["s2"])
        assert abs(stats[s]["s2pond"] - want["s2pond"]) <= 1e-12 * want["s2pond"]


def test_mmsbm_fixture_known_answers(golden_dir, tmp_path, monkeypatch):
    """The reference's own end-to-end tests (tests/test_mmsbm.py:53-102) on this package."""
    monkeypatch.chdir(tmp_path)
    from mmsbm_b200 import MMSBM
    meta = json.load(open(os.path.join(golden_dir, "fixture.json")))
    g = _gold(golden_dir, "fixture.npz")
    mm = MMSBM(2, 2, iterations=10, seed=1)
    mm.fit(mock_data(1))
    pred = mm.predict(mock_data(2))
    sc = mm.score(silent=True)
    assert pred.sum() == pytest.approx(100, 0.01)
    assert rel_err(pred, g["prediction"]) < 1e-9
    st = sc["stats"]
    assert st["accuracy"] == pytest.approx(0.13, 0.01)
    assert st["one_off_accuracy"] == pytest.approx(0.55, 0.01)
    assert st["mae"] == pytest.approx(0.78, 0.01)
    assert st["s2"] == 153
    assert st["s2pond"] == pytest.approx(129.4766730930339, rel=1e-9)
    assert st["likelihood"] == pytest.approx(-13.773187406968459, rel=LIK_TOL)
    for k in ("accuracy", "one_off_accuracy", "mae", "s2"):
        assert float(st[k]) == meta["stats"][k]
    assert sc["objects"]["theta"].sum(axis=0)[0] == pytest.approx(meta["theta_col0_sum"], rel=1e-9)
    assert sc["objects"]["eta"].sum(axis=0)[0] == pytest.approx(meta["eta_col0_sum"], rel=1e-9)
    assert set(sc["objects"]["pr"].keys()) == {"1", "2", "3", "4", "5"}
    assert [float(a.sum().sum()) for a in sc["objects"]["pr"].values()] == pytest.approx(meta["pr_sums"], rel=1e-9)
    assert list(sc["objects"]["theta"].index) == meta["theta_index"]
    assert rel_err(mm.results[0]["theta"], g["theta10"]) < 1e-9
    assert mm.score(silent=False)["stats"]["accuracy"] == st["accuracy"]     # logging branch


def test_save_load_round_trip(tmp_path, monkeypatch):
    """MMSBM.save / MMSBM.load: the restored model predicts and scores bit-identically, keeps the
    dictionaries and every run, and refuses what needs the training rows."""
    monkeypatch.chdir(tmp_path)
    from mmsbm_b200 import MMSBM
    mm = MMSBM(3, 2, iterations=12, sampling=3, seed=5)
    mm.fit(mock_data(1))
    pred = mm.predict(mock_data(2))
    sc = mm.score(silent=True)
    path = str(tmp_path / "model.npz")
    mm.save(path)
    back = MMSBM.load(path)
    assert back.sampling == 3 and back.user_groups == 3 and back.iterations == 12
    assert back.data_handler.return_dicts() == mm.data_handler.return_dicts()
    for a, b in zip(mm.results, back.results):
        for k in ("theta", "eta", "pr"):
            np.testing.assert_array_equal(a[k], b[k])
        assert a["likelihood"] == b["likelihood"]
    np.testing.assert_array_equal(back.predict(mock_data(2)), pred)
    sc2 = back.score(silent=True)
    assert sc2["stats"] == sc["stats"]
    assert sc2["objects"]["theta"].equals(sc["objects"]["theta"])
    with pytest.raises(RuntimeError):
        back._engine.run(1)
    with pytest.raises(AssertionError):
        MMSBM(2, 2).save(path)                       # not fitted


def test_mmsbm_best_run_choice(golden_dir, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    from mmsbm_b200 import MMSBM
    g = _gold(golden_dir, "sampling3.npz")
    mm = MMSBM(2, 2, iterations=10, sampling=3, seed=1)
    mm.fit(mock_data(1), silent=True)
    pred = mm.predict(mock_data(2))
    for s in range(3):
        assert rel_err(mm.results[s]["theta"], g["thetas"][s]) < 1e-9
        assert abs(mm.results[s]["likelihood"] - g["likelihoods"][s]) <= LIK_TOL * abs(g["likelihoods"][s])
    rats = [mm.em.compute_prod_dist(mm.test, a["theta"], a["eta"], a["pr"]) for a in mm.results]
    assert [mm._compute_stats(a)["accuracy"] for a in rats] == g["accuracies"].tolist()
    assert mm.choose_best_run(rats) == int(g["best"]) == 1
    assert mm.likelihood == pytest.approx(float(g["likelihoods"][1]), rel=LIK_TOL)
    assert rel_err(pred, g["prediction"]) < 1e-9
    stats = mm.score(silent=True)["stats"]
    want = dict(zip(g["stats_keys"].tolist(), g["stats_vals"].tolist()))
    for k in ("accuracy", "one_off_accuracy", "mae", "s2"):
        assert float(stats[k]) == want[k]


def test_mmsbm_cv_fit(golden_dir, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    from mmsbm_b200 import MMSBM
    want = json.load(open(os.path.join(golden_dir, "cvfit.json")))
    mm = MMSBM(2, 2, iterations=10, seed=1)
    acc = mm.cv_fit(mock_data(1), folds=2)
    assert acc[0] == pytest.approx(0.125, 0.01) and acc[1] == pytest.approx(0.16, 0.01)
    assert [float(a) for a in acc] == want["accuracies"]
    np.testing.assert_array_equal(np.asarray(mm.test), np.asarray(want["final_test"]))


def test_api_guards_and_helpers(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    from mmsbm_b200 import MMSBM
    from mmsbm_b200.data_handler import DataHandler
    with pytest.raises(AssertionError):
        MMSBM(2, 2, seed=1).predict(mock_data(0))
    with pytest.raises(AssertionError):
        MMSBM(2, 2, seed=1).score()
    mm = MMSBM(1, 1, seed=1)
    monkeypatch.setattr(mm, "_compute_stats", lambda x: {"accuracy": x})
    assert mm.choose_best_run([0.1, 0.7, 0.3]) == 1
    mm = MMSBM(2, 2, iterations=1, sampling=1, seed=2)
    train = DataHandler().format_train_data(mock_data(2, n=15))
    mm._prepare_objects(train)
    res = mm.run_one_sampling(train, seed=123, i=0)
    assert set(res) == {"likelihood", "pr", "theta", "eta"} and res["pr"].shape[:2] == (2, 2)
    want = orc.run_em(train, 123, 2, 2, 1)
    assert rel_err(res["theta"], want["theta"]) < PARAM_TOL
    assert np.isfinite(mm.compute_likelihood(mm.train, res["theta"], res["eta"], res["pr"]))


def test_reference_style_loop_through_the_plugin(golden_dir):
    """The reference's own loop (src/mmsbm.py:243-256) driven through the plugin contract: every
    iteration calls update_coefficients on host arrays, the driver normalises on the host, exactly
    as MMSBM.run_one_sampling does with backend='b200' (INTEGRATION.md, level 1)."""
    from mmsbm_b200 import ExpectationMaximization
    g = _gold(golden_dir, "fixture.npz")
    train = g["train"]
    dims = {"n_samples": len(train), "n_user_groups": 2, "n_item_groups": 2, "n_ratings": 5}
    em = ExpectationMaximization(dims, None, None, None,
                                 {"user": g["norm_user"], "item": g["norm_item"]}, backend="b200")
    assert em._backend == "b200"
    theta, eta, pr = g["theta0"], g["eta0"], g["pr0"]
    for _ in range(10):
        n_theta, n_eta, npr = em.update_coefficients(data=train, theta=theta, eta=eta, pr=pr)
        theta = em.normalize_with_d(n_theta, "user")
        eta = em.normalize_with_d(n_eta, "item")
        pr = em.normalize_with_self(npr)
    assert rel_err(theta, g["theta10"]) < 1e-9 and rel_err(eta, g["eta10"]) < 1e-9
    assert rel_err(pr, g["pr10"]) < 1e-9
    lik = em.compute_likelihood(train, theta, eta, pr)
    assert abs(lik - g["likelihood10"]) <= LIK_TOL * abs(g["likelihood10"])
    rat = em.compute_prod_dist(g["test"], theta, eta, pr)
    assert rel_err(rat, g["prediction"]) < 1e-9
    assert rel_err(em.prod_dist(g["test"][0], theta, eta, pr), g["prediction"][0]) < 1e-9


def test_reference_loader_contract():
    """load_backend returns the reference's 4-tuple; kernels_b200 at the repo root is the
    module the REFERENCE's loader would import for backend='b200'."""
    import kernels_b200 as plugin
    from mmsbm_b200 import load_backend
    co, uc, pdist, name = load_backend("auto")
    assert name == "b200" and co is plugin.compute_omegas and uc is plugin.update_coefficients
    with pytest.raises(ImportError):
        load_backend("numpy")


# ------------------------------------------------------- full-size properties (BASELINE shapes)
@pytest.mark.parametrize("shape", [
    dict(name="ML-1M", N=1_000_000, U=6040, I=3706, K=10, L=10, S=8),
    dict(name="ML-20M", N=20_000_000, U=138_000, I=27_000, K=20, L=20, S=2),
    dict(name="ML-20M six runs per warp + a single", N=20_000_000, U=138_000, I=27_000, K=20, L=20, S=7),
    dict(name="ML-20M sampling=8 (the bench configuration: six runs + a pair)", N=20_000_000, U=138_000,
         I=27_000, K=20, L=20, S=8),
    dict(name="ML-100K (per-CTA piece ranges, one run)", N=100_000, U=943, I=1682, K=10, L=10, S=1),
])
def test_full_size_invariants(shape):
    """At sizes the oracle cannot reach, check what must hold for any input: each rating
    distributes unit mass (sum n_pr = N), theta rows sum to 1, eta rows sum to 1, pr sums
    to 1 over ratings, and a subsample of users / items agrees with the oracle restricted to
    their rows (theta_u' depends only on u's ratings)."""
    from mmsbm_b200 import _lib
    from mmsbm_b200.engine import Engine
    N, U, I, K, L, S = (shape[k] for k in ("N", "U", "I", "K", "L", "S"))
    R = 5
    data = random_triples(53, N, U, I, R)
    theta, eta, pr = random_params(59, U, I, K, L, R, S=S)
    e = Engine(data, U, I, R, K, L)
    e.set_params(theta, eta, pr)
    raw = e.step_raw(_lib.RAW_THETA | _lib.RAW_ETA_PR)
    npr = raw[2].cpu().numpy()
    for s in range(S):
        assert abs(npr[s].sum() - N) <= 1e-9 * N
    nth = raw[0].cpu().numpy()[..., :K]
    net = raw[1].cpu().numpy()[..., :L]
    deg = np.bincount(data[:, 0], minlength=U)
    np.testing.assert_allclose(nth.sum(axis=2), np.broadcast_to(deg, (S, U)), rtol=1e-11)
    # marginals that tie n_pr to the other two sums for EVERY run: all three are sums of the same
    # increments inc[n,k,l], so  sum_lr n_pr[k,l,r] = sum_u n_theta[u,k],  sum_kr n_pr[k,l,r] =
    # sum_i n_eta[i,l],  and  sum_kl n_pr[k,l,r] = number of ratings at level r
    levels = np.bincount(data[:, 2], minlength=R)
    for s in range(S):
        np.testing.assert_allclose(npr[s].sum(axis=(1, 2)), nth[s].sum(axis=0), rtol=1e-10)
        np.testing.assert_allclose(npr[s].sum(axis=(0, 2)), net[s].sum(axis=0), rtol=1e-10)
        np.testing.assert_allclose(npr[s].sum(axis=(0, 1)), levels, rtol=1e-10)
    e.run(1)
    th, et, prn = e.get_params()
    np.testing.assert_allclose(th.sum(axis=2), 1.0, rtol=1e-11)
    np.testing.assert_allclose(et.sum(axis=2), 1.0, rtol=1e-11)
    np.testing.assert_allclose(prn.sum(axis=3), 1.0, rtol=1e-11)
    users = np.array([0, 1, U // 2, U - 1])
    rows_u = data[np.isin(data[:, 0], users)]
    items = np.array([0, I // 3, I - 1])
    rows_i = data[np.isin(data[:, 1], items)]
    degi = np.bincount(data[:, 1], minlength=I)
    for s in range(S):                                       # every run, not only the first
        rt, _, _ = orc.em_sums(rows_u, theta[s], eta[s], pr[s])
        assert rel_err(th[s][users] * np.maximum(deg[users], 1)[:, None], rt[users]) < PARAM_TOL
        _, re_, _ = orc.em_sums(rows_i, theta[s], eta[s], pr[s], chunk=20000)
        assert rel_err(et[s][items] * np.maximum(degi[items], 1)[:, None], re_[items]) < PARAM_TOL


def test_ml20m_eight_runs_restricted_problem_vs_oracle():
    """n_pr (and everything else) of the ML-20M bench configuration -- K = L = 20, sampling = 8, the
    full 138k x 27k id ranges, so the six-run + pair kernels and the full-size tables -- element by
    element against the oracle, on a 2e5-row restriction of the ratings that the oracle finishes in
    seconds; once with the per-CTA piece ranges a problem of this size gets by default and once
    with the launch-wide piece queue the full-size problem uses."""
    import os
    from mmsbm_b200.engine import Engine
    U, I, K, L, S, R, n = 138_000, 27_000, 20, 20, 8, 5, 200_000
    rows = random_triples(61, n, U, I, R)            # n >= U: every user id appears at least once
    theta, eta, pr = random_params(67, U, I, K, L, R, S=S)
    fu, fi = orc.degree_factors(rows, K, L)
    want = [orc.em_iteration(rows, theta[s], eta[s], pr[s], fu, fi, chunk=20000) for s in range(S)]
    want_lik = [sum(orc.likelihood(rows[lo:lo + 20000], *want[s]) for lo in range(0, n, 20000)) for s in range(S)]
    for dyn in ("0", "1"):
        os.environ["MMSBM_DYN"] = dyn
        try:
            e = Engine(rows, U, I, R, K, L)
            e.set_params(theta, eta, pr)
            e.run(1)
            th, et, prn = e.get_params()
            lik = e.likelihood()
        finally:
            del os.environ["MMSBM_DYN"]
        worst = 0.0
        for s in range(S):
            worst = max(worst, rel_err(th[s], want[s][0]), rel_err(et[s], want[s][1]), rel_err(prn[s], want[s][2]))
            assert abs(lik[s] - want_lik[s]) <= LIK_TOL * abs(want_lik[s])
        print(f"ML-20M S=8 restricted, piece queue={dyn}: worst rel err {worst:.3e}")
        assert worst < PARAM_TOL


def test_ml100k_full_fit_likelihood_vs_oracle():
    """BASELINE.json configs[0] in full: 943 x 1682, 1e5 ratings, K = L = 10, one run, 200 iterations
    from the reference's seeded init (src/mmsbm.py:224-233), GPU loop (CUDA-graph replay of
    iteration pairs) against the oracle's loop.  Final likelihood within 1e-8 relative
    (north_star); the drift of theta / eta / pr after 200 iterations is printed and bounded."""
    from mmsbm_b200.engine import Engine
    U, I, N, K, L, R, T = 943, 1682, 100_000, 10, 10, 5, 200
    data = random_triples(71, N, U, I, R, heavy_tail=True)
    fu, fi = orc.degree_factors(data, K, L)
    _, kids = orc.child_seeds(1, 1)
    th, et, pr = orc.seeded_init(kids[0], U, I, K, L, R, fu, fi)
    e = Engine(data, U, I, R, K, L)
    e.set_params(th[None], et[None], pr[None])
    e.run(T)
    g_th, g_et, g_pr = e.get_params()
    g_lik = e.likelihood()[0]
    for _ in range(T):
        th, et, pr = orc.em_iteration(data, th, et, pr, fu, fi)
    want = orc.likelihood(data, th, et, pr)
    drift = (float(np.max(np.abs(g_th[0] - th))), float(np.max(np.abs(g_et[0] - et))), float(np.max(np.abs(g_pr[0] - pr))))
    print(f"ML-100K x {T} iterations: likelihood {g_lik!r} vs {want!r} (rel {abs(g_lik - want) / abs(want):.2e}), "
          f"max abs drift theta/eta/pr {drift}")
    assert abs(g_lik - want) <= LIK_TOL * abs(want)
    assert max(drift) < 1e-8


def test_ml1m_eight_runs_same_best_sample_as_oracle():
    """BASELINE.json configs[1] shape (6040 x 3706, 1e6 ratings, K = L = 10, sampling = 8): after two
    iterations of every run from the reference's seeded init, the per-run accuracy counts on a
    held-out set, the predicted ratings (bit-exact) and hence the run ``predict`` selects
    (src/mmsbm.py:306,474-478) are the oracle's."""
    from mmsbm_b200.engine import Engine, predict_stats
    U, I, N, K, L, R, S, T = 6040, 3706, 1_000_000, 10, 10, 5, 8, 2
    data = random_triples(73, N, U, I, R)
    test = random_triples(79, 100_000, U, I, R)
    fu, fi = orc.degree_factors(data, K, L)
    _, kids = orc.child_seeds(1, S)
    inits = [orc.seeded_init(k, U, I, K, L, R, fu, fi) for k in kids]
    e = Engine(data, U, I, R, K, L)
    e.set_params(*(np.stack([a[j] for a in inits]) for j in range(3)))
    e.run(T)
    stats, pred = predict_stats(e.prod_dist_device(test), test[:, 2], want_pred=True)
    lik = e.likelihood()
    acc_gpu = [s["accuracy"] for s in stats]
    acc_cpu = []
    for s in range(S):
        th, et, pr = inits[s]
        for _ in range(T):
            th, et, pr = orc.em_iteration(data, th, et, pr, fu, fi, chunk=100_000)
        rat = orc.rating_distribution(test, th, et, pr)
        np.testing.assert_array_equal(pred[s], np.argmax(rat, axis=1))
        acc_cpu.append(orc.prediction_stats(rat, test[:, 2], list(range(R)))["accuracy"])
        want = sum(orc.likelihood(data[lo:lo + 100_000], th, et, pr) for lo in range(0, N, 100_000))
        assert abs(lik[s] - want) <= LIK_TOL * abs(want)
    assert acc_gpu == acc_cpu
    assert acc_gpu.index(max(acc_gpu)) == acc_cpu.index(max(acc_cpu))


# ------------------------------------------------------------- sharded runs (one rank here)
@pytest.mark.parametrize("K,L,S", [(20, 20, 8), (32, 32, 1), (10, 10, 3), (7, 5, 2)])
def test_sharded_engine_with_one_rank_equals_engine(K, L, S):
    """mmsbm_em_run_sharded with world = 1 (own ranges = everything, no peers, no collective) walks
    the same kernels over tables kept in the exchange buffer: bit-identical to mmsbm_em_run."""
    from mmsbm_b200.engine import Engine
    from mmsbm_b200.parallel import ShardedEngine
    N, U, I, R = 50000, 600, 400, 5
    data = random_triples(91, N, U, I, R, heavy_tail=True)
    theta, eta, pr = random_params(93, U, I, K, L, R, S=S)
    a = Engine(data, U, I, R, K, L)
    a.set_params(theta, eta, pr)
    a.run(5)
    b = ShardedEngine(data, U, I, R, K, L)
    b.set_params(theta, eta, pr)
    b.run(3)
    b.run(2)                                                 # odd + even: both halves of the tables
    for x, y in zip(a.get_params(), b.get_params()):
        np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(a.likelihood(), b.likelihood())
    ms = b.run(2, prof=True)
    assert ms[0] > 0.0
    b.close()


def test_one_sided_build_equals_a_slice_of_the_full_index():
    """mmsbm_graph_build_side on the rows of a user range (what a caller that pre-partitions its
    ratings would use) == the slice of the full index a ShardedEngine rank works on, and
    mmsbm_sched_build on the degree slice == the schedule the one-sided build makes."""
    import ctypes as C
    import torch
    from mmsbm_b200 import _lib
    from mmsbm_b200.engine import Engine
    lib = _lib.load(require_device=True)
    N, U, I, R = 90000, 500, 300, 5
    data = random_triples(97, N, U, I, R, heavy_tail=True)       # user 0 holds > 2048 ratings: pieces
    full = Engine(data, U, I, R, 4, 4)
    lo, hi = 0, 140
    rows = data[(data[:, 0] >= lo) & (data[:, 0] < hi)].copy()
    rows[:, 0] -= lo
    n, n_ids = len(rows), hi - lo
    dev, i32 = full.device, torch.int32
    cols = [torch.from_numpy(np.ascontiguousarray(rows[:, c], dtype=np.int32)).to(dev) for c in range(3)]
    seg = torch.empty(n_ids * R + 1, dtype=i32, device=dev)
    adj, perm = torch.empty(n, dtype=i32, device=dev), torch.empty(n, dtype=i32, device=dev)
    deg = torch.empty(n_ids, dtype=i32, device=dev)
    ne, need = C.c_int64(0), C.c_size_t(0)
    _lib.check(lib.mmsbm_sched_elems(n, n_ids, C.byref(ne)), "sched_elems")
    sched = torch.zeros(ne.value, dtype=i32, device=dev)
    _lib.check(lib.mmsbm_graph_workspace_bytes(n, n_ids, n_ids, R, C.byref(need)), "graph_workspace_bytes")
    ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.mmsbm_graph_build_side(cols[0].data_ptr(), cols[1].data_ptr(), cols[2].data_ptr(), n, n_ids, R,
                                          seg.data_ptr(), adj.data_ptr(), perm.data_ptr(), deg.data_ptr(),
                                          sched.data_ptr(), ws.data_ptr(), need.value, st), "graph_build_side")
    torch.cuda.synchronize()
    fseg = full.useg.cpu().numpy()
    base = fseg[lo * R]
    np.testing.assert_array_equal(seg.cpu().numpy(), fseg[lo * R:hi * R + 1] - base)
    np.testing.assert_array_equal(adj.cpu().numpy(), full.uadj.cpu().numpy()[base:fseg[hi * R]])
    np.testing.assert_array_equal(deg.cpu().numpy(), full.udeg.cpu().numpy()[lo:hi])
    assert n == fseg[hi * R] - base
    _lib.check(lib.mmsbm_sched_workspace_bytes(n_ids, C.byref(need)), "sched_workspace_bytes")
    ws2 = torch.empty(need.value, dtype=torch.uint8, device=dev)
    sched2 = torch.zeros(ne.value, dtype=i32, device=dev)
    _lib.check(lib.mmsbm_sched_build(full.udeg[lo:].data_ptr(), n_ids, n, sched2.data_ptr(), ws2.data_ptr(),
                                     need.value, st), "sched_build")
    torch.cuda.synchronize()
    a, b = sched.cpu().numpy(), sched2.cpu().numpy()
    assert a[0] > n_ids and a[2] >= 1                        # more pieces than segments: a long one exists
    pmax = n_ids + n // 2048 + 1
    lmax = n // 2048 + 1
    np.testing.assert_array_equal(a[:4], b[:4])
    for off, cnt in ((4, a[0]), (4 + pmax, a[0]), (4 + 2 * pmax, a[0]), (4 + 3 * pmax, a[2]),
                     (4 + 3 * pmax + lmax, a[2] + 1)):       # the filled part of each table
        np.testing.assert_array_equal(a[off:off + cnt], b[off:off + cnt])


# ------------------------------------------------------------- small one-run problems: one cooperative launch
@pytest.mark.parametrize("U,I,N,K,L,R,heavy,T", [
    (943, 1682, 100_000, 10, 10, 5, False, 7),       # the ML-100K shape
    (300, 200, 10_000, 10, 10, 5, True, 4),          # heavy-tailed: the top segments (1024 < ratings <= 2048) take the CTA-wide walk
    (300, 200, 40_000, 10, 10, 5, True, 4),          # a segment of > 2048 ratings: stays on the multi-kernel path
    (5, 10, 100, 2, 2, 5, False, 10),                # the reference fixture's shape (4-double rows, one lane per row)
    (400, 900, 30_000, 7, 8, 4, True, 3),            # 8-double rows, K != L inside one stride
    (50, 40, 3000, 12, 9, 8, False, 1),              # eight rating levels, a single iteration
    (700, 30, 40_000, 3, 4, 3, True, 5),             # more users than items and the reverse below: either side emits n_pr
    (30, 700, 40_000, 4, 3, 3, True, 6),
])
def test_cooperative_small_path_vs_oracle(U, I, N, K, L, R, heavy, T, monkeypatch):
    """mmsbm_em_run takes one-run problems with rows of at most 12 doubles and no segment beyond
    2048 ratings through em_small.cu (the whole loop in one cooperative launch).  T iterations against the oracle's loop (1e-10 per element
    per iteration would allow T * 1e-10; observed ~1e-14), likelihood within 1e-8, ids without any
    rating keep zero rows, and the multi-kernel path (MMSBM_COOP=0) agrees to rounding."""
    from mmsbm_b200 import _lib
    from mmsbm_b200.engine import Engine
    data = random_triples(101, N, U, I, R, heavy_tail=heavy)
    data = data[data[:, 0] != 1]                              # user 1 has no rating at all
    theta, eta, pr = random_params(103, U, I, K, L, R, S=1)
    fu = np.repeat(np.maximum(np.bincount(data[:, 0], minlength=U), 1)[:, None], K, axis=1)
    fi = np.repeat(np.maximum(np.bincount(data[:, 1], minlength=I), 1)[:, None], L, axis=1)
    outs = {}
    for coop in ("1", "0"):
        monkeypatch.setenv("MMSBM_COOP", coop)
        l0 = _lib.launch_count()
        e = Engine(data, U, I, R, K, L)
        e.set_params(theta, eta, pr)
        l1 = _lib.launch_count()
        e.run(T)
        launches = _lib.launch_count() - l1
        outs[coop] = e.get_params() + (e.likelihood(),)
        top = max(np.bincount(data[:, 0]).max(), np.bincount(data[:, 1]).max())
        if coop == "1" and top <= 2048:
            assert launches == 1, launches                   # ONE kernel for all T iterations
        else:
            assert launches > T
        if (U, N) == (300, 10_000):
            assert 1024 < top <= 2048
        del l0
    t, et, p = theta[0], eta[0], pr[0]
    for _ in range(T):
        t, et, p = orc.em_iteration(data, t, et, p, fu, fi)
    want_lik = orc.likelihood(data, t, et, p)
    for coop, (gt, ge, gp, glik) in outs.items():
        errs = (rel_err(gt[0], t), rel_err(ge[0], et), rel_err(gp[0], p))
        print(f"coop={coop} U={U} I={I} K={K} L={L} R={R}: rel err after {T} iterations {errs}")
        assert max(errs) < PARAM_TOL * T
        assert abs(glik[0] - want_lik) <= LIK_TOL * abs(want_lik)
        assert np.all(gt[0][1] == 0.0)
    for a, b in zip(outs["1"][:3], outs["0"][:3]):
        assert rel_err(a, b) < 1e-11
