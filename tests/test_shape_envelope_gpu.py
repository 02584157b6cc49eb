"""Every corner of the shape envelope MMSBM admits, on the B200, against the oracle.

``MMSBM._check_shape`` promises that any K, L <= 256 and R <= 31 is served, provided R * ld <= 1024
when a side has more than 32 groups (ld: the group count rounded up to a multiple of 4).  The
kernels pick among many template instances by row stride, run grouping and shared-memory size; this
file runs the edges of that envelope through each of them:

* a sweep over every row-stride class ld = 4, 8, ..., 256 (square and both lopsided shapes, at the
  largest admitted R and at R = 5, with run counts that reach the pair and six-run groupings),
  comparing one EM step, the likelihood, the rating distributions and fold-in with the oracle;
* end-to-end fits at shapes whose sizes sit at the shared-memory limits;
* a coverage check: every kernel variant the default dispatch can pick is launched by the sweep, and
  the library holds no segment-pass instance the dispatch cannot pick.

The shapes come from ``_check_shape`` itself, so the sweep follows the rule if it ever changes."""
import os
import re
import subprocess

import numpy as np
import pandas as pd
import pytest

from oracle import mmsbm_oracle as orc
from tests import fold_in_reference as fref
from tests.test_em_gpu import LIK_TOL, PARAM_TOL
from tests.test_fold_in_gpu import caps
from tests.util import random_params, random_triples, rel_err

MAX_GROUPS, MAX_LEVELS = 256, 31


def admitted(K, L, R):
    from mmsbm_b200 import MMSBM
    m = MMSBM.__new__(MMSBM)            # _check_shape reads the group counts only
    m.user_groups, m.item_groups = K, L
    try:
        m._check_shape(R)
    except ValueError:
        return False
    return True


def envelope_cases():
    """(K, L, R, S) corner shapes of the envelope: per row-stride class, a square shape and the two
    lopsided ones against a narrow side of 3-5 groups; the wide side's padding (ld - K) rotates
    through 0..3 over the classes.  Each at the largest admitted R and at R = 5; S = 1 and 2, plus
    S = 6 and 8 (six-run and pair groupings) for rows of at most 32 doubles."""
    cases = []
    for ld in range(4, MAX_GROUPS + 1, 4):
        wide = ld - (ld // 4) % 4 if ld > 4 else ld
        narrow = 3 + (ld // 4) % 3
        for K, L in ((ld, max(ld - 1, 1)), (wide, narrow), (narrow, wide)):
            r_max = max(r for r in range(1, MAX_LEVELS + 1) if admitted(K, L, r))
            levels = [r_max] + ([5] if r_max != 5 and admitted(K, L, 5) else [])
            for R in levels:
                for S in (1, 2) + ((6, 8) if ld <= 32 else ()):
                    cases.append((K, L, R, S))
    return cases


CASES = envelope_cases()


def case_id(c):
    return "K%d_L%d_R%d_S%d" % c


def problem(case):
    """A tiny problem: every id and level present, a few hundred ratings (fewer where K*L*R is large,
    to bound the oracle's work), heavy-tailed ids for every other shape."""
    K, L, R, S = case
    U, I = 36, 28
    N = int(np.clip(3e7 / (K * L * R), 200, 400 + 4 * R))
    seed = K * 10007 + L * 101 + R * 7 + S
    data = random_triples(seed, N, U, I, R, heavy_tail=seed % 2 == 1)
    theta, eta, pr = random_params(seed + 1, U, I, K, L, R, S=S)
    return data, (U, I), (theta, eta, pr)


def chunk_rows(K, L):
    """Rows per oracle block: the [chunk, K, L] temporaries stay near 200 MB."""
    return max(1, int(2e8 // (K * L * 8)))


def oracle_likelihood(data, theta, eta, pr):
    c = chunk_rows(theta.shape[1], eta.shape[1])
    return sum(orc.likelihood(data[lo:lo + c], theta, eta, pr) for lo in range(0, len(data), c))


def fold_rows(case, side, n_other, seed):
    """Fold-in rows for new ids of `side`: one id beyond a CTA's rows (cut into pieces, fix-up
    kernel), ids at and just past a warp's slice, and short ones; levels 0..R-1.  Rows of 4 and 8
    doubles take 1.5-3k ratings to pass a CTA: that id is left out there unless the other side is
    as narrow (the oracle's cost grows with K*L per rating)."""
    K, L, R, _ = case
    cap_w, cap_c = caps(K if side == 0 else L)
    degrees = [cap_w, cap_w + 1, 1, 3]
    if cap_c <= 1024 or max(K, L) <= 8:
        degrees = [cap_c + 5] + degrees
    g = np.random.default_rng(seed)
    own = np.repeat(np.arange(len(degrees)), degrees)
    other = g.integers(0, n_other, len(own))
    level = g.integers(0, R, len(own))
    perm = g.permutation(len(own))
    own, other, level = own[perm], other[perm], level[perm]
    rows = np.stack([own, other, level] if side == 0 else [other, own, level], axis=1).astype(np.int64)
    return rows, len(degrees)


def run_case(case, check):
    """Drive every kernel family at `case`; with `check`, compare each result with the oracle."""
    from mmsbm_b200.engine import Engine
    K, L, R, S = case
    data, (U, I), (theta, eta, pr) = problem(case)
    e = Engine(data, U, I, R, K, L)
    e.set_params(theta, eta, pr)

    # fold-in on both sides, with the parameters just set
    for side in (0, 1):
        rows, n_new = fold_rows(case, side, I if side == 0 else U, seed=K + L + R + S + side)
        width = K if side == 0 else L
        init = np.random.default_rng(side).random((S, n_new, width))
        want, done = init, 0
        for it in ((1, 5) if check else (1,)):
            got = e.fold_in(side, rows, init, it)
            if not check:
                continue
            # the reference continues from its previous result: the same iterations, computed once
            if side == 0:
                want = np.stack([fref.fold_in(rows, want[s], eta[s], pr[s], it - done, side=0) for s in range(S)])
            else:
                want = np.stack([fref.fold_in(rows, theta[s], want[s], pr[s], it - done, side=1) for s in range(S)])
            done = it
            err = rel_err(got, want)
            assert err < 1e-10, ("fold-in", side, it, err)

    # one EM step
    e.run(1)
    th, et, prn = e.get_params()
    lik = e.likelihood()
    rat = e.prod_dist_device(data).cpu().numpy()
    if not check:
        return
    fu, fi = orc.degree_factors(data, K, L)
    for s in range(S):
        rt, re_, rp = orc.em_iteration(data, theta[s], eta[s], pr[s], fu, fi, chunk=chunk_rows(K, L))
        err = max(rel_err(th[s], rt), rel_err(et[s], re_), rel_err(prn[s], rp))
        assert err < PARAM_TOL, ("em step", s, err)
        want = oracle_likelihood(data, rt, re_, rp)
        assert abs(lik[s] - want) <= LIK_TOL * abs(want) + 1e-15 * len(data) * K * L, ("likelihood", s, lik[s], want)
        err = rel_err(rat[s], orc.rating_distribution(data, th[s], et[s], prn[s]))
        assert err < 1e-12, ("prod_dist", s, err)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_envelope_vs_oracle(case):
    run_case(case, check=True)


def test_sweep_reaches_the_corners():
    """The generated sweep holds the shapes the shared-memory limits bite at (no GPU needed)."""
    for c in [(32, 31, 31, 1), (32, 31, 31, 2), (20, 19, 31, 8), (256, 255, 4, 1), (256, 4, 4, 2),
              (4, 256, 4, 1), (128, 127, 8, 2), (64, 63, 16, 1), (64, 63, 5, 1)]:
        assert c in CASES, c
    for K, L, R, _ in CASES:
        assert admitted(K, L, R) and (R == 5 or R == MAX_LEVELS or not admitted(K, L, R + 1))


# --------------------------------------------------------------------------------- end to end
E2E = [(32, 32, 31, 1), (32, 32, 29, 2), (20, 20, 31, 8), (64, 64, 7, 1), (100, 100, 5, 1), (256, 256, 4, 1)]


def frame(R, U=40, I=30, n=900, seed=0):
    g = np.random.default_rng(seed)
    data = random_triples(seed, n, U, I, R)
    df = pd.DataFrame({"users": ["u%d" % u for u in data[:, 0]], "items": ["i%d" % i for i in data[:, 1]],
                       "ratings": data[:, 2] + 1})
    new = pd.DataFrame({"users": ["new%d" % (k % 3) for k in range(30)] + ["u%d" % k for k in range(10)],
                        "items": ["i%d" % g.integers(0, I) for _ in range(30)] + ["newi%d" % (k % 2) for k in range(10)],
                        "ratings": g.integers(1, R + 1, 40)})
    return df, new


@pytest.mark.gpu
@pytest.mark.parametrize("case", E2E, ids=case_id)
def test_fit_score_predict_save_load_fold_in(case, tmp_path, monkeypatch):
    from mmsbm_b200 import MMSBM
    monkeypatch.chdir(tmp_path)
    K, L, R, S = case
    df, new = frame(R)
    m = MMSBM(K, L, iterations=6, sampling=S, seed=3)
    m.fit(df, silent=True)
    assert len(m.results) == S and all(np.isfinite(r["likelihood"]) for r in m.results)
    test = df.sample(200, random_state=1)
    pred = m.predict(test)
    assert pred.shape == (200, R) and np.all(np.isfinite(pred))
    stats = m.score(silent=True)["stats"]
    assert 0.0 <= stats["accuracy"] <= 1.0
    m.save(str(tmp_path / "m.npz"))
    loaded = MMSBM.load(str(tmp_path / "m.npz"))
    assert np.array_equal(loaded.predict(test), pred)
    added = loaded.fold_in(new, iterations=5)
    assert added["users"] == ["new0", "new1", "new2"] and added["items"] == ["newi0", "newi1"]
    out = loaded.predict(new)
    assert out.shape == (40, R) and np.all(np.isfinite(out))


@pytest.mark.gpu
def test_sharded_engine_one_rank_at_the_pair_limit():
    """(32, 32, 31, 2): the w rows of a pair of runs do not fit shared memory, so both passes serve
    one run per warp and the exchange tables follow that plan.  World = 1 is bit-identical to
    Engine."""
    from mmsbm_b200.engine import Engine
    from mmsbm_b200.parallel import ShardedEngine
    K, L, R, S = 32, 32, 31, 2
    N, U, I = 20000, 300, 200
    data = random_triples(91, N, U, I, R, heavy_tail=True)
    theta, eta, pr = random_params(93, U, I, K, L, R, S=S)
    a = Engine(data, U, I, R, K, L)
    a.set_params(theta, eta, pr)
    a.run(3)
    b = ShardedEngine(data, U, I, R, K, L)
    b.set_params(theta, eta, pr)
    b.run(2)
    b.run(1)
    for x, y in zip(a.get_params(), b.get_params()):
        np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(a.likelihood(), b.likelihood())
    b.close()


# ---------------------------------------------------------------------------------- coverage
# Every variant the default dispatch can pick.  A kernel or an instance added to the library
# belongs in this list, and the sweep must reach it; the segment-pass instances in the library are
# exactly SEGMENT_PASS.
SEGMENT_PASS = (
    # one run per warp: ld 4, 8, 12..32 (one chunk per lane), then 2 / 4 / 8 chunks per lane
    ["segment_pass_kernel<1,1,1,3,1>", "segment_pass_kernel<2,1,2,3,1>"]
    + ["segment_pass_kernel<%d,1,3,3,1>" % g for g in range(3, 9)]
    + ["segment_pass_kernel<%d,2,1,3,1>" % g for g in range(5, 9)]
    + ["segment_pass_kernel<%d,%d,1,1,1>" % (g, ch) for ch in (4, 8) for g in range(5, 9)]
    # pairs of runs (rows of up to 32 doubles), six runs (rows of 20 doubles)
    + ["segment_pass_kernel<1,1,2,3,2>"] + ["segment_pass_kernel<%d,1,3,3,2>" % g for g in range(2, 9)]
    + ["segment_pass_kernel<5,1,3,3,6>"])
FOLD_IN = ["<4,1>", "<8,1>", "<8,2>", "<8,3>", "<8,4>"] + ["<32,%d>" % j for j in range(2, 9)]
EXPECTED = (SEGMENT_PASS
            + ["fold_in_kernel" + t for t in FOLD_IN] + ["fold_pieces_kernel" + t for t in FOLD_IN]
            + ["row_w_kernel<%d," % ld for ld in range(4, 33, 4)]
            + ["row_n_kernel<%d," % ld for ld in range(4, 33, 4)]
            + ["lik_user_tables_kernel<%d>" % ld for ld in range(4, 33, 4)]
            + ["lik_pass_kernel<%d>" % g for g in range(1, 9)]
            + ["likelihood_kernel", "lik_tables_kernel", "small_gemm_kernel<0>", "small_gemm_kernel<1>",
               "prod_dist_kernel<0>", "prod_dist_kernel<1>"])


def library_segment_pass_instances():
    """'segment_pass_kernel<G,CH,UN,MINB,RUNS>' of every instance in the library _lib loads, read from
    the mangled names that `cuobjdump -symbols` lists."""
    from mmsbm_b200 import _lib
    from mmsbm_b200.build import _nvcc
    nvcc = _nvcc()
    tool = os.path.join(os.path.dirname(nvcc), "cuobjdump") if os.path.isabs(nvcc) else "cuobjdump"
    out = subprocess.run([tool, "-symbols", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    return {"segment_pass_kernel<%s>" % ",".join(re.findall(r"Li(\d+)E", args))
            for args in re.findall(r"segment_pass_kernelI((?:Li\d+E)+)E", out)}


def normalise(name):
    """'void mmsbm::segment_pass_kernel<(int)5, (int)1, ...>(mmsbm::SegArgs)' -> 'segment_pass_kernel<5,1,...>'"""
    name = re.sub(r"\((?:int|bool)\)|\s", "", name).replace("true", "1").replace("false", "0")
    return re.sub(r"^void", "", name).split("(")[0].split("::")[-1]


@pytest.mark.gpu
def test_sweep_launches_every_kernel_variant():
    from torch.profiler import ProfilerActivity, profile
    import torch
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for case in CASES:
            run_case(case, check=False)
        torch.cuda.synchronize()
    launched = {normalise(ev.key) for ev in prof.key_averages()}
    missing = [k for k in EXPECTED if not any(n.startswith(k) for n in launched)]
    assert not missing, missing
    # the reverse: an instance the dispatch cannot pick is code no test runs
    built = library_segment_pass_instances()
    assert built, "no segment_pass_kernel symbol found"
    extra = sorted(built - set(SEGMENT_PASS))
    assert not extra, extra
