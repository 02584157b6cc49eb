"""EM to convergence (``fit(tol=...)``, ``Engine.run_converge``) at the ML-20M shape of
refit_bench.py: 138 493 users, 26 744 items, about 1.4e7 ratings from a planted model (K = L = 20,
R = 5), S = 8 runs, 1 % of the ratings held out.

1. One evaluation of the observed-data log-likelihood against one EM step (CUDA events, after
   warm-up, 20 repetitions each).
2. ``fit`` with 400 iterations against ``fit(tol=1e-4 / 1e-5 / 1e-6, check_every=10)`` with 400 as
   the maximum: wall and EM seconds, every run's stop iteration, held-out accuracy.
3. ``refit`` on all ratings with ``tol`` (maximum 400) after a 400-iteration fit on 90 %, against the
   fixed 25 / 50 / 100 iterations of refit_bench.py, measured here again.
4. The loop's own cost per check on the cooperative one-launch path (ML-100K shape: 943 users,
   1 682 items, 1e5 ratings, K = L = 10, R = 5, S = 1): ``run_converge(400, tol=0)`` minus
   ``run(400)``, divided by the 40 checks.
The card's name and power limit are read in the same run.

    python profiles/scripts/converge_bench.py [--out result.json] [--scale 1.0]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from refit_bench import I, ITERS, K, L, R, S, U, planted_rows, stages  # noqa: E402

TOLS = (1e-4, 1e-5, 1e-6)


def event_ms(call, reps):
    import torch
    call()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        call()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the users and items (rehearsal)")
    args = ap.parse_args()
    import pandas as pd
    import torch
    from fold_in_bench import card
    from mmsbm_b200 import MMSBM
    from mmsbm_b200.engine import Engine

    name, limit = card()
    nu, ni = max(int(U * args.scale), 50), max(int(I * args.scale), 50)
    rows, _ = planted_rows(3, nu, ni)
    g = np.random.default_rng(4)
    held = g.random(len(rows)) < 0.01
    first = g.random(len(rows)) < 0.9

    def frame(r):
        return pd.DataFrame({"users": r[:, 0], "items": r[:, 1], "ratings": r[:, 2] + 1})

    part, full = frame(rows[~held & first]), frame(rows[~held])
    test = frame(rows[held & np.isin(rows[:, 0], rows[~held & first, 0]) & np.isin(rows[:, 1], rows[~held & first, 1])])

    def timed(call):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = call()
        torch.cuda.synchronize()
        return out, time.perf_counter() - t

    def accuracy(model):
        model.predict(test)
        return float(model.score(silent=True)["stats"]["accuracy"])

    out = {}
    # 1. one log-likelihood evaluation against one EM step, all S runs
    train = rows[~held]
    e = Engine(train, int(train[:, 0].max()) + 1, int(train[:, 1].max()) + 1, R, K, L)
    pg = np.random.default_rng(5)
    th, et, pr = pg.random((S, e.U, K)), pg.random((S, e.I, L)), pg.random((S, K, L, R))
    e.set_params(th / th.sum(-1, keepdims=True), et / et.sum(-1, keepdims=True), pr / pr.sum(-1, keepdims=True))
    lik_ms = event_ms(e.loglik_device, 20)
    step_ms = event_ms(lambda: e.run(1), 20)
    out["loglik_vs_step"] = {"loglik_ms": round(lik_ms, 4), "em_step_ms": round(step_ms, 4),
                             "ratio": round(lik_ms / step_ms, 4), "ratings": e.N}
    del e

    warm = MMSBM(K, L, iterations=20, sampling=S, seed=0)          # module load, allocator, both loops
    warm.fit(part.iloc[:200_000], silent=True)
    warm.fit(part.iloc[:200_000], silent=True, tol=1e-4)

    # 2. fixed 400 against tol
    def fit_row(tol):
        m = MMSBM(K, L, iterations=ITERS, sampling=S, seed=1)
        _, wall = timed(lambda: m.fit(part, silent=True, tol=tol))
        row = {"tol": tol, "wall_s": round(wall, 3), **stages(m.timings), "accuracy": accuracy(m)}
        if tol is not None:
            row["stop_iterations"] = [r["iterations"] for r in m.results]
            row["converged"] = [r["converged"] for r in m.results]
        return m, row

    base, out["fit_400"] = fit_row(None)
    for tol in TOLS:
        out[f"fit_tol_{tol:g}"] = fit_row(tol)[1]

    # 3. refit on 100 %: fixed 25 / 50 / 100 against tol, each from a copy of the same fitted model
    snap = ([{k: np.array(v, copy=True) for k, v in r.items()} for r in base.results],
            [dict(d) for d in base.data_handler.return_dicts()], base.p, base.m)

    def refit_row(iters, tol):
        base.results = [{k: np.array(v, copy=True) for k, v in r.items()} for r in snap[0]]
        dh = base.data_handler
        dh.obs_dict, dh.items_dict, dh.ratings_dict = (dict(d) for d in snap[1])
        base.p, base.m = snap[2], snap[3]
        _, wall = timed(lambda: base.refit(full, iterations=iters, tol=tol))
        row = {"iterations": iters, "tol": tol, "wall_s": round(wall, 3), **stages(base.timings),
               "accuracy": accuracy(base)}
        if tol is not None:
            row["stop_iterations"] = [r["iterations"] for r in base.results]
        return row

    for iters in (25, 50, 100):
        out[f"refit_{iters}"] = refit_row(iters, None)
    for tol in TOLS:
        out[f"refit_tol_{tol:g}"] = refit_row(ITERS, tol)

    # 4. cost of the loop per check on the cooperative path (ML-100K shape)
    g2 = np.random.default_rng(6)
    nu2, ni2, n2, k2 = 943, 1682, 100_000, 10
    small = np.stack([g2.integers(0, nu2, n2), g2.integers(0, ni2, n2), g2.integers(0, R, n2)], axis=1)
    small[:nu2, 0] = np.arange(nu2)
    small[:ni2, 1] = np.arange(ni2)
    e2 = Engine(small, nu2, ni2, R, k2, k2)
    p0 = (g2.random((1, nu2, k2)), g2.random((1, ni2, k2)), g2.random((1, k2, k2, R)))
    p0 = tuple(x / x.sum(-1, keepdims=True) for x in p0)

    def plain():
        e2.set_params(*p0)
        e2.run(ITERS)

    def conv():
        e2.set_params(*p0)
        e2.run_converge(ITERS, 0.0, 10)

    plain(), conv()
    tp = min(timed(plain)[1] for _ in range(5))
    tc = min(timed(conv)[1] for _ in range(5))
    out["ml100k_coop_check_cost"] = {"run_400_s": round(tp, 5), "run_converge_400_tol0_s": round(tc, 5),
                                     "checks": ITERS // 10, "us_per_check": round((tc - tp) / (ITERS // 10) * 1e6, 2),
                                     "note": "best of 5, parameter upload included in both"}

    res = {"workload": "ml20m_shape_planted_converge", "gpu": name, "power_limit": limit, "users": nu, "items": ni,
           "ratings_90pct": len(part), "ratings_100pct": len(full), "test_ratings": len(test),
           "K": K, "L": L, "R": R, "S": S, **out}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
