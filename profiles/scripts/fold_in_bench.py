"""Fold-in at the ML-20M shape: 10 % of the users are new (about 2e6 ratings), K = L = 20, R = 5,
S = 8 runs, 400 iterations, on fixed random parameters of the known ids.

Reports the device time of Engine.fold_in (CUDA events, after a warm-up call), the per-iteration
cost and rating-updates/s from the difference of a 400- and a 1-iteration call, the wall time of
MMSBM.fold_in on a DataFrame of the same rows (model restored from a saved file), the card's name
and power limit, and checks 100 sampled new users against the CPU reference after one iteration.

    python profiles/scripts/fold_in_bench.py [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

U_ALL, I, K, L, R, S, ITERS = 138_493, 26_744, 20, 20, 5, 8, 400


def workload(seed=0):
    """Known users, new-user rows [n,3] (new ids 0..n_new-1), heavy-tailed degrees like ML-20M's
    (at least 32 ratings per user, about 2e6 in all) and Zipf-like item popularity."""
    g = np.random.default_rng(seed)
    n_new = U_ALL // 10
    deg = np.minimum((32 * (1 + g.pareto(1.2, n_new))).astype(np.int64), 9254)
    pi = 1.0 / np.arange(1, I + 1) ** 0.9
    pi /= pi.sum()
    users = np.repeat(np.arange(n_new), deg)
    items = g.choice(I, size=len(users), p=pi)
    levels = g.integers(0, R, len(users))
    return U_ALL - n_new, n_new, deg, np.stack([users, items, levels], axis=1).astype(np.int64)


def card():
    import torch
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True,
                               timeout=60).stdout.strip()
    except Exception as e:                                  # report it, the timings still stand
        limit = f"unavailable ({e})"
    return torch.cuda.get_device_name(), limit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from mmsbm_b200 import MMSBM
    from mmsbm_b200.engine import Engine
    from tests import fold_in_reference as fref
    from tests.util import rel_err

    name, limit = card()
    Uk, n_new, deg, rows = workload()
    n = len(rows)
    g = np.random.default_rng(1)
    theta = g.random((S, Uk, K)); theta /= theta.sum(-1, keepdims=True)
    eta = g.random((S, I, L)); eta /= eta.sum(-1, keepdims=True)
    pr = g.random((S, K, L, R)); pr /= pr.sum(-1, keepdims=True)
    init = g.random((S, n_new, K)) / deg[None, :, None]
    eng = Engine.for_prediction(Uk, I, R, K, L)
    eng.set_params(theta, eta, pr)

    def timed(iters, reps):
        ms = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = eng.fold_in(0, rows, init, iters)
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return out, float(np.median(ms)), ms

    timed(ITERS, 1)                                         # warm-up: module load, allocator
    one, ms1, _ = timed(1, 3)
    _, ms400, all400 = timed(ITERS, 3)
    per_iter = (ms400 - ms1) / (ITERS - 1)
    updates = n * S / (per_iter * 1e-3)

    # 100 sampled new users against the CPU reference after one iteration
    ids = np.sort(g.choice(n_new, 100, replace=False))
    sub = rows[np.isin(rows[:, 0], ids)].copy()
    sub[:, 0] = np.searchsorted(ids, sub[:, 0])
    worst = 0.0
    for s in range(S):
        want = fref.fold_in(sub, init[s][ids], eta[s], pr[s], 1, side=0)
        worst = max(worst, rel_err(one[s][ids], want))

    # MMSBM.fold_in on a DataFrame of the same rows, model restored from a file
    import pandas as pd
    users = sorted(str(u) for u in range(Uk))
    items = sorted(str(i) for i in range(I))
    dicts = [[(s, k) for k, s in enumerate(users)], [(s, k) for k, s in enumerate(items)],
             [(str(r + 1), r) for r in range(R)]]
    config = {"user_groups": K, "item_groups": L, "iterations": ITERS, "sampling": S, "debug": False,
              "backend": "auto", "shard": "runs"}
    inv_items = np.array([int(s) for s in items])
    frame = pd.DataFrame({"users": rows[:, 0] + 10 ** 6, "items": inv_items[rows[:, 1]], "ratings": rows[:, 2] + 1})
    def restored():
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "model.npz")
            with open(path, "wb") as fh:
                np.savez(fh, format_version=np.int64(1), config=np.array(json.dumps(config)),
                         dicts=np.array(json.dumps(dicts)), theta=theta, eta=eta, pr=pr,
                         likelihood=np.zeros(S))
            return MMSBM.load(path)

    restored().fold_in(frame.iloc[:50_000])                 # warm-up of the API path
    model = restored()
    torch.cuda.synchronize()
    t = time.perf_counter()
    added = model.fold_in(frame)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t
    assert len(added["users"]) == n_new

    res = {"workload": "ml20m_shape_fold_in_10pct_users", "gpu": name, "power_limit": limit,
           "new_users": n_new, "ratings": n, "max_degree": int(deg.max()), "K": K, "L": L, "R": R, "S": S,
           "iterations": ITERS, "engine_fold_in_ms": round(ms400, 3),
           "engine_fold_in_ms_all": [round(x, 3) for x in all400], "engine_fold_in_1_iter_ms": round(ms1, 3),
           "ms_per_iteration": round(per_iter, 5), "rating_updates_per_s": float("%.4g" % updates),
           "api_fold_in_wall_s": round(wall, 3), "check_100_ids_max_rel_err": worst}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    assert worst < 1e-10, worst


if __name__ == "__main__":
    main()
