"""MMSBM.refit at the ML-20M shape: 138 493 users, 26 744 items, about 1.4e7 ratings drawn from a
planted model (K = L = 20, R = 5) with heavy-tailed user degrees (at least 24 ratings per user) and
Zipf-like item popularity; S = 8 runs.

1 % of the ratings are held out for testing.  A model is fitted with 400 iterations on 90 % of the
rest, then refitted on all of it with 25, 50 and 100 iterations (each refit starts from a copy of the
same fitted model); a cold fit on all of it with 400 iterations is the comparison.  For every call
it reports the wall time (host clock, device synchronised) split into encoding and planning,
initial parameters, index build, EM and the rest, and the held-out accuracy of ``predict`` /
``score``; then the card's name and power limit.  The accuracy of the planted parameters on the
same test rows is the ceiling.

    python profiles/scripts/refit_bench.py [--out result.json] [--scale 1.0]
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

U, I, K, L, R, S, ITERS = 138_493, 26_744, 20, 20, 5, 8, 400


def planted_rows(seed, n_users, n_items):
    """int64 [N,3] from a planted MMSBM (sparse Dirichlet theta / eta / pr as in
    tests/fold_in_reference.planted), drawn on the GPU in chunks."""
    import torch
    g = np.random.default_rng(seed)
    theta = g.dirichlet(np.full(K, 0.2), n_users)
    eta = g.dirichlet(np.full(L, 0.2), n_items)
    pr = g.dirichlet(np.full(R, 0.15), (K, L))
    deg = np.minimum((24 * (1 + g.pareto(1.2, n_users))).astype(np.int64), n_items // 3)
    pi = 1.0 / np.arange(1, n_items + 1) ** 0.9
    pi /= pi.sum()
    users = np.repeat(np.arange(n_users), deg)
    items = g.permutation(n_items)[g.choice(n_items, size=len(users), p=pi)]
    dev = torch.device("cuda")
    th, ep = torch.from_numpy(theta).to(dev), torch.from_numpy(np.einsum("il,klr->ikr", eta, pr)).to(dev)
    levels = np.empty(len(users), dtype=np.int64)
    tg = torch.Generator(device=dev).manual_seed(seed)
    for lo in range(0, len(users), 1 << 21):
        u = torch.from_numpy(users[lo:lo + (1 << 21)]).to(dev)
        i = torch.from_numpy(items[lo:lo + (1 << 21)]).to(dev)
        p = torch.einsum("nk,nkr->nr", th[u], ep[i])
        levels[lo:lo + len(u)] = torch.multinomial(p, 1, generator=tg).squeeze(1).cpu().numpy()
    rows = np.stack([users, items, levels], axis=1)
    return rows, (theta, eta, pr)


def planted_accuracy(rows, params):
    """Accuracy of the planted parameters themselves on ``rows``: the ceiling of any fit."""
    theta, eta, pr = params
    best = np.argmax(np.einsum("nk,nl,klr->nr", theta[rows[:, 0]], eta[rows[:, 1]], pr), axis=1)
    return float(np.mean(best == rows[:, 2]))


def stages(timings):
    t = dict(timings)
    out = {"encode_plan_s": t.pop("encode", 0.0) + t.pop("encode_plan", 0.0),
           "init_s": t.pop("init_draws", 0.0),
           "index_build_s": t.pop("rows_h2d_index_build", 0.0),
           "em_s": t.pop("em_iterations", 0.0)}
    out["other_s"] = sum(t.values())
    return {k: round(v, 3) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the users and items (rehearsal)")
    args = ap.parse_args()
    import pandas as pd
    import torch
    from fold_in_bench import card
    from mmsbm_b200 import MMSBM

    name, limit = card()
    nu, ni = max(int(U * args.scale), 50), max(int(I * args.scale), 50)
    rows, params = planted_rows(3, nu, ni)
    g = np.random.default_rng(4)
    held = g.random(len(rows)) < 0.01
    first = g.random(len(rows)) < 0.9

    def frame(r):
        return pd.DataFrame({"users": r[:, 0], "items": r[:, 1], "ratings": r[:, 2] + 1})

    part, full = frame(rows[~held & first]), frame(rows[~held])
    test = frame(rows[held & np.isin(rows[:, 0], rows[~held & first, 0]) & np.isin(rows[:, 1], rows[~held & first, 1])])

    warm = MMSBM(K, L, iterations=20, sampling=S, seed=0)      # module load, allocator, refit path
    warm.fit(part.iloc[:200_000], silent=True)
    warm.refit(part.iloc[:210_000], iterations=5)

    def timed(call):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = call()
        torch.cuda.synchronize()
        return out, time.perf_counter() - t

    def accuracy(model):
        model.predict(test)
        return float(model.score(silent=True)["stats"]["accuracy"])

    base = MMSBM(K, L, iterations=ITERS, sampling=S, seed=1)
    _, wall = timed(lambda: base.fit(part, silent=True))
    out = {"fit_90pct": {"iterations": ITERS, "wall_s": round(wall, 3), **stages(base.timings),
                         "accuracy": accuracy(base)}}
    snap = ([{k: np.array(v, copy=True) for k, v in r.items()} for r in base.results],
            [dict(d) for d in base.data_handler.return_dicts()], base.p, base.m)
    for iters in (25, 50, 100):
        base.results = [{k: np.array(v, copy=True) for k, v in r.items()} for r in snap[0]]
        dh = base.data_handler
        dh.obs_dict, dh.items_dict, dh.ratings_dict = (dict(d) for d in snap[1])
        base.p, base.m = snap[2], snap[3]
        added, wall = timed(lambda: base.refit(full, iterations=iters))
        out[f"refit_{iters}"] = {"iterations": iters, "wall_s": round(wall, 3), **stages(base.timings),
                                 "new_users": len(added["users"]), "new_items": len(added["items"]),
                                 "accuracy": accuracy(base)}
    cold = MMSBM(K, L, iterations=ITERS, sampling=S, seed=1)
    _, wall = timed(lambda: cold.fit(full, silent=True))
    out["cold_fit_100pct"] = {"iterations": ITERS, "wall_s": round(wall, 3), **stages(cold.timings),
                              "accuracy": accuracy(cold)}

    res = {"workload": "ml20m_shape_planted_refit", "gpu": name, "power_limit": limit, "users": nu, "items": ni,
           "ratings_90pct": len(part), "ratings_100pct": len(full), "test_ratings": len(test),
           "planted_accuracy": planted_accuracy(test.to_numpy() - [0, 0, 1], params),
           "K": K, "L": L, "R": R, "S": S, **out}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
