"""Multi-GPU checks of MMSBM.refit, launched by tests/test_refit_multi_gpu.py under torchrun (one
rank per GPU).  The refit set drops some known ids and adds new ones.
  1. fit + refit with runs sharded over ranks == the same fit + refit in one process (bit-identical);
  2. fit + refit with shard="ratings" == the one-process fit + refit within the tolerance of the
     rating-sharded fit in tests/multi_gpu_check.py (1e-9 per element, likelihood 1e-8)."""
import os
import sys

import numpy as np
import pandas as pd
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    os.chdir(os.environ.get("MMSBM_TMP", "/tmp"))
    import mmsbm_b200.mmsbm as mmsbm_mod
    from mmsbm_b200 import MMSBM
    from tests.util import rel_err

    g = np.random.default_rng(5)
    n = 30000
    df = pd.DataFrame({"users": g.integers(0, 400, n), "items": g.integers(0, 250, n),
                       "ratings": g.integers(1, 6, n)})
    old = df.iloc[:24000]
    new = pd.DataFrame({"users": g.integers(380, 420, 600), "items": g.integers(230, 270, 600),
                        "ratings": g.integers(1, 6, 600)})
    data = pd.concat([df[(df["users"] != 7) & (df["items"] != 11)], new])     # user 7, item 11: no rows
    S, K, L, it = 4, 6, 5, 6

    # reference: the same calls with the model believing it runs alone (the runs are independent, so
    # every rank computes all of them; gather_runs then merges identical results)
    solo_info = mmsbm_mod.dist_info
    mmsbm_mod.dist_info = lambda: (0, 1)
    try:
        solo = MMSBM(K, L, iterations=it, sampling=S, seed=3)
        solo.fit(old, silent=True)
        want_added = solo.refit(data, iterations=it, seed=2)
    finally:
        mmsbm_mod.dist_info = solo_info
    want = solo.results
    assert want_added["users"] and want_added["items"]

    a = MMSBM(K, L, iterations=it, sampling=S, seed=3)
    a.fit(old, silent=True)
    assert a.refit(data, iterations=it, seed=2) == want_added
    for s in range(S):
        for key in ("theta", "eta", "pr"):
            assert np.array_equal(a.results[s][key], want[s][key]), (s, key)
        assert a.results[s]["likelihood"] == want[s]["likelihood"]
    test = data.iloc[:500]
    assert np.array_equal(a.predict(test), solo.predict(test))

    b = MMSBM(K, L, iterations=it, sampling=S, seed=3, shard="ratings")
    b.fit(old, silent=True)
    assert b.refit(data, iterations=it, seed=2) == want_added
    worst = 0.0
    for s in range(S):
        for key in ("theta", "eta", "pr"):
            worst = max(worst, rel_err(b.results[s][key], want[s][key]))
        assert abs(b.results[s]["likelihood"] - want[s]["likelihood"]) <= 1e-8 * abs(want[s]["likelihood"])
        u7, i11 = b.data_handler.obs_dict["7"], b.data_handler.items_dict["11"]
        assert np.array_equal(b.results[s]["theta"][u7], want[s]["theta"][u7])
        assert np.array_equal(b.results[s]["eta"][i11], want[s]["eta"][i11])
    assert worst < 1e-9, worst
    assert rel_err(b.predict(test), solo.predict(test)) < 1e-9
    dist.barrier()
    if dist.get_rank() == 0:
        print(f"refit multi-gpu ok: world={dist.get_world_size()} rating-sharded worst rel err {worst:.2e}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
