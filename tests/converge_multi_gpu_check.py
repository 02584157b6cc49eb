"""Multi-GPU check of MMSBM.fit(tol=...) with runs sharded over ranks, launched by
tests/test_converge_multi_gpu.py under torchrun (one rank per GPU): every run stops at the same
iteration and holds the same parameters (within 1e-12) as in a one-process fit."""
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
    S, K, L, it, tol = 4, 6, 5, 200, 1e-6
    solo_info = mmsbm_mod.dist_info
    mmsbm_mod.dist_info = lambda: (0, 1)
    try:
        solo = MMSBM(K, L, iterations=it, sampling=S, seed=3)
        solo.fit(df, silent=True, tol=tol)
    finally:
        mmsbm_mod.dist_info = solo_info
    a = MMSBM(K, L, iterations=it, sampling=S, seed=3)
    a.fit(df, silent=True, tol=tol)
    worst = 0.0
    for s in range(S):
        assert a.results[s]["iterations"] == solo.results[s]["iterations"], s
        assert a.results[s]["converged"] == solo.results[s]["converged"], s
        for key in ("theta", "eta", "pr"):
            worst = max(worst, rel_err(a.results[s][key], solo.results[s][key]))
    assert worst <= 1e-12, worst
    dist.barrier()
    if dist.get_rank() == 0:
        print(f"converge multi-gpu ok: world={dist.get_world_size()} worst rel err {worst:.2e}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
