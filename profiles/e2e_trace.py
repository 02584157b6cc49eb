import os, sys, time, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from mmsbm_b200 import _lib
U, I, N, K, L, S = bench.WORKLOADS["ml20m"]; R = 5
data = bench.synth_triples(U, I, N)
seeds = np.random.default_rng(1).bit_generator._seed_seq.spawn(S)
th0, et0, pr0 = bench.seeded_inits(data, U, I, K, L, seeds)
lib = _lib.load(True)
def pinned(a):
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory(); return t, t.numpy()
keep = [pinned(a) for a in (data, th0, et0, pr0)]
h = [k[1] for k in keep]
outs = [torch.empty(a.shape, dtype=torch.float64).pin_memory() for a in (th0, et0, pr0)]
lik = torch.empty(S, dtype=torch.float64).pin_memory()
for it in range(3):
    t0 = time.perf_counter()
    _lib.check(lib.mmsbm_host_fit(h[0].ctypes.data, N, U, I, R, K, L, S, 20, h[1].ctypes.data, h[2].ctypes.data, h[3].ctypes.data,
                                  outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(), lik.data_ptr()), "fit")
    print("total", (time.perf_counter() - t0) * 1e3, "ms", file=sys.stderr)
