#!/usr/bin/env python
"""Benchmark of the EM hot path on synthetic ratings of a BASELINE.json shape.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload ml20m|ml1m|ml100k|netflix|ml1m_cv] [--iters-per-step T]

metric = rating-updates/s = ratings x EM iterations x runs / time.  A *step* is one fit-sized
pass of the hot path: T EM iterations (default 400, the reference's default ``iterations``;
BASELINE.json's ML-20M config names none) of all S runs (``sampling``, S in TOTAL whatever the
number of GPUs: strong scaling) over the same synthetic ratings.

N = 1
  value        K steps on data and parameters resident in HBM (Engine.run -> mmsbm_em_run), CUDA
               events on the launching stream.
  e2e          the same T iterations through the host-pointer C ABI (mmsbm_host_fit, what the
               reference-side ctypes stub binds): H2D of the int64 [N,3] rows and theta0/eta0/pr0
               from pinned memory, index build, EM loop, likelihood, D2H of the fitted
               parameters -- all inside the timed region.  ``verify`` checks its outputs against
               the oracle (one more iteration of a user and an item; likelihood of a row sample).
  api_e2e      one ``mmsbm_b200.MMSBM(K, L, T, S, seed=1).fit(DataFrame)`` + ``predict`` + ``score``
               through the public API (what the reference's benchmark_mmsbm.py:59-73 times), with
               its stage split.
  roofline     ``hbm``: DRAM bytes of all kernels of one iteration (ncu record named in the line)
               / the iteration time measured here, against MEASURED_PEAKS.json; ``gather``: the
               row bytes the two segment passes gather (served by L2) / their CUDA-event time,
               against the measured pure-gather floor (profiles/peaks.json) -- the binding
               resource; ``alg``: SURVEY.md 8(d)'s algorithmic bytes, for continuity.
  cpu_baseline the reference's own numba / numpy kernels (baseline/_ref, installed by
               oracle/install_reference.py; the oracle port when that directory is absent) on a
               bounded row sample, on the box's host cores.

N > 1 (torchrun, one rank per GPU; ``scaling: strong``)
  Two ways to put S runs on N GPUs are timed back to back and the faster one is the ``value``:
  ``runs`` (S/N independent runs per GPU over a replica of the ratings, no collective) and
  ``sharded`` (all S runs on every GPU, ratings split by user range x item range:
  mmsbm_em_run_sharded -- copy-engine exchange of parameter rows over NVLink + one NCCL
  all-reduce of n_pr per iteration).  ``netflix_ratings_sharded`` in the same line times the
  Netflix-shaped single run (BASELINE.json configs[4]) the sharded way and compares its
  likelihood with the one-GPU loop run on rank 0.

``--impl reference`` times the reference's CPU implementation of the path (baseline/_ref: its
``kernels_numba.update_coefficients`` + ``ExpectationMaximization`` normalisations, numpy when
numba is missing), one process per run like its spawn pool (src/mmsbm.py:182-185), on a bounded
row sample; rank 0 only.

``--dump-outputs DIR`` (N = 1) writes what the timed ``Engine.run`` loop left after its last step,
as a caller reads it back with ``Engine.get_params``: DIR/theta.npy [S,U,K], DIR/eta.npy [S,I,L]
and DIR/pr.npy [S,K,L,R], float64.  An array above a third of 64 MB keeps a fixed sample of its
id axis (rows drawn with seed 0, sorted; the same rows for the same shape), so that the outputs of
two builds on the same arguments can be compared element for element.  The ml1m_cv workload
writes DIR/cv_accuracies.npy.

The benchmark writes nothing into the source tree: it runs in a temporary working directory (the
MMSBM logger writes mmsbm.log into the working directory) and writes no bytecode.
"""
import argparse
import contextlib
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
REF_DIR = os.path.join(ROOT, "baseline", "_ref")

WORKLOADS = {
    # name: (U, I, N, K, L, S)   R = 5 everywhere (BASELINE.json configs)
    "ml100k": (943, 1682, 100_000, 10, 10, 1),
    "ml1m": (6040, 3706, 1_000_000, 10, 10, 8),
    "ml1m_cv": (6040, 3706, 1_000_000, 10, 10, 4),
    "ml20m": (138_000, 27_000, 20_000_000, 20, 20, 8),
    "netflix": (480_000, 17_700, 100_000_000, 32, 32, 1),
}
R = 5
FALLBACK_HBM_GBS = 6650.0   # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def _zipf_ids(g, n_ids, size):
    """Heavy-tailed ids: P(id = k) ~ 1/(k+1) (Zipf exponent 1), by inverse-CDF sampling."""
    cdf = np.cumsum(1.0 / np.arange(1, n_ids + 1))
    cdf /= cdf[-1]
    return np.searchsorted(cdf, g.random(size), side="left").astype(np.int64)


def synth_triples(U, I, N, seed=0, ids="uniform"):
    """Uniform ids like the reference's benchmark_mmsbm.py:23-31, or Zipf-like heavy-tailed ids
    (SURVEY.md 8d); every id forced to appear."""
    g = np.random.default_rng(seed)
    data = np.empty((N, 3), dtype=np.int64)
    if ids == "zipf":
        data[:, 0] = _zipf_ids(g, U, N)
        data[:, 1] = _zipf_ids(g, I, N)
    else:
        data[:, 0] = g.integers(0, U, N)
        data[:, 1] = g.integers(0, I, N)
    data[:, 2] = g.integers(0, R, N)
    data[:U, 0] = np.arange(U)
    data[:I, 1] = np.arange(I)
    data[:R, 2] = np.arange(R)
    return data


def seeded_inits(data, U, I, K, L, seeds):
    """theta0/eta0/pr0 exactly as src/mmsbm.py:224-233 for each SeedSequence child."""
    du = np.maximum(np.bincount(data[:, 0], minlength=U), 1)[:, None]
    di = np.maximum(np.bincount(data[:, 1], minlength=I), 1)[:, None]
    th, et, pr = [], [], []
    for s in seeds:
        g = np.random.default_rng(s)
        th.append(g.random((U, K)) / du)
        et.append(g.random((I, L)) / di)
        p = g.random((K, L, R))
        pr.append(p / p.sum(axis=2, keepdims=True))
    return np.stack(th), np.stack(et), np.stack(pr)


def child_seeds(n):
    return np.random.default_rng(1).bit_generator._seed_seq.spawn(n)


def b_alg(U, I, N, K, L, S):
    """Algorithmic bytes per rating-update, SURVEY.md section 8(d)."""
    return 8.0 * (K + L) + 16.0 / S + 16.0 * (K * U + L * I) / N


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays, id_axis=1):
    """Write each array as out_dir/<name>.npy (float64).  One larger than DUMP_BYTES / len(arrays)
    keeps a fixed, seeded sample of its ``id_axis`` so that all files together stay within
    DUMP_BYTES."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096                  # room for the .npy header
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.nbytes > share:
            per_row = a.nbytes // a.shape[id_axis]
            rows = np.sort(np.random.default_rng(0).choice(a.shape[id_axis], share // per_row, replace=False))
            a = np.take(a, rows, axis=id_axis)
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def _json(path):
    try:
        with open(path) as fh:
            return json.load(fh)
    except Exception:
        return None


def hbm_peak():
    d = _json(os.path.join(ROOT, "MEASURED_PEAKS.json"))
    if d and "hbm_gbs" in d:
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json"
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- CPU arms
def reference_available():
    return os.path.exists(os.path.join(REF_DIR, "kernels_numpy.py"))


def _reference_step(backend, data, K, L):
    """One EM iteration of ONE run with the reference's own code (baseline/_ref): its kernel
    module's update_coefficients + its ExpectationMaximization normalisations
    (src/mmsbm.py:244-250).  Returns (step function, backend actually used, kind)."""
    if reference_available():
        if REF_DIR not in sys.path:
            sys.path.insert(0, REF_DIR)
        import expectation_maximization as ref_em     # the reference's module (flat py_modules)
        du = np.maximum(np.bincount(data[:, 0]), 1)
        di = np.maximum(np.bincount(data[:, 1]), 1)
        factors = {"user": np.repeat(du[:, None], K, axis=1), "item": np.repeat(di[:, None], L, axis=1)}
        dims = {"n_samples": len(data), "n_user_groups": K, "n_item_groups": L, "n_ratings": R}
        em = ref_em.ExpectationMaximization(dims, None, None, None, factors, backend=backend)

        def step(th, et, pr):
            nt, ne, npr = em.update_coefficients(data, th, et, pr)
            return em.normalize_with_d(nt, "user"), em.normalize_with_d(ne, "item"), em.normalize_with_self(npr)
        return step, em._backend, "reference"
    from oracle import mmsbm_oracle as orc
    f = orc.degree_factors(data, K, L)
    if backend in ("auto", "numba"):
        try:
            from oracle import mmsbm_oracle_numba as onb
            return (lambda th, et, pr: onb.em_iteration(data, th, et, pr, *f)), "numba", "port"
        except ImportError:
            pass
    return (lambda th, et, pr: orc.em_iteration(data, th, et, pr, *f, chunk=50_000)), "numpy", "port"


def cpu_baseline(U, I, K, L, n_rows, backend, repeats=3):
    """One run, one EM iteration on an n_rows sample, best of ``repeats``; all host threads the
    backend uses by itself (numba: its parallel omega phase; numpy: one)."""
    data = synth_triples(U, I, max(n_rows, max(U, I)), seed=0)
    try:
        step, used, kind = _reference_step(backend, data, K, L)
    except ImportError as e:
        return {"unavailable": str(e)}
    th, et, pr = (a[0] for a in seeded_inits(data, U, I, K, L, [1]))
    step(th, et, pr)                                           # numba JIT outside the timing
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        step(th, et, pr)
        best = min(best, time.perf_counter() - t0)
    cores = 1
    if used == "numba":
        import numba
        cores = int(numba.get_num_threads())
    src = ("baseline/_ref kernels_%s.update_coefficients + ExpectationMaximization normalisations "
           "(the unmodified reference)" % used) if kind == "reference" else \
        ("oracle port of the reference's %s backend (baseline/_ref absent)" % used)
    return {"value": data.shape[0] / best, "unit": "rating-updates/s", "cores": cores, "kind": kind,
            "backend": used,
            "sample": f"{data.shape[0]} rows of the same U/I/K/L, 1 run, 1 EM iteration incl. the three "
                      f"normalisations, best of {repeats}, JIT excluded; {src}"}


_W = {}


def _ref_worker_init(U, I, K, L, n_rows, backend, threads):
    data = synth_triples(U, I, max(n_rows, max(U, I)), seed=0)
    if backend != "numpy":
        try:
            import numba
            numba.set_num_threads(max(1, min(threads, numba.config.NUMBA_NUM_THREADS)))
        except ImportError:
            backend = "numpy"
    step, used, kind = _reference_step(backend, data, K, L)
    _W.update(data=data, step=step, shape=(U, I, K, L), used=used, kind=kind)
    th, et, pr = (a[0] for a in seeded_inits(data, U, I, K, L, [0]))
    step(th, et, pr)                                           # JIT compile in the initializer


def _ref_worker_step(args):
    seed, iters = args
    U, I, K, L = _W["shape"]
    th, et, pr = (a[0] for a in seeded_inits(_W["data"], U, I, K, L, [seed]))
    for _ in range(iters):
        th, et, pr = _W["step"](th, et, pr)
    return float(th.sum()), _W["used"], _W["kind"]


def run_reference_arm(args, shape):
    """The reference's CPU implementation of the path, one process per run like its spawn pool
    (src/mmsbm.py:182-185), on a bounded row sample."""
    import multiprocessing as mp
    if int(os.environ.get("RANK", "0")) != 0:
        return
    U, I, N, K, L, S = shape
    n_rows = max(args.cpu_rows, max(U, I))
    cores = os.cpu_count() or 1
    procs = min(S, cores)
    iters = 1
    backend = args.cpu_backend
    threads = max(1, cores // procs)
    ctx = mp.get_context("spawn")                 # the reference's own start method (src/mmsbm.py:182)
    with ctx.Pool(processes=procs, initializer=_ref_worker_init,
                  initargs=(U, I, K, L, n_rows, backend, threads)) as pool:
        for _ in range(args.warmup):
            pool.map(_ref_worker_step, [(s, iters) for s in range(S)])
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = pool.map(_ref_worker_step, [(s, iters) for s in range(S)])
        dt = time.perf_counter() - t0
    used, kind = out[0][1], out[0][2]
    if used != "numba":
        threads = 1
    value = n_rows * iters * S * args.steps / dt
    what = ("the unmodified reference from baseline/_ref (kernels_%s.update_coefficients + its "
            "ExpectationMaximization normalisations)" % used) if kind == "reference" else \
        ("oracle port of the reference's %s backend (baseline/_ref absent)" % used)
    sample = (f"{n_rows} rows of the {args.workload} shape (same U/I/K/L/R), {S} runs x {iters} EM iteration per "
              f"step, one process per run ({procs} processes x {threads} thread(s), {cores} host cores), "
              f"{what}, init included")
    line = {
        "impl": "reference", "metric": "rating-updates/sec", "value": value, "unit": "rating-updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "users": U, "items": I, "ratings": N, "K": K, "L": L, "R": R,
                   "sampling": S, "cpu_sample_rows": n_rows},
        "cpu_baseline": {"value": value, "unit": "rating-updates/s", "cores": procs * threads, "kind": kind,
                         "backend": used, "sample": sample},
        "e2e": {"value": value, "unit": "rating-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm helpers
class Ctx:
    """torch / process-group plumbing of one rank."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the b200 arm has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, warmup):
        """W untimed calls, then exactly K calls between barrier + synchronize on both sides, CUDA
        events on the current stream, max over ranks.  Returns ms for the K calls."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def kernel_times(eng, lib, _lib, shape, reps=5):
    """Device ms of the stages of one iteration (CUDA events inside the library)."""
    U, I, N, K, L, S = shape
    ms7 = (ctypes.c_float * 7)()
    acc = np.zeros(7)
    for _ in range(reps):
        b = eng._alt
        _lib.check(lib.mmsbm_em_step_profiled(
            *eng._graph_args(), eng.N, U, I, R, K, L, S, eng.theta.data_ptr(), eng.eta.data_ptr(),
            eng.pr.data_ptr(), b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr(), 0,
            eng._ws.data_ptr(), eng._ws_bytes, eng._stream(), ctypes.addressof(ms7)), "em_step_profiled")
        acc += np.array(list(ms7))
        eng.swap()
    k = acc / reps
    return {"p_tables_w": float(k[0]), "by_user": float(k[1]), "n_users": float(k[2]), "by_item": float(k[3]),
            "n_items": float(k[4]), "pr": float(k[5] + k[6])}


def roofline_block(workload, shape, k_ms, ms_per_iteration, use_record=True):
    """See the module docstring.  Every fraction is (measured bytes) / (measured time) / (measured
    peak); the ncu record and the peaks file are named so that each can be recomputed."""
    U, I, N, K, L, S = shape
    ldk, ldl = 4 * ((K + 3) // 4), 4 * ((L + 3) // 4)
    peak, peak_src = hbm_peak()
    seg_ms = k_ms["by_user"] + k_ms["by_item"]
    rec = (_json(os.path.join(ROOT, "profiles", "ncu_records.json")) or {}).get(workload) if use_record else None
    peaks = _json(os.path.join(ROOT, "profiles", "peaks.json")) or {}
    out = {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None,
           "peak_source": peak_src, "kernel": "segment_pass_kernel (by-user + by-item launches of one iteration)",
           "kernel_ms": k_ms, "share_of_iteration": seg_ms / sum(k_ms.values())}
    if rec:
        dram = float(rec["dram_bytes_per_iteration"])
        out["achieved"] = dram / (ms_per_iteration * 1e-3) / 1e9
        out["frac"] = out["achieved"] / peak
        out["traffic"] = float(rec.get("segment_pass_dram_bytes", dram))
        out["ncu_record"] = rec.get("source")
        out["fp64_pipe_pct"] = rec.get("fp64_pipe_pct")
        out["lsu_pipe_pct"] = rec.get("lsu_pipe_pct")
        out["l2_hit_pct"] = rec.get("l2_hit_pct")
    gather_bytes = float(N) * S * 8.0 * (ldl + ldk)          # neighbour rows the two passes read (L1 <- L2)
    g_peak = peaks.get("gather_gbs")
    out["gather"] = {"bytes_per_iteration": gather_bytes, "achieved_gbs": gather_bytes / (seg_ms * 1e-3) / 1e9,
                     "peak_gbs": g_peak, "frac": (gather_bytes / (seg_ms * 1e-3) / 1e9 / g_peak) if g_peak else None,
                     "peak_source": peaks.get("gather_source")}
    out["binding_resource"] = ("L1/LSU data pipe of the row gathers (L2-served: the tables fit the 126 MB L2); "
                               "HBM moves only `traffic`")
    alg = b_alg(U, I, N, K, L, S)
    out["alg"] = {"bytes_per_update": alg, "gbs": alg * N * S / (ms_per_iteration * 1e-3) / 1e9,
                  "note": "SURVEY.md 8(d) counts every gathered row as memory traffic; most of it never "
                          "reaches HBM, so this is not a fraction of the HBM peak"}
    return out


def verify_outputs(data, shape, th, et, pr, lik, T):
    """Checker leg (oracle = test infrastructure): holds the e2e outputs to the oracle.
      * one MORE iteration from them: theta row of a user and eta row of an item, GPU vs the oracle
        restricted to that id's ratings (an id's new row depends on its own ratings only);
      * the likelihood of a bounded row sample under the fitted parameters, GPU vs oracle."""
    from mmsbm_b200.engine import Engine
    from oracle import mmsbm_oracle as orc
    U, I, N, K, L, S = shape
    eng = Engine(data, U, I, R, K, L)
    eng.set_params(th, et, pr)
    lik2 = eng.likelihood()
    eng.run(1)
    th1, et1, _ = eng.get_params()
    u, i = int(U // 3), int(I // 2)
    rows_u, rows_i = data[data[:, 0] == u], data[data[:, 1] == i]
    nt, _, _ = orc.em_sums(rows_u, th[0], et[0], pr[0])
    _, ne, _ = orc.em_sums(rows_i, th[0], et[0], pr[0])
    want_u, want_i = nt[u] / max(len(rows_u), 1), ne[i] / max(len(rows_i), 1)
    rel = lambda a, b: float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))
    n_s = min(N, 100_000)
    sample = data[:n_s]
    e2 = Engine(sample, U, I, R, K, L)
    e2.set_params(th[:1], et[:1], pr[:1])
    got = float(e2.likelihood()[0])
    want = sum(orc.likelihood(sample[lo:lo + 20_000], th[0], et[0], pr[0]) for lo in range(0, n_s, 20_000))
    return {"after_iterations": T, "user_row_rel_err": rel(th1[0][u], want_u), "item_row_rel_err": rel(et1[0][i], want_i),
            "likelihood_sample_rows": n_s, "likelihood_sample_rel_err": abs(got - want) / abs(want),
            "likelihood_recomputed_rel_diff": float(np.max(np.abs(lik2 - lik) / np.abs(lik))),
            "tolerances": {"rows": 1e-10, "likelihood": 1e-8}}


def api_e2e(data, shape, T):
    """fit + predict + score through the public API on a DataFrame, wall clock, with the stage
    split MMSBM records (benchmark_mmsbm.py:59-73 times the same two calls)."""
    import pandas as pd
    import torch
    from mmsbm_b200 import MMSBM
    U, I, N, K, L, S = shape
    df = pd.DataFrame({"users": data[:, 0], "items": data[:, 1], "ratings": data[:, 2] + 1})
    test = df.iloc[:200_000]
    m = MMSBM(K, L, iterations=T, sampling=S, seed=1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.fit(df, silent=True)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    m.predict(test)
    sc = m.score(silent=True)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    return {"value": float(N) * T * S / (t1 - t0), "unit": "rating-updates/s", "fit_s": t1 - t0,
            "predict_score_s": t2 - t1, "stages_s": getattr(m, "timings", None),
            "api": f"mmsbm_b200.MMSBM({K}, {L}, iterations={T}, sampling={S}, seed=1).fit(DataFrame of {N} rows) "
                   f"then predict(200000 rows) + score()",
            "accuracy": float(sc["stats"]["accuracy"]), "likelihood": float(sc["stats"]["likelihood"])}


# ----------------------------------------------------------------------------- GPU arm, N = 1
def run_single(args, shape, cx):
    torch = cx.torch
    from mmsbm_b200 import _lib
    from mmsbm_b200.engine import Engine
    U, I, N, K, L, S = shape
    T = args.iters_per_step
    lib = _lib.load(require_device=True)

    t0 = time.perf_counter()
    data = synth_triples(U, I, N, seed=0, ids=args.ids)
    th0, et0, pr0 = seeded_inits(data, U, I, K, L, child_seeds(S))
    gen_s = time.perf_counter() - t0

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng = Engine(data, U, I, R, K, L)
    torch.cuda.synchronize()
    build_ms = (time.perf_counter() - t0) * 1e3
    eng.set_params(th0, et0, pr0)

    clocks = ClockSampler(cx.local_rank)
    try:
        for _ in range(args.warmup):
            eng.run(T)
        cx.barrier()
        launches1 = _lib.launch_count()
        ms = cx.timed(lambda: eng.run(T), args.steps, 0)
        launches = _lib.launch_count() - launches1
    finally:
        clk = clocks.stop()
    if args.dump_outputs:                       # before kernel_times, which steps the engine further
        th, et, pr = eng.get_params()
        dump_outputs(args.dump_outputs, {"theta": th, "eta": et, "pr": pr})
        del th, et, pr
    value = float(N) * T * S * args.steps / (ms * 1e-3)
    ms_it = ms / args.steps / T

    k_ms = kernel_times(eng, lib, _lib, shape)
    cooperative = launches == args.steps        # one launch per fit: the small-problem kernel (em_small.cu)
    roofline = roofline_block(args.workload, shape, k_ms, ms_it, use_record=not cooperative)
    if cooperative:
        roofline["kernel"] = ("em_small_kernel: the whole fit is ONE cooperative launch (two grid barriers per "
                              "iteration); latency-bound, no bandwidth fraction applies. kernel_ms / gather are the "
                              "stages of the multi-kernel step (mmsbm_em_step), for reference only")
        roofline["binding_resource"] = "latency of the dependent chain inside an iteration (grid barriers, L2 round trips)"

    # ---- end to end through the host-pointer C ABI ----
    e2e = verify = None
    if not args.no_e2e:
        def pinned(a):
            t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
            return t, t.numpy()
        keep = [pinned(a) for a in (data, th0, et0, pr0)]
        h_data, h_th, h_et, h_pr = (k[1] for k in keep)
        outs = [torch.empty(a.shape, dtype=torch.float64).pin_memory() for a in (th0, et0, pr0)]
        lik = torch.empty(S, dtype=torch.float64).pin_memory()

        def fit_once():
            _lib.check(lib.mmsbm_host_fit(
                h_data.ctypes.data, N, U, I, R, K, L, S, T, h_th.ctypes.data, h_et.ctypes.data, h_pr.ctypes.data,
                outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(), lik.data_ptr()), "host_fit")
        fit_once()
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fit_once()
        cx.barrier()
        dt = time.perf_counter() - t0
        h2d = int(h_data.nbytes + h_th.nbytes + h_et.nbytes + h_pr.nbytes)
        d2h = int(sum(o.numel() * 8 for o in outs) + S * 8)
        e2e = {"value": float(N) * T * S * args.steps / dt, "unit": "rating-updates/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": dt / args.steps * 1e3,
               "api": "mmsbm_host_fit (C ABI, host pointers): H2D rows+theta0/eta0/pr0, index build, "
                      f"{T} EM iterations, likelihood, D2H theta/eta/pr/likelihood",
               "likelihood_run0": float(lik[0])}
        if not args.no_verify:
            del eng
            torch.cuda.empty_cache()
            verify = verify_outputs(data, shape, outs[0].numpy(), outs[1].numpy(), outs[2].numpy(),
                                    lik.numpy().copy(), T)
            e2e["verify"] = verify

    api = None
    if not args.no_api_e2e:
        torch.cuda.empty_cache()
        api = api_e2e(data, shape, T)

    cpu = cpu_np = None
    if not args.no_cpu:
        cpu = cpu_baseline(U, I, K, L, args.cpu_rows, "auto")
        cpu_np = cpu_baseline(U, I, K, L, args.cpu_rows, "numpy", repeats=2)

    line = {
        "metric": "rating-updates/sec", "value": value, "unit": "rating-updates/s",
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": args.workload, "users": U, "items": I, "ratings": N, "K": K, "L": L, "R": R,
                   "sampling": S, "iterations_per_step": T, "ids": f"{args.ids}, seed 0",
                   "init": "reference seeded init, model seed 1",
                   "parallelism": "one GPU, all runs batched in one launch row per run group",
                   "l2": "no explicit flush: one iteration touches the parameters of all runs, the W/G tables "
                         "and both index arrays (~1.5 GB at ml20m, L2 = 126 MB); see DESIGN.md"},
        "roofline": roofline, "cpu_baseline": cpu, "cpu_baseline_numpy": cpu_np, "e2e": e2e, "api_e2e": api,
        "gpu_launches": int(launches), "clocks": clk, "index_build_ms": build_ms, "host_datagen_s": gen_s,
        "ms_per_iteration": ms_it,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm, N > 1
def sharded_record(cx, data, shape, T, steps, warmup, check_single_gpu):
    """One set of S runs sharded over all ranks (ShardedEngine): device time of ``steps`` x T
    iterations, the exchange share, the likelihood -- and, on request, the same iterations on rank
    0's GPU alone for the parity figure."""
    torch = cx.torch
    from mmsbm_b200 import _lib
    from mmsbm_b200.parallel import ShardedEngine
    U, I, N, K, L, S = shape
    th0, et0, pr0 = seeded_inits(data, U, I, K, L, child_seeds(S))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sh = ShardedEngine(data, U, I, R, K, L)
    sh.set_params(th0, et0, pr0)
    cx.barrier()
    setup_s = time.perf_counter() - t0
    l0 = _lib.launch_count()
    ms = cx.timed(lambda: sh.run(T), steps, warmup)
    launches = (_lib.launch_count() - l0) * steps // max(steps + warmup, 1)
    prof = sh.run(min(T, 20) // 2 * 2, prof=True)          # even count: parameters stay in the same buffers
    lik = sh.likelihood()
    total_it = (steps + warmup) * T + min(T, 20) // 2 * 2
    rec = {"value": float(N) * T * S * steps / (ms * 1e-3), "unit": "rating-updates/s",
           "ms_per_iteration": ms / steps / T, "ms_per_step": ms / steps,
           "pr_wait_ms_per_iteration": cx.max_over_ranks(prof[1]),
           "stage_ms_when_profiled": dict(zip(("iteration", "wait_n_pr", "p_tables_w", "pass_1", "n_publish_pr_1",
                                               "pass_2", "n_publish_2", "host_issue"), [cx.max_over_ranks(x) for x in prof[:8]])),
           "exchange": "theta / eta rows: copy-engine DMA into every peer's exchange buffer (CUDA IPC over "
                       "NVLink, one copy stream per peer), overlapped with the other pass (the passes alternate "
                       f"their order); one ncclAllReduce of n_pr ({S * K * L * R * 8} bytes) and two one-element "
                       "arrival barriers per iteration on a side stream",
           "exchange_bytes_out_per_iteration": int((sh.Uo * sh.ldk + sh.Io * sh.ldl) * 8 * S * (cx.world - 1)),
           "local_ratings": [int(sh.Nu), int(sh.Ni)], "setup_s": setup_s, "gpu_launches_per_rank": int(launches),
           "likelihood_run0": float(lik[0]), "iterations_run": total_it}
    sh.close()
    del sh
    torch.cuda.empty_cache()
    if check_single_gpu:
        want = None
        if cx.rank == 0:
            from mmsbm_b200.engine import Engine
            e = Engine(data, U, I, R, K, L)
            e.set_params(th0, et0, pr0)
            e.run(total_it)
            want = float(e.likelihood()[0])
            del e
            torch.cuda.empty_cache()
        cx.barrier()
        if cx.rank == 0:
            rec["likelihood_run0_one_gpu"] = want
            rec["likelihood_rel_diff_vs_one_gpu"] = abs(rec["likelihood_run0"] - want) / abs(want)
    return rec


def runs_record(cx, data, shape, T, steps, warmup):
    """S runs in total, S / world independent runs per GPU over a replica of the ratings."""
    torch = cx.torch
    from mmsbm_b200 import _lib
    from mmsbm_b200.engine import Engine
    from mmsbm_b200.parallel import shard_runs
    U, I, N, K, L, S = shape
    mine = shard_runs(S, cx.rank, cx.world)
    eng = None
    if mine:
        seeds = child_seeds(S)
        th0, et0, pr0 = seeded_inits(data, U, I, K, L, [seeds[s] for s in mine])
        eng = Engine(data, U, I, R, K, L)
        eng.set_params(th0, et0, pr0)
    l0 = _lib.launch_count()
    ms = cx.timed((lambda: eng.run(T)) if eng is not None else (lambda: None), steps, warmup)
    launches = (_lib.launch_count() - l0) * steps // max(steps + warmup, 1)
    lik0 = float(eng.likelihood()[0]) if (eng is not None and cx.rank == 0) else None
    del eng
    torch.cuda.empty_cache()
    per = [len(shard_runs(S, r, cx.world)) for r in range(cx.world)]
    return {"value": float(N) * T * S * steps / (ms * 1e-3), "unit": "rating-updates/s",
            "ms_per_iteration": ms / steps / T, "ms_per_step": ms / steps, "runs_per_gpu": per,
            "gpu_launches_per_rank": int(launches), "likelihood_run0": lik0}


def e2e_multi(cx, data, shape, T, mode, steps):
    """End to end from HOST buffers at N > 1, the way `mode` places the runs: H2D of the rows and of the
    initial parameters, index build, T iterations, likelihood and D2H of the results inside the timed
    region (wall clock between barriers, max over ranks)."""
    torch = cx.torch
    from mmsbm_b200 import _lib
    from mmsbm_b200.parallel import ShardedEngine, shard_runs
    U, I, N, K, L, S = shape
    lib = _lib.load(require_device=True)
    seeds = child_seeds(S)
    if mode == "runs":
        mine = shard_runs(S, cx.rank, cx.world)
        Sl = len(mine)
        if Sl:
            th0, et0, pr0 = seeded_inits(data, U, I, K, L, [seeds[s] for s in mine])
            pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
            h = [pin(a) for a in (data, th0, et0, pr0)]
            outs = [torch.empty(a.shape, dtype=torch.float64).pin_memory() for a in (th0, et0, pr0)]
            lik = torch.empty(Sl, dtype=torch.float64).pin_memory()

        def once():
            if Sl:
                _lib.check(lib.mmsbm_host_fit(h[0].data_ptr(), N, U, I, R, K, L, Sl, T, h[1].data_ptr(),
                                              h[2].data_ptr(), h[3].data_ptr(), outs[0].data_ptr(),
                                              outs[1].data_ptr(), outs[2].data_ptr(), lik.data_ptr()), "host_fit")
        h2d = (N * 24 + (U * K + I * L + K * L * R) * 8 * Sl) if Sl else 0
        d2h = ((U * K + I * L + K * L * R + 1) * 8 * Sl) if Sl else 0
        api = "mmsbm_host_fit (C ABI, host pointers) of the rank's runs"
    else:
        th0, et0, pr0 = seeded_inits(data, U, I, K, L, seeds)
        box = {}

        def once():
            sh = ShardedEngine(data, U, I, R, K, L)
            sh.set_params(th0, et0, pr0)
            sh.run(T)
            box["lik"] = sh.likelihood()
            box["params"] = sh.get_params()
            box["bytes"] = ((sh.Nu + sh.Ni) * 24 + (sh.Uo * K + sh.Io * L + K * L * R) * 8 * S,
                            (U * K + I * L + K * L * R + 1) * 8 * S)
            sh.close()
        api = ("ShardedEngine from host arrays: partition + H2D of the rank's rows, two index builds, "
               "H2D of the own parameter rows, mmsbm_em_run_sharded, likelihood, D2H of all parameters")
    once()
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        once()
    cx.barrier()
    dt = cx.max_over_ranks(time.perf_counter() - t0)
    if mode != "runs":
        h2d, d2h = box["bytes"]
    tot = cx.torch.tensor([float(h2d), float(d2h)], dtype=cx.torch.float64, device="cuda")
    cx.dist.all_reduce(tot)
    return {"value": float(N) * T * S * steps / dt, "unit": "rating-updates/s",
            "h2d_bytes_per_step": int(tot[0].item()), "d2h_bytes_per_step": int(tot[1].item()),
            "ms_per_step": dt / steps * 1e3, "steps": steps, "api": api}


def run_multi(args, shape, cx):
    U, I, N, K, L, S = shape
    T = args.iters_per_step
    data = synth_triples(U, I, N, seed=0, ids=args.ids)
    clocks = ClockSampler(cx.local_rank)
    modes = {}
    want = [m for m in ("runs", "sharded") if args.mode in ("best", m)]
    try:
        for mode in want:
            if mode == "runs":
                modes[mode] = runs_record(cx, data, shape, T, args.steps, args.warmup)
            else:
                modes[mode] = sharded_record(cx, data, shape, T, args.steps, args.warmup, check_single_gpu=False)
    finally:
        clk = clocks.stop()
    best = max(modes, key=lambda m: modes[m]["value"])
    b = modes[best]
    e2e = None if args.no_e2e else e2e_multi(cx, data, shape, T, best, min(args.steps, 3))
    del data

    netflix = None
    if args.workload == "ml20m" and not args.no_netflix:
        nU, nI, nN, nK, nL, nS = WORKLOADS["netflix"]
        nf_data = synth_triples(nU, nI, nN, seed=0)
        netflix = sharded_record(cx, nf_data, WORKLOADS["netflix"], args.netflix_iters, 2, 1, check_single_gpu=True)
        if netflix is not None:
            netflix["config"] = {"workload": "netflix", "users": nU, "items": nI, "ratings": nN, "K": nK, "L": nL,
                                 "R": R, "sampling": nS, "iterations_per_step": args.netflix_iters,
                                 "steps": 2, "warmup": 1}
        del nf_data

    if cx.rank == 0:
        par = {"runs": f"{S} runs in total, {b.get('runs_per_gpu')} per GPU over a replica of the ratings, "
                       "no data-path collective",
               "sharded": f"all {S} runs on every GPU, ratings sharded by user range x item range over "
                          f"{cx.world} GPUs (mmsbm_em_run_sharded): copy-engine exchange of theta / eta rows over "
                          "NVLink + one NCCL all-reduce of n_pr per iteration"}[best]
        line = {
            "metric": "rating-updates/sec", "value": b["value"], "unit": "rating-updates/s",
            "n_gpus": cx.world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": b["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": args.workload, "users": U, "items": I, "ratings": N, "K": K, "L": L, "R": R,
                       "sampling": S, "iterations_per_step": T, "ids": f"{args.ids}, seed 0",
                       "init": "reference seeded init, model seed 1", "parallelism": par, "mode": best,
                       "l2": "no explicit flush: an iteration touches parameters, W/G tables and index arrays "
                             "far larger than the 126 MB L2"},
            "modes": modes, "netflix_ratings_sharded": netflix,
            "roofline": None, "cpu_baseline": None,
            "e2e": e2e, "gpu_launches": int(b["gpu_launches_per_rank"]) * cx.world, "clocks": clk,
            "ms_per_iteration": b["ms_per_iteration"],
        }
        print(json.dumps(line), flush=True)


def run_cv(args, shape, cx):
    """BASELINE.json configs[2]: ML-1M-shaped 5-fold cross-validation, K=L=10, sampling=4, the folds x
    runs jobs sharded over the GPUs (20 jobs on 8 GPUs: 3/3/3/3/2/2/2/2).

    The folds are 5 row-wise splits made here (each holds out a fifth of the ratings, ~0.8e6 train
    rows per fold as SURVEY.md section 8 assumes) and fed to ``MMSBM._cv_execute`` -- everything
    ``cv_fit`` does after its fold construction (encoding, index build, the sharded fits, predict,
    score, best fold).  The reference's own fold rule (src/mmsbm.py:415-439, helpers.py:16-24: per
    user up to n_items / folds = 741 held-out rows per fold) holds out EVERY rating of a user with
    fewer than 741 ratings in fold 1, i.e. the whole ML-1M-shaped set at once; ``cv_fit`` reproduces
    that rule faithfully (tests), which leaves nothing to time at this shape."""
    import pandas as pd
    from mmsbm_b200 import MMSBM
    from mmsbm_b200.parallel import shard_jobs
    U, I, N, K, L, S = shape
    T, folds = args.iters_per_step, 5
    data = synth_triples(U, I, N, seed=0, ids=args.ids)
    df = pd.DataFrame({"users": data[:, 0], "items": data[:, 1], "ratings": data[:, 2] + 1})
    fold_of = np.random.default_rng(7).integers(0, folds, N)
    fold_of[:max(U, I)] = -1                                # the rows that introduce every id stay in training
    pairs = [(df[fold_of != f], df[fold_of == f]) for f in range(folds)]
    n_train = [int((fold_of != f).sum()) for f in range(folds)]
    times = []
    acc = None
    for k in range(args.warmup + args.steps):
        m = MMSBM(K, L, iterations=T, sampling=S, seed=1)
        cx.barrier()
        t0 = time.perf_counter()
        acc = m._cv_execute(pairs)
        cx.barrier()
        dt = cx.max_over_ranks(time.perf_counter() - t0)
        if k >= args.warmup:
            times.append(dt)
    if cx.rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"cv_accuracies": np.asarray(acc, dtype=np.float64)}, id_axis=0)
    if cx.rank == 0:
        per = [len(shard_jobs(folds, S, r, cx.world)) for r in range(cx.world)]
        dt = float(np.mean(times))
        print(json.dumps({
            "metric": "rating-updates/sec", "value": float(sum(n_train)) * T * S / dt, "unit": "rating-updates/s",
            "n_gpus": cx.world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "ml1m_cv", "users": U, "items": I, "ratings": N, "K": K, "L": L, "R": R,
                       "sampling": S, "folds": folds, "iterations_per_step": T, "train_rows_per_fold": n_train,
                       "parallelism": f"folds x runs jobs per GPU {per}", "balance": min(per) / max(per) if max(per) else None,
                       "api": "mmsbm_b200.MMSBM._cv_execute(5 row-wise folds): what cv_fit does after building its "
                              "folds -- encoding, index builds, the folds x runs fits, predict and score of every fold; "
                              "wall clock"},
            "cv_accuracies": [float(a) for a in acc], "wall_s_per_cv": times,
            "roofline": None, "cpu_baseline": None, "e2e": None, "gpu_launches": None}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="ml20m", choices=sorted(WORKLOADS))
    ap.add_argument("--iters-per-step", type=int, default=400)
    ap.add_argument("--cpu-rows", type=int, default=200_000)
    ap.add_argument("--cpu-backend", default="auto", choices=["auto", "numba", "numpy"],
                    help="which of the reference's CPU backends to time (auto: its own order, numba then numpy)")
    ap.add_argument("--ids", default="uniform", choices=["uniform", "zipf"])
    ap.add_argument("--mode", default="best", choices=["best", "runs", "sharded"],
                    help="N > 1: time both ways of placing the runs and report the faster (default), or one")
    ap.add_argument("--netflix-iters", type=int, default=50)
    ap.add_argument("--no-netflix", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-api-e2e", action="store_true",
                    help="N = 1: skip the fit + predict + score through the public MMSBM API")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    shape = WORKLOADS[args.workload]
    if args.dump_outputs:
        args.dump_outputs = os.path.abspath(args.dump_outputs)
        if args.impl == "reference" or (int(os.environ.get("WORLD_SIZE", "1")) > 1 and args.workload != "ml1m_cv"):
            raise SystemExit("bench.py: --dump-outputs is supported for --impl b200 on one GPU and for ml1m_cv")
    with tempfile.TemporaryDirectory(prefix="mmsbm_bench_") as work, contextlib.chdir(work):
        if args.impl == "reference":
            run_reference_arm(args, shape)
            return
        cx = Ctx()
        try:
            if args.workload == "ml1m_cv":
                run_cv(args, shape, cx)
            elif cx.world == 1:
                run_single(args, shape, cx)
            else:
                run_multi(args, shape, cx)
        finally:
            cx.close()


if __name__ == "__main__":
    main()
