"""Build libmmsbm_b200.so in-tree with nvcc for sm_100a (run by __graft_entry__.build()).

    python -m mmsbm_b200.build [--force]
"""
import concurrent.futures as cf
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmmsbm_b200.so")
SOURCES = ["em_step.cu", "em_small.cu", "seg_inst_ch1.cu", "seg_inst_ch2.cu", "seg_inst_ch4.cu", "seg_inst_pair.cu", "seg_inst_hexa.cu", "graph_build.cu",
           "reductions.cu", "host_api.cu", "sharded_run.cu", "fold_in.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-O3,-Wall", "-DMMSBM_B200",   # no --use_fast_math: IEEE fp64 throughout
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False, check=False):
    """Compile every .cu to an object (in parallel) and link the shared library.
    ``check=True`` builds libmmsbm_b200_check.so with device-side bounds checks
    (-DMMSBM_BOUNDS_CHECK); select it at run time with MMSBM_B200_LIB=<path>."""
    nvcc = _nvcc()
    suffix, extra, lib = ("_chk.o", ["-DMMSBM_BOUNDS_CHECK"], LIB.replace(".so", "_check.so")) if check \
        else (".o", ["-DNDEBUG"], LIB)
    headers = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "segment_pass.cuh"), os.path.join(CSRC, "em_internal.cuh"),
               os.path.join(HERE, "..", "include", "mmsbm_b200.h"), os.path.abspath(__file__)]
    objs, jobs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(CSRC, src[:-3] + suffix)
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            jobs.append(cmd)
    if jobs:
        with cf.ThreadPoolExecutor(max_workers=len(jobs)) as ex:
            for cmd, res in zip(jobs, ex.map(lambda c: subprocess.run(c, capture_output=True, text=True), jobs)):
                if verbose or res.returncode:
                    sys.stderr.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
                if res.returncode:
                    raise RuntimeError("nvcc failed for " + cmd[-3])
    if jobs or force or _stale(lib, objs):
        cmd = [nvcc, "-shared", "-o", lib] + objs + ["-lcudart", "-ldl"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("link failed")
    return lib


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv, check="--check" in sys.argv))
