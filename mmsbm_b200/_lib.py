"""ctypes binding of libmmsbm_b200.so (include/mmsbm_b200.h).

There is no CPU fallback: if the library has not been built, or no CUDA device is
usable, importing the kernels raises ``ImportError`` -- the same signal the
reference's backend loader uses for an unavailable backend (src/backend.py:23-28,
src/kernels_cupy.py:10-17).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MMSBM_B200_LIB") or os.path.join(_HERE, "libmmsbm_b200.so")

RAW_THETA = 1
RAW_ETA_PR = 2

_i32, _i64, _sz, _vp = C.c_int32, C.c_int64, C.c_size_t, C.c_void_p


class Shard(C.Structure):
    """mmsbm_shard_t of include/mmsbm_b200.h: one rank's part of a sharded set of runs."""
    _fields_ = [("useg", _vp), ("uadj", _vp), ("udeg", _vp), ("usched", _vp), ("n_ratings_u", _i64),
                ("iseg", _vp), ("iadj", _vp), ("ideg", _vp), ("isched", _vp), ("n_ratings_i", _i64),
                ("n_users_own", _i32), ("user_lo", _i32), ("n_items_own", _i32), ("item_lo", _i32),
                ("n_users", _i32), ("n_items", _i32), ("n_levels", _i32), ("K", _i32), ("L", _i32),
                ("n_runs", _i32), ("rank", _i32), ("world", _i32),
                ("exchange", C.POINTER(_vp)), ("nccl_comm", _vp)]


_shp = C.POINTER(Shard)
_PROTOS = {
    "mmsbm_abi_version": (C.c_int, []),
    "mmsbm_last_error": (C.c_char_p, []),
    "mmsbm_device_count": (C.c_int, []),
    "mmsbm_launch_count": (_i64, []),
    "mmsbm_row_stride": (C.c_int, [_i32]),
    "mmsbm_split_triples": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "mmsbm_graph_workspace_bytes": (C.c_int, [_i64, _i32, _i32, _i32, C.POINTER(_sz)]),
    "mmsbm_sched_elems": (C.c_int, [_i64, _i32, C.POINTER(_i64)]),
    "mmsbm_graph_build": (C.c_int, [_vp] * 3 + [_i64, _i32, _i32, _i32] + [_vp] * 10 + [_vp, _sz, _vp]),
    "mmsbm_graph_build_side": (C.c_int, [_vp] * 3 + [_i64, _i32, _i32] + [_vp] * 5 + [_vp, _sz, _vp]),
    "mmsbm_sched_workspace_bytes": (C.c_int, [_i32, C.POINTER(_sz)]),
    "mmsbm_sched_build": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _sz, _vp]),
    "mmsbm_nccl_load": (C.c_int, [C.c_char_p]),
    "mmsbm_nccl_unique_id": (C.c_int, [_vp]),
    "mmsbm_nccl_comm_init": (C.c_int, [_vp, _i32, _i32, C.POINTER(_vp)]),
    "mmsbm_nccl_comm_destroy": (C.c_int, [_vp]),
    "mmsbm_ipc_alloc": (C.c_int, [_sz, C.POINTER(_vp), _vp]),
    "mmsbm_ipc_open": (C.c_int, [_vp, C.POINTER(_vp)]),
    "mmsbm_ipc_close": (C.c_int, [_vp]),
    "mmsbm_ipc_free": (C.c_int, [_vp]),
    "mmsbm_shard_exchange_bytes": (C.c_int, [_i32] * 5 + [C.POINTER(_sz)]),
    "mmsbm_shard_workspace_bytes": (C.c_int, [_shp, C.POINTER(_sz)]),
    "mmsbm_shard_publish": (C.c_int, [_shp, _vp, _vp, _i32, _vp]),
    "mmsbm_em_run_sharded": (C.c_int, [_shp, _i32] + [_vp] * 6 + [_i32, _vp, _sz, _vp, _vp]),
    "mmsbm_em_workspace_bytes": (C.c_int, [_i64] + [_i32] * 6 + [C.POINTER(_sz)]),
    "mmsbm_em_step": (C.c_int, [_vp] * 8 + [_i64] + [_i32] * 6 + [_vp] * 6 + [_i32, _vp, _sz, _vp]),
    "mmsbm_em_step_profiled": (C.c_int, [_vp] * 8 + [_i64] + [_i32] * 6 + [_vp] * 6 + [_i32, _vp, _sz, _vp, _vp]),
    "mmsbm_em_run": (C.c_int, [_vp] * 8 + [_i64] + [_i32] * 7 + [_vp] * 6 + [_vp, _sz, _vp]),
    "mmsbm_fold_in_workspace_bytes": (C.c_int, [_i64] + [_i32] * 7 + [C.POINTER(_sz)]),
    "mmsbm_fold_in": (C.c_int, [_vp] * 3 + [_i64] + [_i32] * 8 + [_vp] * 3 + [_vp, _sz, _vp]),
    "mmsbm_em_converge_workspace_bytes": (C.c_int, [_i64] + [_i32] * 6 + [C.POINTER(_sz)]),
    "mmsbm_em_run_converge": (C.c_int, [_vp] * 8 + [_i64] + [_i32] * 8 + [C.c_double] + [_vp] * 9 + [_vp, _sz, _vp]),
    "mmsbm_em_finalize": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _i32, _i32, _i32, _vp]),
    "mmsbm_likelihood_workspace_bytes": (C.c_int, [_i64] + [_i32] * 6 + [C.POINTER(_sz)]),
    "mmsbm_likelihood_min_workspace_bytes": (C.c_int, [_i64] + [_i32] * 6 + [C.POINTER(_sz)]),
    "mmsbm_likelihood": (C.c_int, [_vp, _vp, _vp, _i64] + [_i32] * 6 + [_vp] * 4 + [_vp, _sz, _vp]),
    "mmsbm_loglik_workspace_bytes": (C.c_int, [_i64] + [_i32] * 6 + [C.POINTER(_sz)]),
    "mmsbm_loglik": (C.c_int, [_vp, _vp, _vp, _i64] + [_i32] * 6 + [_vp] * 4 + [_vp, _sz, _vp]),
    "mmsbm_prod_dist": (C.c_int, [_vp, _vp, _i64] + [_i32] * 6 + [_vp] * 4 + [_vp]),
    "mmsbm_stats_workspace_bytes": (C.c_int, [_i64, _i32, C.POINTER(_sz)]),
    "mmsbm_predict_stats": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "mmsbm_mean_over_runs": (C.c_int, [_vp, _i64, _i32, _vp, _vp]),
    "mmsbm_compute_omegas": (C.c_int, [_vp] * 3 + [_i64, _i32, _i32, _i32] + [_vp] * 4 + [_vp]),
    "mmsbm_index_cache_stats": (C.c_int, [C.POINTER(_i64), C.POINTER(_i64)]),
    "mmsbm_index_cache_clear": (C.c_int, []),
    "mmsbm_host_compute_omegas": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _i32, _i32, _vp, _i32, _vp]),
    "mmsbm_host_update_coefficients": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _i32, _i32, _vp, _i32,
                                                 _vp, _vp, _vp]),
    "mmsbm_host_prod_dist": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _i32, _i32, _vp, _i32, _vp]),
    "mmsbm_host_likelihood": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _i32, _i32, _vp, _i32, _vp]),
    "mmsbm_host_fit": (C.c_int, [_vp, _i64] + [_i32] * 7 + [_vp] * 7),
}
EXPORTS = tuple(sorted(_PROTOS))

_lib = None


class MmsbmError(RuntimeError):
    pass


def load(require_device=False):
    """Load the shared library (once).  Raises ImportError when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not built: run `python -m mmsbm_b200.build` "
                "(nvcc, sm_100a). mmsbm_b200 has no CPU fallback.")
        try:
            lib = C.CDLL(LIB_PATH)
        except OSError as e:  # e.g. libcudart missing
            raise ImportError(f"cannot load {LIB_PATH}: {e}") from e
        for name, (res, args) in _PROTOS.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.mmsbm_abi_version() != 4:
            raise ImportError("libmmsbm_b200.so: ABI version mismatch, rebuild it")
        _lib = lib
    if require_device and _lib.mmsbm_device_count() <= 0:
        raise ImportError("mmsbm_b200: no usable CUDA device ("
                          + _lib.mmsbm_last_error().decode() + "); there is no CPU fallback")
    return _lib


def check(rc, what):
    if rc != 0:
        msg = load().mmsbm_last_error().decode(errors="replace")
        raise MmsbmError(f"{what} failed (code {rc}): {msg}")


def launch_count():
    return int(load().mmsbm_launch_count())
