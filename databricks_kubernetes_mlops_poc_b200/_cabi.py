"""ctypes binding of ``libb200forest.so`` (C ABI declared in ``include/b2f.h``).

This is the thin layer the reference's ``CustomModel`` (reference
``databricks/src/02-register-model.ipynb:305-353``) would bind to replace its sklearn
call -- see INTEGRATION.md.  ctypes releases the GIL for the duration of every call,
so one Python thread per GPU can drive the engine concurrently.

There is no CPU fallback: if the shared library is missing or no CUDA device is usable,
loading / model creation raises and nothing is computed.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

ROW_WORDS = 24
ROW_BYTES = 96
PACKED_ROW_WORDS = 16
PACKED_ROW_BYTES = 64
ROWS_WORDS24 = 0
ROWS_PACKED64 = 1
ROWS_RANKED = 2
SCORED_DTYPE = np.dtype([("proba1", np.float32), ("label", np.int32)])  # b2f_scored
SCORED_FULL_DTYPE = np.dtype(  # b2f_scored_full, 24 bytes
    [("proba1", np.float64), ("label", np.int32), ("is_outlier", np.int32), ("outlier_score", np.float32), ("reserved", np.int32)]
)
MOMENT_VALUES = ROW_WORDS * 3

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "lib", "libb200forest.so")

WALK_NAMES = {0: "smem", 1: "global"}
AGG_NAMES = {0: "rf_mean", 1: "gbdt_logistic", 2: "iforest"}


class B2FError(RuntimeError):
    """An engine call failed; the reference convention is "any exception -> HTTP 500"."""


class Info(C.Structure):
    _fields_ = [
        ("device", C.c_int32),
        ("sm_count", C.c_int32),
        ("agg_mode", C.c_int32),
        ("walk_mode", C.c_int32),
        ("n_trees", C.c_int32),
        ("n_groups", C.c_int32),
        ("max_depth", C.c_int32),
        ("n_cat", C.c_int32),
        ("n_num", C.c_int32),
        ("smem_bytes", C.c_int32),
        ("block_threads", C.c_int32),
        ("rows_per_warp", C.c_int32),
        ("forest_bytes", C.c_int64),
        ("launches", C.c_int64),
        ("launches_tile", C.c_int64),
        ("tile_min_rows", C.c_int64),
        ("tile_ok", C.c_int32),
        ("tile_resident", C.c_int32),
        ("packed_ok", C.c_int32),
        ("tile_warps", C.c_int32),
        ("launches_split", C.c_int64),
        ("split_max_rows", C.c_int64),
        ("outlier_trees", C.c_int32),
        ("rank_ok", C.c_int32),
        ("launches_rank", C.c_int64),
        ("rank_smem_bytes", C.c_int32),
        ("rank_row_bytes", C.c_int32),
        ("rank_stream", C.c_int32),
        ("rank_last_pdl", C.c_int32),
    ]


class RankInfo(C.Structure):
    """b2f_rank_info: the ranked row layout and the size of the forest's rank layout."""

    _fields_ = [
        ("ok", C.c_int32),
        ("row_bytes", C.c_int32),
        ("cat_bytes", C.c_int32),
        ("n_cat", C.c_int32),
        ("n_num", C.c_int32),
        ("depth", C.c_int32),
        ("n_trees", C.c_int32),
        ("layout_bytes", C.c_int32),
        ("cat_shift", C.c_int32 * 16),
        ("cat_bits", C.c_int32 * 16),
        ("n_thresholds", C.c_int32 * 24),
        ("n_pairs", C.c_int32),
        ("pairs", C.c_uint32 * 128),
        ("why", C.c_char * 160),
    ]


class StrColumn(C.Structure):
    """b2f_str_column: one Arrow string array handed to the native row encoder."""

    _fields_ = [
        ("offsets", C.c_void_p),
        ("data", C.c_void_p),
        ("validity", C.c_void_p),
        ("offset", C.c_int64),
        ("data_bytes", C.c_int64),
        ("offsets_are_64", C.c_int32),
        ("reserved", C.c_int32),
    ]


# name -> (restype, argtypes); every symbol declared in include/b2f.h must appear here
SIGNATURES = {
    "b2f_version": (C.c_char_p, []),
    "b2f_last_error": (C.c_char_p, []),
    "b2f_device_count": (C.c_int, []),
    "b2f_blob_validate": (C.c_int, [C.c_void_p, C.c_size_t]),
    "b2f_model_create": (C.c_void_p, [C.c_void_p, C.c_size_t, C.c_int]),
    "b2f_model_destroy": (None, [C.c_void_p]),
    "b2f_model_info": (C.c_int, [C.c_void_p, C.POINTER(Info)]),
    "b2f_ranker_create": (C.c_void_p, [C.c_void_p, C.c_size_t]),
    "b2f_ranker_destroy": (None, [C.c_void_p]),
    "b2f_ranker_info": (C.c_int, [C.c_void_p, C.POINTER(RankInfo)]),
    "b2f_ranker_thresholds": (C.POINTER(C.c_float), [C.c_void_p, C.c_int, C.POINTER(C.c_int32)]),
    "b2f_ranker_layout": (C.c_void_p, [C.c_void_p, C.POINTER(C.c_int64)]),
    "b2f_ranker_rank_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int]),
    "b2f_model_rank_info": (C.c_int, [C.c_void_p, C.POINTER(RankInfo)]),
    "b2f_encoder_attach_ranker": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b2f_encoder_create": (C.c_void_p, [C.c_int, C.c_int, C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p]),
    "b2f_encoder_destroy": (None, [C.c_void_p]),
    "b2f_encoder_codes": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(StrColumn), C.c_void_p, C.c_int]),
    "b2f_encoder_encode": (
        C.c_int,
        [C.c_void_p, C.c_int64, C.POINTER(StrColumn), C.POINTER(C.c_void_p), C.c_void_p, C.c_int, C.c_void_p, C.c_int],
    ),
    "b2f_pinned_alloc": (C.c_void_p, [C.c_size_t]),
    "b2f_pinned_alloc_near": (C.c_void_p, [C.c_int, C.c_size_t]),
    "b2f_pinned_alloc_striped": (C.c_void_p, [C.POINTER(C.c_void_p), C.c_int, C.c_size_t, C.c_size_t]),
    "b2f_pinned_free_striped": (None, [C.c_void_p]),
    "b2f_scorer_create": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_int]),
    "b2f_scorer_destroy": (None, [C.c_void_p]),
    "b2f_scorer_trace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "b2f_scorer_chunk_range": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "b2f_host_threads_default": (C.c_int, [C.c_int]),
    "b2f_host_cpu_limit": (C.c_double, []),
    "b2f_device_numa_node": (C.c_int, [C.c_int, C.POINTER(C.c_int)]),
    "b2f_bind_caller_near": (C.c_int, [C.c_int]),
    "b2f_scorer_start": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(StrColumn), C.POINTER(C.c_void_p), C.c_void_p, C.c_int, C.c_int, C.c_int64]),
    "b2f_scorer_wait": (C.c_int, [C.c_void_p, C.c_int]),
    "b2f_scorer_results": (C.c_void_p, [C.c_void_p]),
    "b2f_scorer_chunk_rows": (C.c_int64, [C.c_void_p]),
    "b2f_scorer_threads": (C.c_int, [C.c_void_p]),
    "b2f_pinned_free": (None, [C.c_void_p]),
    "b2f_predict": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "b2f_predict_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "b2f_predict_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "b2f_predict_pairs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "b2f_model_attach_outlier_forest": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "b2f_predict_full": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "b2f_predict_async_ex": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_uint64)],
    ),
    "b2f_predict_multi_ex": (
        C.c_int,
        [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p],
    ),
    "b2f_predict_device_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "b2f_predict_stream_timed_ex": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p],
    ),
    "b2f_predict_async": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_uint64)],
    ),
    "b2f_wait": (C.c_int, [C.c_void_p, C.c_uint64]),
    "b2f_predict_multi": (
        C.c_int,
        [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p],
    ),
    "b2f_predict_stream": (
        C.c_int,
        [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int],
    ),
    "b2f_device_alloc": (C.c_void_p, [C.c_void_p, C.c_size_t]),
    "b2f_device_free": (None, [C.c_void_p, C.c_void_p]),
    "b2f_copy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b2f_copy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b2f_predict_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p]),
    "b2f_sync": (C.c_int, [C.c_void_p]),
    "b2f_predict_device_timed": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p],
    ),
    "b2f_predict_stream_timed": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p],
    ),
    "b2f_moments": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "b2f_moments_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "b2f_moments_device_timed": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p],
    ),
    "b2f_moments_merge": (None, [C.c_void_p, C.c_int, C.c_void_p]),
    "b2f_comm_unique_id": (C.c_int, [C.c_void_p]),
    "b2f_comm_init_rank": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "b2f_comm_init_all": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "b2f_moments_allgather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2f_moments_multi": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int64, C.c_void_p]),
    "b2f_json_parser_create": (C.c_void_p, [C.c_int, C.c_int, C.c_char_p, C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p]),
    "b2f_json_parser_destroy": (None, [C.c_void_p]),
    "b2f_json_parser_parse": (C.c_int64, [C.c_void_p, C.c_char_p, C.c_int64]),
    "b2f_json_parser_numeric": (C.POINTER(C.c_double), [C.c_void_p, C.c_int]),
    "b2f_json_parser_str_offsets": (C.POINTER(C.c_int32), [C.c_void_p, C.c_int]),
    "b2f_json_parser_str_data": (C.POINTER(C.c_uint8), [C.c_void_p, C.c_int, C.POINTER(C.c_int64)]),
    "b2f_drift_create": (C.c_void_p, [C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "b2f_drift_destroy": (None, [C.c_void_p]),
    "b2f_drift_score": (
        C.c_int,
        [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_float)],
    ),
    "b2f_drift_launches": (C.c_int64, [C.c_void_p]),
    "b2f_kstwo_sf": (C.c_double, [C.c_double, C.c_double]),
}

_lib = None


def load_library(path: str | None = None):
    """dlopen the engine and attach prototypes.  Raises B2FError if it is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise B2FError(
            f"{p} not found: the CUDA engine is not built (run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C databricks_kubernetes_mlops_poc_b200/csrc`). There is no CPU fallback."
        )
    lib = C.CDLL(p)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == header/lib drift
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def last_error() -> str:
    return (load_library().b2f_last_error() or b"").decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise B2FError(f"{what} failed (rc={rc}): {last_error()}")


def ptr(a) -> C.c_void_p:
    """numpy array (or None) -> void*"""
    if a is None:
        return C.c_void_p(0)
    return C.c_void_p(a.ctypes.data)


class PinnedBuffer:
    """A page-locked host allocation exposed as numpy views (the request ring lives in these)."""

    def __init__(self, nbytes: int, device: int | None = None):
        """``device``: place the pages on that GPU's NUMA node (b2f_pinned_alloc_near)."""
        self._lib = load_library()
        self.nbytes = int(nbytes)
        self.addr = self._lib.b2f_pinned_alloc(self.nbytes) if device is None else self._lib.b2f_pinned_alloc_near(int(device), self.nbytes)
        if not self.addr:
            raise B2FError(f"b2f_pinned_alloc({nbytes}) failed: {last_error()}")
        self._raw = (C.c_uint8 * self.nbytes).from_address(self.addr)

    def view(self, dtype, shape, offset: int = 0) -> np.ndarray:
        n = int(np.prod(shape))
        a = np.frombuffer(self._raw, dtype=dtype, count=n, offset=offset)
        return a.reshape(shape)

    def close(self) -> None:
        if self.addr:
            self._raw = None
            self._lib.b2f_pinned_free(self.addr)
            self.addr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
