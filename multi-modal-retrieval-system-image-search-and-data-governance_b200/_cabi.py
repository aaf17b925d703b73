"""ctypes binding of libmmrs_b200.so (include/mmrs_b200.h).  No torch types cross this line:
only raw pointers (tensor.data_ptr()), sizes and a cudaStream_t handle."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = _PKG_DIR / "lib" / "libmmrs_b200.so"

OK = 0
ERR_ARG, ERR_CUDA, ERR_ARCH, ERR_WORKSPACE, ERR_ZERO_NORM, ERR_CAPACITY, ERR_INTERNAL, ERR_RETRY, ERR_TIMEOUT = -1, -2, -3, -4, -5, -6, -7, -8, -9
ERR_NONFINITE = -10
ABI_VERSION = 3
DTYPE_F32, DTYPE_BF16, DTYPE_BF16X3, DTYPE_I8 = 0, 1, 2, 3
PATH_AUTO, PATH_GEMV, PATH_MMA = 0, 1, 2
PATHS = {"auto": PATH_AUTO, "gemv": PATH_GEMV, "mma": PATH_MMA}
LABEL_SAME, LABEL_OTHER = 0, 1
LABEL_MATCH = {"same": LABEL_SAME, "other": LABEL_OTHER}


class MmrsError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"mmrs_b200 error {code}: {message}")
        self.code = code


class NonFiniteError(MmrsError, ValueError):
    """int8 quantisation met a row (gallery or query) holding a NaN or an infinity."""


def open_library(path: Path) -> C.CDLL:
    """Load the library at `path`, refusing one built from another version of include/mmrs_b200.h:
    ctypes cannot see argument lists, so a stale library would read this binding's arguments wrongly."""
    lib = C.CDLL(str(path))
    lib.mmrs_abi_version.restype = C.c_int
    lib.mmrs_abi_version.argtypes = []
    found = lib.mmrs_abi_version()
    if found != ABI_VERSION:
        raise ImportError(f"{path} has C ABI version {found}, this package needs {ABI_VERSION}: rebuild it with "
                          f"`python {_PKG_DIR / 'build.py'} --force`")
    return lib


def _load() -> C.CDLL:
    if not LIB_PATH.exists():
        # build in-tree on first use (needs nvcc); never fall back to anything else
        from .build import build
        build()
    if not LIB_PATH.exists():
        raise ImportError(f"{LIB_PATH} is missing and could not be built: the mmrs_b200 CUDA "
                          "library is required (there is no CPU fallback)")
    return open_library(LIB_PATH)


lib = _load()

_vp, _i32, _i64, _f32, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); kept in sync with include/mmrs_b200.h (tests/test_abi.py parses
# the header and checks every declared symbol is exported and listed here)
SIGNATURES = {
    "mmrs_abi_version": (C.c_int, []),
    "mmrs_last_error": (C.c_char_p, []),
    "mmrs_device_check": (C.c_int, [C.c_int]),
    "mmrs_full_scores_workspace_bytes": (_sz, [_i64, _i32, _i32, _i32]),
    "mmrs_full_scores": (C.c_int, [_vp, _i64, _i32, _i64, _i32, _vp, _i32, _i64, _i32, _f32, _i32,
                                   _vp, _i64, _vp, _sz, _vp]),
    "mmrs_split_bf16x3": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _i64, _vp]),
    "mmrs_quantize_rows_i8": (C.c_int, [_vp, _i32, _i64, _i32, _i64, _vp, _i64, _vp]),
    "mmrs_search_workspace_bytes": (_sz, [_i64, _i32, _i32, _i32, _i32]),
    "mmrs_search_topk": (C.c_int, [_vp, _i64, _i32, _i64, _i32, _vp, _i32, _i64, _i32, _i32, _f32,
                                   _i64, _i32, _vp, _vp, _vp, _sz, _vp]),
    "mmrs_search_host_staging_bytes": (_sz, [_i32, _i32, _i32]),
    "mmrs_search_topk_host": (C.c_int, [_vp, _i64, _i32, _i64, _i32, _vp, _i32, _i64, _i32, _i32,
                                        _f32, _i64, _i32, _vp, _vp, _vp, _sz, _vp]),
    # the async, exhaustive, keys and fused forms end in: row filter, row labels, query labels, label_match, stream
    "mmrs_search_topk_async": (C.c_int, [_vp, _i64, _i32, _i64, _i32, _vp, _i32, _i64, _i32, _i32, _f32,
                                         _i64, _i32, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _i32, _vp]),
    "mmrs_search_topk_host_async": (C.c_int, [_vp, _i64, _i32, _i64, _i32, _vp, _i32, _i64, _i32, _i32,
                                              _f32, _i64, _i32, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _i32,
                                              _vp]),
    "mmrs_search_status": (C.c_int, [_vp]),
    "mmrs_search_exhaustive_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "mmrs_search_topk_exhaustive": (C.c_int, [_vp, _i64, _i32, _i64, _i32, _vp, _i32, _i64, _i32, _i32, _f32,
                                              _i64, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _i32, _vp]),
    # refined top-k: rescore candidate rows against a full-precision store (device or registered host memory)
    "mmrs_refine_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "mmrs_refine_topk": (C.c_int, [_vp, _i32, _i64, _i32, _i64, _vp, _i32, _i64, _i32, _f32, _vp, _i32, _i64, _i32,
                                   _vp, _vp, _vp, _sz, _vp, _vp]),
    "mmrs_host_register": (C.c_int, [_vp, _sz, _vp]),
    "mmrs_host_unregister": (C.c_int, [_vp]),
    "mmrs_search_topk_fused_gather_async": (C.c_int, [_vp, _i64, _i32, _i64, _i32, _vp, _i32, _i64, _i32, _i32, _i32,
                                                      _f32, _i64, _i32, _vp, _vp, _vp, _vp, _i32, _i32, _i64,
                                                      _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _i32, _vp]),
    "mmrs_gather_status": (C.c_int, [_vp, _i32]),
    "mmrs_search_topk_keys_async": (C.c_int, [_vp, _i64, _i32, _i64, _i32, _vp, _i32, _i64, _i32, _i32, _f32,
                                              _i64, _i32, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _i32, _vp]),
    "mmrs_topk_merge_keys_async": (C.c_int, [_vp, _i32, _i32, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _i32, _vp]),
    "mmrs_topk_merge_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "mmrs_topk_merge": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "mmrs_selfjoin_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "mmrs_selfjoin_pairs": (C.c_int, [_vp, _i64, _i32, _i64, _i32, _f32, _i64, _i64, _vp, _i64,
                                      _vp, _vp, _sz, _vp]),
    "mmrs_selfjoin_tc_workspace_bytes": (_sz, [_i64, _i64]),
    "mmrs_selfjoin_pairs_tc": (C.c_int, [_vp, _i64, _vp, _i64, _i64, _i32, _f32, _f32, _i32, _i32, _vp, _i64,
                                         _vp, _i64, _vp, _sz, _vp]),
    "mmrs_selfjoin_stored_workspace_bytes": (_sz, [_i64, _i32, _i64]),
    "mmrs_selfjoin_pairs_stored": (C.c_int, [_vp, _i32, _i64, _i64, _i32, _f32, _f32, _i32, _i32, _vp, _i64, _vp, _i64,
                                             _vp, _sz, _vp]),
    "mmrs_sort_pairs_workspace_bytes": (_sz, [_i64]),
    "mmrs_sort_pairs": (C.c_int, [_vp, _i64, _vp, _sz, _vp]),
    "mmrs_row_norm_range": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _vp]),
    "mmrs_row_norm_range_bf16": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _vp]),
    "mmrs_graph_stats": (C.c_int, [_vp]),
    "mmrs_threshold_sweep_f64": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i32, _vp, _vp, _sz, _vp]),
    "mmrs_threshold_sweep_workspace_bytes": (_sz, [_i32]),
    "mmrs_launch_count": (_i64, []),
    "mmrs_profile_enable": (C.c_int, [C.c_int]),
    "mmrs_profile_read": (C.c_int, [_vp, _vp, _vp, _vp, _i32]),
    "mmrs_threshold_sweep_labeled": (C.c_int, [_vp, _vp, _i64, _i64, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "mmrs_threshold_sweep": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i32, _vp, _vp, _sz, _vp]),
    "mmrs_pack_row_filter": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp]),
    # per-class threshold tuning of a batch of prototypes (best_thresholds)
    "mmrs_threshold_sweep_batched_workspace_bytes": (_sz, [_i32, _i32]),
    "mmrs_score_range_batched": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _vp, _vp]),
    "mmrs_threshold_sweep_batched": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp,
                                               _vp, _sz, _vp]),
    # range search: the rows at or above a per-query threshold, one row window per call
    "mmrs_range_search_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "mmrs_range_search_window": (C.c_int, [_vp, _i64, _i32, _i64, _i32, _vp, _i32, _i64, _i32, _f32, _i32, _vp, _i64,
                                           _i64, _vp, _vp, _vp, _i32, _vp, _vp, _sz, _vp]),
    "mmrs_range_search_scatter": (C.c_int, [_i32, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    # duplicate resolve: the greedy first-keeper decision on a pair list
    "mmrs_resolve_duplicates_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "mmrs_resolve_duplicates": (C.c_int, [_vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
}
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


def last_error() -> str:
    return (lib.mmrs_last_error() or b"").decode("utf-8", "replace")


def check(status: int) -> None:
    if status == ERR_NONFINITE:
        raise NonFiniteError(status, last_error())
    if status != OK:
        raise MmrsError(status, last_error())


def require_b200(device_index: int) -> None:
    """Fail loudly unless `device_index` is a B200; called by every compute entry point."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("mmrs_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")
    check(lib.mmrs_device_check(int(device_index)))
