"""ctypes binding of librsb.so (include/rsb.h).  There is NO CPU fallback: if the CUDA library cannot be
loaded (or built with nvcc) importing this module's `lib()` raises."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_uint8, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# RSB_LIBRARY: load another build of the SAME CUDA library (kernel A/B experiments, scripts/build_variants.sh)
LIB_PATH = os.environ.get("RSB_LIBRARY") or os.path.join(_HERE, "librsb.so")

RSB_OK = 0
RSB_ERR_INVALID, RSB_ERR_CUDA, RSB_ERR_STATE, RSB_ERR_UNSUPPORTED, RSB_ERR_OOM = -1, -2, -3, -4, -5
RSB_FLAT, RSB_IVFFLAT, RSB_IVFPQ = 0, 1, 2
RSB_GEMM_ROWS_REVERSED = 0x100      # rsb_gemm_f16 epilogue flag
(INFO_KIND, INFO_D, INFO_NLIST, INFO_M, INFO_NBITS, INFO_NTOTAL, INFO_IS_TRAINED, INFO_MAX_LIST_LEN,
 INFO_INDEX_BYTES) = range(9)
PROF_NAMES = ("coarse_ms", "setup_ms", "lut_ms", "scan_ms", "merge_ms", "scan_bytes", "pairs", "launches", "scan_path")

# every symbol include/rsb.h declares: (name, restype, argtypes)
_H = c_void_p
SIGNATURES = [
    ("rsb_version", c_int, []),
    ("rsb_last_error", c_char_p, []),
    ("rsb_flat_create", c_int, [c_int, POINTER(_H)]),
    ("rsb_ivfflat_create", c_int, [c_int, c_int, POINTER(_H)]),
    ("rsb_ivfpq_create", c_int, [c_int, c_int, c_int, c_int, POINTER(_H)]),
    ("rsb_free", c_int, [_H]),
    ("rsb_set_centroids", c_int, [_H, c_void_p, c_void_p]),
    ("rsb_set_pq_codebook", c_int, [_H, c_void_p, c_void_p]),
    ("rsb_get_centroids", c_int, [_H, c_void_p, c_void_p]),
    ("rsb_get_pq_codebook", c_int, [_H, c_void_p, c_void_p]),
    ("rsb_add_workspace_bytes", c_size_t, [_H, c_int64]),
    ("rsb_add", c_int, [_H, c_void_p, c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    ("rsb_add_preassigned", c_int, [_H, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    ("rsb_add_codes", c_int, [_H, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    ("rsb_finalize", c_int, [_H, c_void_p]),
    ("rsb_info", c_int, [_H, c_int, POINTER(c_int64)]),
    ("rsb_list_sizes", c_int, [_H, c_void_p, c_void_p]),
    ("rsb_export_lists", c_int, [_H, c_void_p, c_void_p, c_void_p, c_void_p]),
    ("rsb_workspace_bytes", c_size_t, [_H, c_int, c_int, c_int]),
    ("rsb_search", c_int, [_H, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    ("rsb_search_preassigned", c_int, [_H, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_size_t, c_void_p]),
    ("rsb_search_preassigned_shared", c_int, [_H, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                              c_void_p, c_size_t, c_void_p, c_void_p, c_int, c_void_p]),
    ("rsb_kmeans_accumulate", c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    ("rsb_pq_assign", c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    ("rsb_pq_accumulate", c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    ("rsb_peer_broadcast", c_int, [c_void_p, c_size_t, c_void_p, c_int, c_size_t, c_void_p]),
    ("rsb_coarse", c_int, [_H, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    ("rsb_merge_topk", c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    ("rsb_merge_topk_peers", c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    ("rsb_merge_topk_peers_scatter", c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                             c_int, c_void_p]),
    ("rsb_knn_workspace_bytes", c_size_t, [c_int, c_int64, c_int]),
    ("rsb_knn_ip", c_int, [c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_int64, c_void_p, c_void_p,
                           c_void_p, c_size_t, c_void_p]),
    ("rsb_set_option", c_int, [_H, c_int, c_int64]),
    ("rsb_set_profiling", c_int, [_H, c_int]),
    ("rsb_get_profile", c_int, [_H, POINTER(c_double), c_int]),
    ("rsb_bert_last_error", c_char_p, []),
    ("rsb_bert_create", c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, POINTER(_H)]),
    ("rsb_bert_free", c_int, [_H]),
    ("rsb_bert_load", c_int, [_H, c_char_p, c_void_p, c_int64, c_void_p]),
    ("rsb_bert_workspace_bytes", c_size_t, [_H, c_int]),
    ("rsb_bert_forward", c_int, [_H, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                 c_size_t, c_void_p]),
    ("rsb_bert_launches", c_int64, [_H]),
    ("rsb_bert_attention", c_int, [_H, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    ("rsb_bert_layernorm", c_int, [_H, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    ("rsb_gemm_f16", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    ("rsb_debug_smem_base", c_int, []),
    ("rsb_pq_layout_offset", c_int, [c_int, c_int, c_int]),
    ("rsb_pq_lut_index", c_int, [c_int, c_int, c_int]),
]

_lib = None


class RsbError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        # building is not a fallback: it produces the same CUDA library
        from . import _build
        _build.build()
    try:
        L = ctypes.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise ImportError(
            f"librsb.so could not be loaded from {LIB_PATH}: {e}. retrieval_scaling_b200 has no CPU path; "
            f"build it with `python -m retrieval_scaling_b200._build`.") from e
    for name, res, args in SIGNATURES:
        fn = getattr(L, name)  # AttributeError here == header/library mismatch, by design
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(rc: int) -> None:
    if rc == RSB_OK:
        return
    msg = lib().rsb_last_error().decode("utf-8", "replace")
    if rc == RSB_ERR_INVALID:
        raise ValueError(msg)
    if rc == RSB_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == RSB_ERR_OOM:
        raise MemoryError(msg)
    raise RsbError(f"librsb error {rc}: {msg}")
