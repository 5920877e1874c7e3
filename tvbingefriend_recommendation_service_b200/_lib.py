"""ctypes binding of ``libtvbf.so`` (C ABI in ``include/tvbf.h``).

There is no CPU fallback: if the library is missing, or no sm_100 device is present, the
functions here raise.  PyTorch only provides device memory and streams; every pointer handed
to the library is ``tensor.data_ptr()``.
"""

from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libtvbf.so"

TVBF_OK = 0
TEXT_FP16, TEXT_BF16 = 0, 1
GROUP_ABSENT, GROUP_PACKED, GROUP_FOLDED = 0, 1, 2
META_MEAN3, META_HSTACK = 0, 1

c_void_p, c_int32, c_int64, c_double, c_size_t = C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_size_t


class TvbfError(RuntimeError):
    """A libtvbf call returned a non-zero status."""


class Features(C.Structure):
    _fields_ = [
        ("n_shows", c_int32), ("n_pad", c_int32), ("k_pad", c_int32), ("text_dtype", c_int32),
        ("text_scale_log2", c_int32), ("vocab", c_int32),
        ("operand", c_void_p),
        ("text_indptr", c_void_p), ("text_indices", c_void_p), ("text_values", c_void_p),
        ("genre_mode", c_int32), ("genre_dim", c_int32), ("genre_dense", c_void_p),
        ("meta_mode", c_int32), ("meta_kind", c_int32), ("meta_groups", c_int32),
        ("meta_dims", c_int32 * 3), ("meta_dense", c_void_p * 3),
        ("col_side", c_void_p), ("meta_scale", c_void_p),
        ("genre_hi", c_void_p),
        ("text_signed", c_int32),
        ("bits_folded", c_int32), ("fold_col0", c_int32), ("fold_weights", c_double * 3),
        ("text_cols", c_int32),
        ("text_nnz", C.c_int64),
    ]


class Params(C.Structure):
    _fields_ = [
        ("genre_weight", c_double), ("text_weight", c_double), ("metadata_weight", c_double),
        ("min_similarity", c_double),
        ("k", c_int32), ("exclude_self", c_int32), ("row_begin", c_int32), ("row_end", c_int32),
        ("splits", c_int32), ("candidates", c_int32), ("force_exact", c_int32),
        ("skip_fallback", c_int32),
        ("text_rel_err", c_double),
        ("phases", c_int32), ("tuning", c_int32),
    ]


class TopKOut(C.Structure):
    _fields_ = [
        ("indices", c_void_p), ("counts", c_void_p), ("hybrid", c_void_p), ("genre", c_void_p),
        ("text", c_void_p), ("metadata", c_void_p), ("stats", c_void_p),
    ]


# name -> (restype, argtypes); every symbol include/tvbf.h declares
SIGNATURES = {
    "tvbf_version": (C.c_int, []),
    "tvbf_last_error": (C.c_char_p, []),
    "tvbf_kernel_launches": (C.c_uint64, []),
    "tvbf_noncooperative_fallbacks": (C.c_uint64, []),
    "tvbf_device_info": (C.c_int, [C.POINTER(c_int32)] * 3),
    "tvbf_prep_csr_normalize": (C.c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p]),
    "tvbf_prep_csr_to_operand": (C.c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_int32,
                                           c_int32, c_double, c_int32, c_void_p]),
    "tvbf_prep_fold_bits": (C.c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_int32, c_int32,
                                      c_double, c_double, c_int32, c_void_p]),
    "tvbf_merge_plan_workspace_bytes": (c_size_t, [c_int32]),
    "tvbf_merge_plan": (C.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_size_t, c_void_p]),
    "tvbf_prep_csr_to_operand_mapped": (C.c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p,
                                                  c_void_p, c_void_p, c_int32, c_int32, c_double, c_int32, c_void_p]),
    "tvbf_prep_clear_csr_positions": (C.c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_int32, c_int32,
                                                c_void_p]),
    "tvbf_device_zero": (C.c_int, [c_void_p, c_size_t, c_void_p]),
    "tvbf_peer_push": (C.c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_void_p]),
    "tvbf_prep_dense_normalize": (C.c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "tvbf_prep_dense_to_operand": (C.c_int, [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_int32,
                                             c_double, c_int32, c_void_p]),
    "tvbf_prep_genre_bits": (C.c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "tvbf_prep_meta_ids": (C.c_int, [c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_int32,
                                     c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "tvbf_ingest_genre": (C.c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                    c_void_p]),
    "tvbf_ingest_meta": (C.c_int, [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_int32, c_int32,
                                   c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "tvbf_ingest_csr": (C.c_int, [c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p]),
    "tvbf_topk_workspace_bytes": (c_size_t, [C.POINTER(Features), C.POINTER(Params)]),
    "tvbf_hybrid_topk": (C.c_int, [C.POINTER(Features), C.POINTER(Params), C.POINTER(TopKOut),
                                   c_void_p, c_size_t, c_void_p]),
    "tvbf_topk_sweep_workspace_bytes": (c_size_t, [C.POINTER(Features), C.POINTER(Params), c_int32]),
    "tvbf_hybrid_topk_sweep": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_int32, C.POINTER(TopKOut),
                                         c_void_p, c_size_t, c_void_p]),
    "tvbf_sym_eligible": (C.c_int, [C.POINTER(Features), C.POINTER(Params)]),
    "tvbf_sym_list_len": (c_int32, [C.POINTER(Features), C.POINTER(Params)]),
    "tvbf_sym_workspace_bytes": (c_size_t, [C.POINTER(Features), C.POINTER(Params), c_int32]),
    "tvbf_sym_seed": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_int32, c_int32, c_void_p, c_void_p,
                                c_size_t, c_void_p]),
    "tvbf_sym_sweep": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_int32, c_int32, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tvbf_sym_sweep_peer": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_int32, c_int32, c_void_p,
                                      C.POINTER(C.c_uint64), c_int32, c_void_p, c_size_t, c_void_p]),
    "tvbf_rescore_lists": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_void_p, c_void_p, c_void_p, c_int32,
                                     c_int32, c_int32, C.POINTER(TopKOut), c_void_p, c_size_t, c_void_p]),
    "tvbf_append_workspace_bytes": (c_size_t, [C.POINTER(Features), C.POINTER(Params), c_int32]),
    "tvbf_append_topk": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_int32, C.POINTER(TopKOut),
                                   C.POINTER(TopKOut), c_void_p, c_void_p, c_size_t, c_void_p]),
    "tvbf_update_workspace_bytes": (c_size_t, [C.POINTER(Features), C.POINTER(Params), c_int32]),
    "tvbf_update_topk": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_void_p, c_int32, C.POINTER(TopKOut),
                                   C.POINTER(TopKOut), c_void_p, c_void_p, c_size_t, c_void_p]),
    "tvbf_remove_workspace_bytes": (c_size_t, [C.POINTER(Features), C.POINTER(Params), c_int32]),
    "tvbf_remove_topk": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_void_p, c_int32, C.POINTER(TopKOut),
                                   C.POINTER(TopKOut), c_void_p, c_void_p, c_size_t, c_void_p]),
    "tvbf_refresh_workspace_bytes": (c_size_t, [C.POINTER(Features), C.POINTER(Params), c_int32, c_int32, c_int32]),
    "tvbf_refresh_topk": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_void_p, c_int32, c_void_p, c_int32,
                                    c_int32, C.POINTER(TopKOut), C.POINTER(TopKOut), c_void_p, c_void_p, c_size_t,
                                    c_void_p]),
    "tvbf_exact_workspace_bytes": (c_size_t, [C.POINTER(Features), c_int32]),
    "tvbf_exact_rows": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_void_p, c_int32,
                                  C.POINTER(TopKOut), c_void_p, c_size_t, c_void_p]),
    "tvbf_matrix_rows_topk": (C.c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                        C.POINTER(Params), c_void_p, c_int32, C.POINTER(TopKOut),
                                        c_void_p, c_size_t, c_void_p]),
    "tvbf_csr_to_dense_f64": (C.c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "tvbf_cosine_matrix_f64": (C.c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "tvbf_hybrid_combine_f64": (C.c_int, [c_void_p, c_void_p, c_void_p, c_double, c_double, c_double,
                                          c_int64, c_void_p, c_void_p]),
    "tvbf_matrix_stats_workspace_bytes": (c_size_t, []),
    "tvbf_matrix_stats_f64": (C.c_int, [c_void_p, c_int32, C.POINTER(c_double), c_void_p, c_size_t,
                                        c_void_p]),
    "tvbf_stats_accum_bytes": (c_size_t, []),
    "tvbf_text_moments_workspace_bytes": (c_size_t, [C.POINTER(Features), c_int32]),
    "tvbf_text_moments": (C.c_int, [C.POINTER(Features), c_int32, c_void_p, c_void_p, c_size_t, c_void_p]),
    "tvbf_similarity_stats": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_void_p, c_void_p, c_size_t,
                                        c_void_p]),
    "tvbf_score_pairs": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_void_p, c_int32, c_void_p, c_void_p]),
    "tvbf_debug_schedule": (c_int32, [c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                      C.POINTER(c_int32), c_int32]),
    "tvbf_append_plan_tiles": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_int32, C.POINTER(c_int64)]),
    "tvbf_debug_append_schedule": (c_int32, [c_int32, c_int32, c_int32, C.POINTER(c_int32), c_int32]),
    "tvbf_update_plan_tiles": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_int32, C.POINTER(c_int64)]),
    "tvbf_debug_update_schedule": (c_int32, [c_int32, c_int32, c_int32, C.POINTER(c_int32), c_int32]),
    "tvbf_remove_plan_tiles": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_int32, C.POINTER(c_int64)]),
    "tvbf_refresh_plan_tiles": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_int32, c_int32,
                                          C.POINTER(c_int64)]),
    "tvbf_plan_tiles": (C.c_int, [C.POINTER(Features), C.POINTER(Params), c_int32, c_int32, c_int32,
                                  C.POINTER(c_int64)]),
    "tvbf_debug_slack": (C.c_int, [C.POINTER(Features), C.POINTER(Params), C.POINTER(C.c_float)]),
    "tvbf_debug_gemm_tile": (C.c_int, [C.POINTER(Features), c_int32, c_int32, c_void_p, c_void_p]),
    "tvbf_debug_gemm_tile_pair": (C.c_int, [C.POINTER(Features), c_int32, c_int32, c_void_p, c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Load ``libtvbf.so`` (built in-tree by ``build.py``); raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise TvbfError(
            f"{LIB_PATH} is missing: build it with "
            "`python -m tvbingefriend_recommendation_service_b200.build`. "
            "There is no CPU fallback for this path.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status != TVBF_OK:
        msg = load().tvbf_last_error()
        raise TvbfError(f"{what} failed ({status}): {msg.decode() if msg else 'no message'}")


def require_device() -> tuple[int, int, int]:
    """(sm_count, cc_major, cc_minor) of the current CUDA device; raises unless it is sm_100."""
    import torch

    if not torch.cuda.is_available():
        raise TvbfError("no CUDA device: the hybrid top-K path runs only on sm_100a (B200); "
                        "there is no CPU fallback")
    sm, maj, mnr = c_int32(), c_int32(), c_int32()
    check(load().tvbf_device_info(C.byref(sm), C.byref(maj), C.byref(mnr)), "tvbf_device_info")
    return sm.value, maj.value, mnr.value
