"""ctypes binding of librpk.so (include/rpk.h).  There is no fallback: if the CUDA library is
missing or no B200 is visible, every entry point raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RPK_LIB") or os.path.join(_HERE, "librpk.so")  # RPK_LIB: an instrumented build (profiles/)

_lib = None

_i32p, _i64p, _f64p, _vp = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p  # raw addresses (host or device)

_SIGNATURES = {
    "rpk_abi_version": (C.c_int, []),
    "rpk_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "rpk_destroy": (None, [C.c_void_p]),
    "rpk_last_error": (C.c_char_p, [C.c_void_p]),
    "rpk_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rpk_sync": (C.c_int, [C.c_void_p]),
    "rpk_launch_count": (C.c_int64, [C.c_void_p]),
    "rpk_debug_flags": (C.c_int, [C.c_void_p, C.c_int]),
    "rpk_fit_topk": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, _i64p, _i32p, C.c_int, _f64p, C.c_int,
                               C.c_int64, C.c_int64, _i32p, _i32p, _f64p, _i32p]),
    "rpk_fit_topk_real": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, _i64p, _i32p, _f64p, C.c_int, _f64p, C.c_int,
                                    C.c_int64, C.c_int64, _i32p, _f64p, _i32p]),
    "rpk_fit_item_counts": (C.c_int, [C.c_void_p, _i32p, C.c_int64]),
    "rpk_model_load_topk": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, _i32p, _f64p, _i32p]),
    "rpk_model_load_topk_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int64, _i32p, _f64p, _i32p, _i64p]),
    "rpk_model_scale_exp": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, _f64p, _i32p, C.POINTER(C.c_int32)]),
    "rpk_model_pack_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int64, _i32p, _f64p, _i32p, C.c_int, _vp]),
    "rpk_model_load_packed_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int64, _vp, _i32p, _i64p, C.c_int]),
    "rpk_model_vmax": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, _f64p, _i32p, _f64p]),
    "rpk_model_pack_rows_v": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int64, _i32p, _f64p, _i32p, _f64p, _vp]),
    "rpk_model_load_packed_rows_v": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int64, _vp, _i32p, _i64p, _f64p]),
    "rpk_fit_token": (C.c_int64, [C.c_void_p]),
    "rpk_model_load_last_fit": (C.c_int, [C.c_void_p, C.c_int64]),
    "rpk_model_load_csr": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p]),
    "rpk_model_load_signed_csr": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p]),
    "rpk_predict_topn": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, C.c_int, C.c_int, _i32p, _f64p, _i32p]),
    "rpk_predict_item_filter": (C.c_int, [C.c_void_p, _vp, C.c_int64]),
    "rpk_predict_csr_count": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, C.c_int, _i64p]),
    "rpk_predict_csr_fill": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, C.c_int, _i64p, _i32p, _f64p]),
    "rpk_topk_csr": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p, C.c_int, _i32p, _i32p]),
    "rpk_coverage_topn": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int64, _i32p, _i32p, _i64p, _i64p, _vp]),
    "rpk_gram_dense_f64": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, _i64p, _i32p, _f64p]),
    "rpk_ease_from_inverse": (C.c_int, [C.c_void_p, C.c_int64, _f64p, _f64p, _f64p]),
    "rpk_ease_prune": (C.c_int, [C.c_void_p, C.c_int64, _f64p, C.c_int64, _i64p, _i32p, _f64p, _i64p]),
    "rpk_predict_dense_topn": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, C.c_int64, _f64p, C.c_int, C.c_int,
                                         _i32p, _f64p, _i32p]),
    "rpk_predict_dense_full": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, C.c_int64, _f64p, C.c_int, _f64p]),
    "rpk_gram_dense_u16": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _vp, _vp]),
    "rpk_trace": (C.c_int, [C.c_void_p, C.c_int]),
    "rpk_trace_report": (C.c_char_p, [C.c_void_p]),
    "rpk_fit_config": (C.c_int, [C.c_void_p, C.c_int]),
    "rpk_spgemm_topn": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p,
                                  C.c_int, C.c_int, _i32p, _f64p, _i32p]),
    "rpk_spgemm_count": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p,
                                   C.c_int, _i64p]),
    "rpk_spgemm_fill": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p, C.c_int64, C.c_int64, _i64p, _i32p, _f64p,
                                  C.c_int, _i64p, C.c_int64, _i32p, _f64p]),
    "rpk_split_fraction": (C.c_int, [C.c_void_p, C.c_int64, _i64p, _i64p, _i64p, C.c_int64, C.c_double, C.c_uint64, _vp]),
    "rpk_fit_strip_rows": (C.c_int, [C.c_void_p, C.c_int64]),
    "rpk_last_timings": (C.c_int, [C.c_void_p, _vp]),
    "rpk_embed_topk": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, _f64p, C.c_int, C.c_int, C.c_int64, C.c_int64, _i32p, _f64p,
                                 _i32p]),
    "rpk_embed_screen_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, _f64p, C.c_int, _vp]),
    "rpk_factor_topn": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int, _f64p, _f64p, C.c_int64, _i64p, _i32p, C.c_int,
                                  C.c_int, _i32p, _f64p, _i32p]),
    "rpk_factor_full": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int, _f64p, _f64p, C.c_int64, _i64p, _i32p, C.c_int,
                                  _f64p]),
    "rpk_factor_screen_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int, _f64p, _f64p, _vp]),
    "rpk_metrics_topn": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, _i32p, _i32p, _i64p, _i32p, C.c_int64, C.c_int,
                                   _i32p, _i32p, _f64p, _f64p, C.c_int, _f64p, _f64p, _i64p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class RpkError(RuntimeError):
    """A call into librpk.so failed."""


def load():
    """Load librpk.so once.  Raises RpkError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RpkError(
            f"{LIB_PATH} is missing: build it with `make -C recpack_b200/csrc` (or __graft_entry__.build()). "
            "recpack_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.rpk_abi_version() != 3:
        raise RpkError("librpk.so ABI version mismatch; rebuild it")
    _lib = lib
    return lib
