"""ctypes binding of libtss.so (include/tss.h).  The library is the product; this module only declares signatures.

There is no fallback: if libtss.so has not been built (python -m timberborn_support_solver_b200.build) importing
fails, and creating an engine without a CUDA device raises TssError(TSS_E_CUDA).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TSS_LIB") or os.path.join(HERE, "libtss.so")   # TSS_LIB: load another BUILD of libtss (kernel experiments)

TSS_VERSION = 103   # include/tss.h
TSS_OK, TSS_UNKNOWN, TSS_SAT, TSS_UNSAT = 0, 0, 10, 20
TSS_E_INVALID, TSS_E_CAPACITY, TSS_E_CUDA, TSS_E_UNSUPPORTED, TSS_E_PARSE = -1, -2, -3, -4, -5
ERROR_NAMES = {-1: "TSS_E_INVALID", -2: "TSS_E_CAPACITY", -3: "TSS_E_CUDA", -4: "TSS_E_UNSUPPORTED", -5: "TSS_E_PARSE"}


class Platform(C.Structure):  # tss_platform
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("def_w", C.c_int32), ("def_h", C.c_int32), ("rotated", C.c_int32)]


class Dims(C.Structure):  # tss_dims
    _fields_ = [("w", C.c_int32), ("h", C.c_int32)]


class Stats(C.Structure):  # tss_stats
    _fields_ = [("layouts_evaluated", C.c_uint64), ("candidates_scored", C.c_uint64), ("sls_steps", C.c_uint64),
                ("clauses_checked", C.c_uint64), ("kernel_launches", C.c_uint64), ("n_solves", C.c_uint64),
                ("device_ms", C.c_double), ("best_count", C.c_int32), ("interrupted", C.c_int32), ("last_solve_steps", C.c_int64),
                ("sls_flips", C.c_uint64)]


class InstanceInfo(C.Structure):  # tss_instance_info
    _fields_ = [("w", C.c_int32), ("h", C.c_int32), ("n_defs", C.c_int32), ("card_limit_1x1", C.c_int32), ("n_other_card_limits", C.c_int32),
                ("has_weight_limit", C.c_int32), ("weight_limit", C.c_int64), ("n_weights", C.c_int32), ("exact", C.c_int32)]


class SearchParams(C.Structure):  # tss_search_params
    _fields_ = [("seed", C.c_uint64), ("n_chains", C.c_int32), ("chain_offset", C.c_int32), ("noise_pct", C.c_int32),
                ("kernel", C.c_int32)]


# every symbol include/tss.h declares: name -> (restype, argtypes)
_P = C.POINTER
_vp, _i32, _i64, _u64, _u32, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_uint32, C.c_size_t
_u8p, _i32p, _u32p, _i64p = _P(C.c_uint8), _P(C.c_int32), _P(C.c_uint32), _P(C.c_int64)
SIGNATURES = {
    "tss_version": (C.c_int, []),
    "tss_debug_smem_violations": (C.c_int, []),
    "tss_engine_create": (C.c_int, [C.c_int, _P(_vp)]),
    "tss_engine_destroy": (None, [_vp]),
    "tss_engine_set_stream": (C.c_int, [_vp, _vp]),
    "tss_last_error": (C.c_char_p, [_vp]),
    "tss_interrupt": (None, [_vp]),
    "tss_clear_interrupt": (None, [_vp]),
    "tss_get_stats": (C.c_int, [_vp, _P(Stats)]),
    "tss_device_info": (C.c_int, [_vp, C.c_char_p, C.c_int, _P(C.c_int), _P(C.c_int)]),
    "tss_world_parse_toml": (C.c_int, [C.c_char_p, _u8p, _sz, _i32p, _i32p, _i32p, C.c_char_p, _sz]),
    "tss_world_to_toml": (C.c_int, [_u8p, _i32, _i32, C.c_char_p, _sz]),
    "tss_world_synthetic": (C.c_int, [_i32, _i32, _u64, _u64, _u32, _u8p]),
    "tss_encoding_create": (C.c_int, [_u8p, _i32, _i32, _P(Dims), _i32, _P(_vp)]),
    "tss_encoding_destroy": (None, [_vp]),
    "tss_encoding_sizes": (C.c_int, [_vp, _i32p, _i32p, _i64p, _i32p]),
    "tss_encoding_dims": (C.c_int, [_vp, _P(Dims)]),
    "tss_encoding_var_maps": (C.c_int, [_vp, _i32p, _i32p]),
    "tss_encoding_cnf": (C.c_int, [_vp, _i32p, _u32p]),
    "tss_encoding_with_limits": (C.c_int, [_vp, _i32p, _i32, _i32p, _i32, _i32, _i64, _i32p, _i32p, _i64p, _i32p, _u32p]),
    "tss_layout_from_assignment": (C.c_int, [_vp, _u8p, _i32, _P(Platform), _i32, _i32p]),
    "tss_layout_to_assignment": (C.c_int, [_vp, _vp, _P(Platform), _i32, _u8p]),
    "tss_layout_trivial_optimization": (C.c_int, [_u8p, _i32, _i32, _P(Platform), _i32]),
    "tss_layout_merge_supports": (C.c_int, [_u8p, _i32, _i32, _P(Dims), _i32, _P(Platform), _i32, _i32]),
    "tss_layout_total_weight": (_i64, [_P(Platform), _i32, _i32p, _i32]),
    "tss_platform_overlaps": (C.c_int, [_P(Platform), _P(Platform)]),
    "tss_validate": (C.c_int, [_vp, _u8p, _i32, _i32, _P(Platform), _i32, _u8p, _u8p]),
    "tss_eval_sites": (C.c_int, [_vp, _u8p, _i32, _i32, _u8p, _i64, _i32p, _i32p]),
    "tss_eval_packed": (C.c_int, [_vp, _u32p, _i32, _i32, _u32p, _i64, _i32p, _i32p]),
    "tss_eval_compact_dev": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _i64, _i32, _vp]),
    "tss_compact_row_bytes": (_sz, [_i32, _i32]),
    "tss_compact_layout_bytes": (_sz, [_i32, _i32]),
    "tss_eval_platforms": (C.c_int, [_vp, _u8p, _i32, _i32, _P(Platform), _u32p, _i64, _i32p]),
    "tss_cnf_upload": (C.c_int, [_vp, _i32p, _u32p, _i32, _i32, _P(_vp)]),
    "tss_cnf_destroy": (None, [_vp]),
    "tss_cnf_check": (C.c_int, [_vp, _vp, _u8p, _i64, _i32p, _i32p]),
    "tss_cnf_propagate": (C.c_int, [_vp, _vp, _u8p, _i64, _i32p, _i32p]),
    "tss_search_create": (C.c_int, [_vp, _u8p, _i32, _i32, _P(Dims), _i32, _P(SearchParams), _P(_vp)]),
    "tss_search_destroy": (None, [_vp]),
    "tss_search_run": (C.c_int, [_vp, _i64, _i32]),
    "tss_search_best_count": (C.c_int, [_vp, _i32p]),
    "tss_search_set_bound": (C.c_int, [_vp, _i32]),
    "tss_search_best_layout": (C.c_int, [_vp, _P(Platform), _i32, _i32p]),
    "tss_search_n_chains": (C.c_int, [_vp]),
    "tss_search_kernel": (C.c_int, [_vp]),
    "tss_search_global_best": (C.c_int, [_vp, _i32p]),
    "tss_comm_unique_id": (C.c_int, [_vp, _u8p]),
    "tss_comm_init": (C.c_int, [_vp, _u8p, _i32, _i32]),
    "tss_comm_world": (C.c_int, [_vp]),
    "tss_search_read_chains": (C.c_int, [_vp, _u32p, _u32p, _i32p, _i32p, _u32p, _P(C.c_uint64)]),
    "tss_search_write_chains": (C.c_int, [_vp, _u32p]),
    "tss_search_read_placements": (C.c_int, [_vp, _P(C.c_uint16), _i32p, _P(C.c_uint16), _i32p, _i32p, _u32p, _P(Dims), _i32p]),
    "tss_sls_spec_probe": (None, [_u32p]),
    "tss_search_set_weights": (C.c_int, [_vp, _i32p, _i32]),
    "tss_solve_min_weight": (C.c_int, [_vp, _u8p, _i32, _i32, _P(Dims), _i32, _i32p, _i32, _i64, _u64, _i32, _i64, _P(Platform), _i32, _i32p, _i64p]),
    "tss_solve_upper_bound": (C.c_int, [_vp, _u8p, _i32, _i32, _P(Dims), _i32, _i32, _u64, _i32, _i64, _P(Platform), _i32, _i32p]),
    "tss_card_limit_classes": (C.c_int, [_P(Dims), _i32, _i32p, _i32, _i32p, _i32p, _i32p, _i32p]),
    "tss_search_set_card_limits": (C.c_int, [_vp, _i32p, _i32]),
    "tss_solve_with_limits": (C.c_int, [_vp, _u8p, _i32, _i32, _P(Dims), _i32, _i32p, _i32, _i32p, _i32, _i64, _u64, _i32, _i64, _P(Platform), _i32, _i32p, _i64p]),
    "tss_lower_bound": (C.c_int, [_vp, _u8p, _i32, _i32, _P(Dims), _i32, _u64, _i32, _i32p, _i32, _i32p]),
    "tss_lower_bound_lp": (C.c_int, [_vp, _u8p, _i32, _i32, _P(Dims), _i32, _i32p, _i32, _i32, _i64, _i32p, _i64p, _i64p, _i64p, _i32p]),
    "tss_solve_batch": (C.c_int, [_vp, _u8p, _i32, _i32, _i64, _u64, _i64, _i32, _i32p, _u32p]),
    "tss_instance_find": (C.c_int, [_i32p, _u32p, _i32, _i32, _P(_vp), _P(InstanceInfo), _i32p, _i32]),
    "tss_encoding_terrain": (C.c_int, [_vp, _u8p, _sz, _i32p, _i32p]),
    "tss_encoding_defs": (C.c_int, [_vp, _P(Dims), _i32, _i32p]),
    "tss_cnf_num_vars": (C.c_int, [_vp]),
    "tss_witness_for_cnf": (C.c_int, [_vp, _vp, _vp, _P(Platform), _i32, _u8p]),
    "tss_solve_instance": (C.c_int, [_vp, _vp, _vp, _P(InstanceInfo), _i32p, _u64, _i64, _u8p]),
    "tss_cnf_complete": (C.c_int, [_vp, _vp, _u8p, _i32p, _i32p]),
    "tss_engine_certified_unsat": (C.c_int, [_vp, C.c_int]),
    "tss_measure_peaks": (C.c_int, [_vp, _P(C.c_double), _i32]),
}

_lib = None


def load() -> C.CDLL:
    """Loads libtss.so and applies the signatures.  Raises if the library is missing — there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH) and not os.environ.get("TSS_LIB"):
            try:  # a fresh checkout has no artefact yet: compile it in-tree (nvcc, sm_100a) — building is not a fallback
                from . import build as _build
                _build.build()
            except Exception as exc:  # noqa: BLE001
                raise ImportError(f"{LIB_PATH} is missing and could not be built: {exc}.  The GPU path has no CPU fallback.") from exc
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -m timberborn_support_solver_b200.build` "
                              "(nvcc, sm_100a).  The GPU path has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        if not os.environ.get("TSS_LIB") and (any(not hasattr(lib, name) for name in SIGNATURES) or lib.tss_version() != TSS_VERSION):
            # a stale artefact of an older source tree (a declared symbol is missing / other ABI version): rebuild it in-tree
            # once and load the new file; still no fallback — if that fails the import fails
            from . import build as _build
            import shutil
            import tempfile
            _build.build(force=True)
            tmp = os.path.join(tempfile.mkdtemp(prefix="tss_"), "libtss.so")   # (dlopen caches by path: load the fresh build under another name)
            shutil.copy(LIB_PATH, tmp)
            lib = C.CDLL(tmp)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if lib.tss_version() != TSS_VERSION:
            raise ImportError(f"{LIB_PATH} has ABI version {lib.tss_version()}, this package binds {TSS_VERSION}")
        _lib = lib
    return _lib
