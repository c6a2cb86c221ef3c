"""ctypes binding of librwr_b200.so -- exactly the symbols include/rwr_b200.h declares.

Fails loudly when the shared library is missing: there is no Python/NumPy/torch fallback for the hot path.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# RWR_B200_LIB: another build of the same library (the checked build: `make -C csrc CHECKED=1`)
LIB_PATH = os.environ.get("RWR_B200_LIB") or os.path.join(_HERE, "librwr_b200.so")

ABI_VERSION = 2
RWR_OK = 0
RWR_E_INVALID, RWR_E_BADSEED, RWR_E_ALREADY_BUILT, RWR_E_BADINDEX, RWR_E_NOT_BUILT = -1, -2, -3, -4, -5
RWR_E_CUDA, RWR_E_NCCL, RWR_E_OOM, RWR_E_UNSUPPORTED = -6, -7, -8, -9
FP64, FP32 = 0, 1
LAYOUT_AUTO, LAYOUT_VALUED, LAYOUT_INDEX = 0, 1, 2
INIT_UNIFORM, INIT_NODE, INIT_RESTART = 0, 1, 2


class rwr_opts(C.Structure):
    _fields_ = [("device", C.c_int32), ("layout", C.c_int32), ("relabel", C.c_int32), ("hub_entries", C.c_int32),
                ("batch_width", C.c_int32), ("kernel", C.c_int32), ("stream", C.c_uint64),
                ("hot_min_degree", C.c_int32), ("undefined_type_mask", C.c_int32), ("zero_weight_type_mask", C.c_int32),
                ("x_blocks", C.c_int32), ("empty_seed_ok", C.c_int32), ("reserved", C.c_int32)]


class rwr_synth_spec(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("n_users", C.c_int32), ("n_items", C.c_int32), ("n_third", C.c_int32),
                ("authorship_per_mille", C.c_int32), ("n_like", C.c_int64), ("n_friend", C.c_int64),
                ("n_follow", C.c_int64), ("n_mention", C.c_int64), ("undefined_per_mille", C.c_int32),
                ("scramble", C.c_int32), ("p1_byte", C.c_int32), ("reserved", C.c_int32)]


class rwr_graph_info(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("built", C.c_int32), ("n_links_raw", C.c_int64), ("nnz", C.c_int64),
                ("n_dangling", C.c_int32), ("layout", C.c_int32), ("relabelled", C.c_int32), ("n_hot", C.c_int32),
                ("hub_entries_fp64", C.c_int32), ("hub_entries_fp32", C.c_int32), ("n_chunks", C.c_int32),
                ("max_in_degree", C.c_int32), ("max_out_degree", C.c_int32), ("build_ms", C.c_float),
                ("synth_ms", C.c_float), ("device_bytes", C.c_int64), ("row_begin", C.c_int32), ("row_end", C.c_int32),
                ("n_ranks", C.c_int32), ("x_blocks", C.c_int32)]


class rwr_run_info(C.Structure):
    _fields_ = [("n_seeds", C.c_int32), ("n_nodes", C.c_int32), ("precision", C.c_int32), ("iterations", C.c_int32),
                ("residual", C.c_double), ("iterate_ms", C.c_float), ("total_ms", C.c_float),
                ("kernel_launches", C.c_int64)]


# name -> (restype, argtypes); every symbol of include/rwr_b200.h
_vp, _i32, _i64, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double
_pp = C.POINTER(C.c_void_p)
SYMBOLS = {
    "rwr_abi_version": (C.c_int, []),
    "rwr_device_count": (C.c_int, []),
    "rwr_last_error": (C.c_char_p, []),
    "rwr_graph_create": (C.c_int, [_i32, _vp, _vp, _i64, _vp, _vp, _vp, _vp, C.POINTER(rwr_opts), _pp]),
    "rwr_synth_create": (C.c_int, [C.POINTER(rwr_synth_spec), C.POINTER(rwr_opts), _pp]),
    "rwr_graph_build": (C.c_int, [_vp]),
    "rwr_graph_get_info": (C.c_int, [_vp, C.POINTER(rwr_graph_info)]),
    "rwr_graph_export_links": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "rwr_graph_get_csr": (C.c_int, [_vp, _vp, _vp, _vp]),
    "rwr_graph_get_csr_types": (C.c_int, [_vp, _vp]),
    "rwr_graph_get_degrees": (C.c_int, [_vp, _vp, _vp]),
    "rwr_graph_destroy": (None, [_vp]),
    "rwr_run_fixed": (C.c_int, [_vp, _vp, _i32, _f64, _i32, _i32, _pp]),
    "rwr_run_threshold": (C.c_int, [_vp, _vp, _i32, _f64, _f64, _i32, _i32, _vp, _pp]),
    "rwr_run_fixed_restart": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _f64, _i32, _i32, _pp]),
    "rwr_run_threshold_restart": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _f64, _f64, _i32, _i32, _vp, _pp]),
    "rwr_rerun_fixed": (C.c_int, [_vp, _vp, _f64, _i32]),
    "rwr_continue_fixed": (C.c_int, [_vp, _i32]),
    "rwr_continue_threshold": (C.c_int, [_vp, _f64, _i32, _vp]),
    "rwr_set_rank": (C.c_int, [_vp, _i32, _vp]),
    "rwr_result_get_info": (C.c_int, [_vp, C.POINTER(rwr_run_info)]),
    "rwr_scores": (C.c_int, [_vp, _i32, _vp]),
    "rwr_topk": (C.c_int, [_vp, _i32, _vp, _vp, _vp]),
    "rwr_rank_all": (C.c_int, [_vp, _i32, _vp, _vp, _i64, _vp]),
    "rwr_result_destroy": (None, [_vp]),
    "rwr_recommend": (C.c_int, [_vp, _vp, _i32, _f64, _i32, _i32, _i32, _vp, _vp, _vp, C.POINTER(rwr_run_info)]),
    "rwr_profile_iteration": (C.c_int, [_vp, _i32, _f64, _i32, _i32, _vp, _vp]),
    "rwr_probe_tile_ranks": (C.c_int, [_vp, _vp, _i32, _f64, _i32, _i32, _vp]),
    "rwr_evaluate": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp]),
    "rwr_methodology_masks": (C.c_int, [_i32, _vp, _vp, _vp]),
    "rwr_graph_hold_out": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _vp, _vp, _i64, _vp]),
    "rwr_evaluate_users": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _f64, _i32, _i32, _i32, _vp, _vp, _vp, _vp,
                                     C.POINTER(rwr_run_info)]),
    "rwr_comm_unique_id": (C.c_int, [_vp]),
    "rwr_comm_create": (C.c_int, [_i32, _i32, _vp, C.POINTER(rwr_opts), _pp]),
    "rwr_comm_destroy": (None, [_vp]),
    "rwr_synth_create_partitioned": (C.c_int, [C.POINTER(rwr_synth_spec), C.POINTER(rwr_opts), _vp, _pp]),
    "rwr_graph_create_partitioned": (C.c_int, [_i32, _vp, _vp, _i64, _vp, _vp, _vp, _vp, C.POINTER(rwr_opts), _vp, _pp]),
}

_lib = None


def lib() -> C.CDLL:
    """Loads librwr_b200.so (once).  Raises -- never falls back -- when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA extension first (python -c 'import __graft_entry__ as g; "
                "g.build()' or make -C recommendersystems_b200/csrc). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)          # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        if L.rwr_abi_version() != ABI_VERSION:
            raise ImportError("librwr_b200.so ABI version mismatch")
        _lib = L
    return _lib


def last_error() -> str:
    return lib().rwr_last_error().decode("utf-8", "replace")
