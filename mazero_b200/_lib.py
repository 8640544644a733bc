"""ctypes binding of libmaz_b200.so (C ABI: include/maz_tree.h).

There is no CPU fallback: if the shared library is missing this module raises at import time, and every
compute entry point returns MAZ_ERR_CUDA when no CUDA device is usable.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmaz_b200.so")

MAZ_OK, MAZ_ERR_INVALID, MAZ_ERR_CUDA, MAZ_ERR_UNSUPPORTED, MAZ_ERR_DEVICE = 0, 1, 2, 3, 4

_f32p = C.c_void_p   # raw addresses: host numpy buffers or device pointers, depending on the entry point
_i32p = C.c_void_p

# name -> (restype, argtypes).  Must list EVERY symbol include/maz_tree.h declares (tests check this).
SIGNATURES = {
    "maz_abi_version": (C.c_int, []),
    "maz_last_error": (C.c_char_p, []),
    "maz_tree_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                  C.c_uint, C.c_float, C.c_float]),
    "maz_tree_create_ex": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                     C.c_uint, C.c_float, C.c_float, C.c_int, C.c_uint]),
    "maz_tree_destroy": (None, [C.c_void_p]),
    "maz_tree_reset": (C.c_int, [C.c_void_p, C.c_uint, C.c_float, C.c_float, C.c_float, C.c_uint]),
    "maz_tree_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "maz_tree_check": (C.c_int, [C.c_void_p]),
    "maz_tree_set_puct": (C.c_int, [C.c_void_p, C.c_float, C.c_float]),
    "maz_tree_prepare": (C.c_int, [C.c_void_p, _f32p, _f32p, _f32p, _f32p, C.c_int, C.c_float, _f32p]),
    "maz_tree_batch_selection": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_float, _i32p, _i32p, _i32p]),
    "maz_tree_batch_expansion_and_backup": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_int, _f32p, _f32p, _f32p, _f32p]),
    "maz_tree_prepare_dev": (C.c_int, [C.c_void_p, _f32p, _f32p, _f32p, _f32p, C.c_int, C.c_float, _f32p]),
    "maz_tree_batch_selection_dev": (C.c_int, [C.c_void_p, C.c_float, C.c_float, C.c_float, _i32p, _i32p, _i32p]),
    "maz_tree_batch_expansion_and_backup_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_int, _f32p, _f32p, _f32p, _f32p]),
    "maz_tree_expansion_backup_selection_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_int, _f32p, _f32p, _f32p, _f32p,
                                                          C.c_float, C.c_float, _i32p, _i32p, _i32p]),
    "maz_tree_get_roots_values": (C.c_int, [C.c_void_p, _f32p]),
    "maz_tree_get_roots_marginal_visit_count": (C.c_int, [C.c_void_p, _i32p]),
    "maz_tree_get_roots_marginal_priors": (C.c_int, [C.c_void_p, _f32p]),
    "maz_tree_get_roots_num_children": (C.c_int, [C.c_void_p, _i32p]),
    "maz_tree_readout": (C.c_int, [C.c_void_p, C.c_float] + [C.c_void_p] * 15),
    "maz_tree_readout_dev": (C.c_int, [C.c_void_p, C.c_float] + [C.c_void_p] * 15),
    "maz_tree_stats": (C.c_int, [C.c_void_p, _i32p, _i32p, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "maz_tree_set_debug_clock": (C.c_int, [C.c_void_p, C.c_void_p]),
    "maz_tree_arena_bytes": (C.c_size_t, [C.c_void_p]),
    # include/maz_infer.h
    "maz_dbg_umma_gemm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "maz_infer_recurrent": (C.c_int, [C.c_void_p, C.c_void_p]),
    "maz_infer_recurrent_small": (C.c_int, [C.c_void_p, C.c_void_p]),
    "maz_infer_small_nq": (C.c_int, []),
    "maz_infer_configure": (C.c_int, [C.c_int, C.c_int]),
    "maz_infer_initial": (C.c_int, [C.c_void_p, C.c_void_p]),
    "maz_mlp_recurrent": (C.c_int, [C.c_void_p, C.c_void_p]),
    "maz_mlp_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    # include/maz_hostrng.h
    "maz_legacy_dirichlet": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.c_double, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    # include/maz_turn.h
    "maz_root_prepare_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                       C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "maz_dirichlet_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_ulonglong, C.c_void_p]),
    "maz_agent_turn_dev": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    # include/maz_search.h
    "maz_search_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p]),
    "maz_search_destroy": (None, [C.c_void_p]),
    "maz_search_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "maz_search_strategy": (C.c_int, [C.c_void_p]),
    "maz_search_device_bytes": (C.c_size_t, [C.c_void_p]),
    "maz_search_pool": (C.c_void_p, [C.c_void_p]),
    "maz_search_tree": (C.c_void_p, [C.c_void_p]),
    "maz_search_root_arrays": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "maz_search_run_dev": (C.c_int, [C.c_void_p, C.c_void_p]),
    "maz_search_run": (C.c_int, [C.c_void_p, C.c_void_p]),
    "maz_search_check": (C.c_int, [C.c_void_p]),
    "maz_search_set_record": (C.c_int, [C.c_void_p] * 7),
    "maz_search_set_debug_clock": (C.c_int, [C.c_void_p, C.c_void_p]),
    "maz_search_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "maz_search_loop_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "maz_search_roots_per_cta": (C.c_int, [C.c_void_p]),
}

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -m mazero_b200.build` (nvcc, sm_100a). "
        "mazero_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


def last_error():
    return lib.maz_last_error().decode(errors="replace")


def check(rc):
    """Reference convention: C++ runtime_error -> Python RuntimeError (ctree.pxd:14-20)."""
    if rc != MAZ_OK:
        raise RuntimeError(f"libmaz_b200 error {rc}: {last_error()}")
