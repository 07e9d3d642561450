"""ctypes binding of libolapgpu.so (C ABI declared in include/olap_gpu.h).

This is the Python stand-in for the N-API shim shown in INTEGRATION.md: argument
unpacking, pointer extraction and error translation only.  The library is built
in-tree by ``__graft_entry__.build()`` (olap_in_memory_b200/csrc/Makefile).
There is no fallback: a missing library or a missing CUDA device raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# OLAP_LIB: another build of the same ABI (A/B timing of older commits, tools/ab_drillup.sh); symbols
# such a build lacks are skipped, calling them raises AttributeError
LIB_PATH = os.environ.get("OLAP_LIB") or os.path.join(_HERE, "libolapgpu.so")

OK = 0
E_INVALID, E_CUDA, E_NOMEM, E_UNSUPPORTED = -1, -2, -3, -4

TYPES = {"int32": 0, "uint32": 1, "float32": 2, "float64": 3}
TYPE_NAMES = {v: k for k, v in TYPES.items()}
DEFAULT_ZERO, DEFAULT_NAN = 0, 1
METHODS = {"sum": 0, "average": 1, "highest": 2, "lowest": 3, "first": 4, "last": 5, "product": 6}
COUNT = 7  # extension, see OLAP_COUNT in include/olap_gpu.h


class OlapError(RuntimeError):
    """CUDA / resource failure reported by the native library."""


class OlapValueError(ValueError):
    """Argument error; the message is the reference's own Error text."""


_lib = None

p_store = C.c_void_p
pp_store = C.POINTER(C.c_void_p)
p_i64 = C.POINTER(C.c_int64)
p_i32 = C.POINTER(C.c_int32)
p_int = C.POINTER(C.c_int)
p_f32 = C.POINTER(C.c_float)
p_f64 = C.POINTER(C.c_double)
p_u8 = C.POINTER(C.c_uint8)
pp_i32 = C.POINTER(p_i32)
pp_f64 = C.POINTER(p_f64)

# name -> (restype, argtypes): every symbol include/olap_gpu.h declares
SIGNATURES = {
    "olap_abi_version": (C.c_int, []),
    "olap_init": (C.c_int, [C.c_int]),
    "olap_set_stream": (C.c_int, [C.c_void_p]),
    "olap_set_async": (C.c_int, [C.c_int]),
    "olap_sync": (C.c_int, []),
    "olap_set_shareable": (C.c_int, [C.c_int]),
    "olap_last_error": (C.c_char_p, []),
    "olap_method_from_name": (C.c_int, [C.c_char_p, p_int]),
    "olap_kernel_launches": (C.c_int64, []),
    "olap_last_op_ms": (C.c_double, []),
    "olap_last_op_path": (C.c_char_p, []),
    "olap_guard_violations": (C.c_int64, []),
    "olap_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "olap_host_free": (C.c_int, [C.c_void_p]),
    "olap_store_create": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_int, pp_store]),
    "olap_store_create_batch": (C.c_int, [C.c_int, C.c_int64, p_int, p_int, C.c_int, C.c_int, pp_store]),
    "olap_store_destroy": (C.c_int, [p_store]),
    "olap_store_clone": (C.c_int, [p_store, pp_store]),
    "olap_peer_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p), C.c_char_p]),
    "olap_peer_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "olap_peer_close": (C.c_int, [C.c_void_p]),
    "olap_peer_free": (C.c_int, [C.c_void_p]),
    "olap_store_wrap": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, pp_store]),
    "olap_drill_up_rows": (C.c_int, [pp_store, C.c_int, p_int, C.c_int64, C.c_int64, C.c_int64, p_i32,
                                     C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "olap_store_ipc_export": (C.c_int, [p_store, C.c_char_p, p_i64, p_i64]),
    "olap_peer_map": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "olap_peer_unmap_all": (C.c_int, []),
    "olap_drill_up_pull": (C.c_int, [pp_store, C.c_int, p_int, C.c_int64, C.c_int64, p_i32, p_i32, p_i64, C.c_int, p_i64,
                                     C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, pp_store]),
    "olap_store_copy_status": (C.c_int, [p_store, p_store]),
    "olap_store_size": (C.c_int64, [p_store]),
    "olap_store_byte_length": (C.c_int64, [p_store]),
    "olap_store_type": (C.c_int, [p_store]),
    "olap_store_default_kind": (C.c_int, [p_store]),
    "olap_store_has_status": (C.c_int, [p_store]),
    "olap_store_values_ptr": (C.c_void_p, [p_store]),
    "olap_store_status_ptr": (C.c_void_p, [p_store]),
    "olap_store_values_cptr": (C.c_void_p, [p_store]),
    "olap_store_status_cptr": (C.c_void_p, [p_store]),
    "olap_store_canonicalise": (C.c_int, [p_store]),
    "olap_store_status_derived": (C.c_int, [p_store]),
    "olap_store_upload_f32": (C.c_int, [p_store, C.c_void_p, C.c_int64]),
    "olap_store_upload_f64": (C.c_int, [p_store, C.c_void_p, C.c_int64]),
    "olap_store_download_f32": (C.c_int, [p_store, C.c_void_p, C.c_int64]),
    "olap_store_download_f64": (C.c_int, [p_store, C.c_void_p, C.c_int64]),
    "olap_store_get_value": (C.c_int, [p_store, C.c_int64, p_f64]),
    "olap_store_set_value": (C.c_int, [p_store, C.c_int64, C.c_double]),
    "olap_store_set_values": (C.c_int, [p_store, C.c_void_p, C.c_void_p, C.c_int64]),
    "olap_store_fill": (C.c_int, [p_store, C.c_double]),
    "olap_store_total": (C.c_int, [p_store, p_f64]),
    "olap_store_presence": (C.c_int, [p_store, C.c_void_p, C.c_int64]),
    "olap_store_count_present": (C.c_int, [p_store, p_i64]),
    "olap_store_status": (C.c_int, [p_store, C.c_void_p, C.c_int64]),
    "olap_store_export_sparse": (C.c_int, [p_store, C.c_int64, C.c_void_p, C.c_void_p, p_i64]),
    "olap_store_import_sparse": (C.c_int, [p_store, C.c_void_p, C.c_void_p, C.c_int64]),
    "olap_drill_up": (C.c_int, [pp_store, C.c_int, p_int, C.c_int, p_i64, p_i64, pp_i32, pp_store]),
    "olap_drill_down": (C.c_int, [pp_store, C.c_int, p_int, C.c_int, p_i64, p_i64, pp_i32, pp_f64, p_i64, pp_store]),
    "olap_dice": (C.c_int, [pp_store, C.c_int, C.c_int, p_i64, p_i64, pp_i32, pp_store]),
    "olap_reorder": (C.c_int, [pp_store, C.c_int, C.c_int, p_i64, p_i32, pp_store]),
    "olap_load": (C.c_int, [p_store, p_store, C.c_int, p_i64, p_i64, pp_i32]),
    "olap_region_sum": (C.c_int, [p_store, C.c_int, p_i64, p_i64, pp_i32, p_f64]),
    "olap_region_copy": (C.c_int, [p_store, p_store, C.c_int, p_i64, p_i64, pp_i32]),
    "olap_eval": (C.c_int, [C.c_char_p, pp_store, C.c_int, p_f64, C.c_int, C.c_void_p, C.c_int, C.c_int, pp_store]),
    "olap_region_eval_sum": (C.c_int, [C.c_char_p, pp_store, C.c_int, C.c_int, p_i64, p_i64, pp_i32, p_f64]),
    "olap_region_eval_copy": (C.c_int, [p_store, C.c_char_p, pp_store, C.c_int, C.c_int, p_i64, p_i64, pp_i32]),
    "olap_status_merge": (C.c_int, [pp_store, C.c_int, C.c_void_p, C.c_int64]),
    "olap_status_map_export": (C.c_int, [pp_store, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, p_i64]),
}


def load_library(path: str = LIB_PATH):
    """dlopen the library and declare every signature (no device needed)."""
    if not os.path.exists(path):
        raise OlapError(
            f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(olap_in_memory_b200/csrc/Makefile). This store has no CPU fallback."
        )
    lib = C.CDLL(path)
    for name, (restype, argtypes) in SIGNATURES.items():
        if os.environ.get("OLAP_LIB") and not hasattr(lib, name):
            continue
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    return lib


def lib():
    global _lib
    if _lib is None:
        _lib = load_library()
        if _lib.olap_abi_version() != 1:
            raise OlapError("libolapgpu.so ABI version mismatch")
    return _lib


def check(rc: int):
    if rc == OK:
        return
    message = (lib().olap_last_error() or b"").decode("utf-8", "replace")
    if rc == E_INVALID:
        raise OlapValueError(message)
    raise OlapError(message)


def init(device: int = 0):
    check(lib().olap_init(device))


# ---- small marshalling helpers -----------------------------------------------------
def i64_array(values):
    arr = (C.c_int64 * max(1, len(values)))(*[int(v) for v in values])
    return arr


def int_array(values):
    return (C.c_int * max(1, len(values)))(*[int(v) for v in values])


def store_array(handles):
    return (C.c_void_p * max(1, len(handles)))(*handles)


def map_arrays(maps):
    """list of int sequences -> (keepalive numpy arrays, int32** argument)"""
    keep = [None if m is None else np.ascontiguousarray(np.asarray(m, dtype=np.int32)) for m in maps]
    ptrs = (p_i32 * max(1, len(keep)))(*[p_i32() if a is None else a.ctypes.data_as(p_i32) for a in keep])
    return keep, ptrs
