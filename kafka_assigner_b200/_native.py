"""ctypes binding of libkassign.so (include/kassign.h). Fails loudly when the library is missing:
there is no CPU fallback anywhere in the product path."""
import ctypes
import os

from . import build as _build


class KaStatus(ctypes.Structure):
    _fields_ = [("code", ctypes.c_int32), ("topic_index", ctypes.c_int32), ("partition", ctypes.c_int32),
                ("a", ctypes.c_int32), ("b", ctypes.c_int32)]


class KaPlanTotals(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int64) for n in ("rows", "rows_reordered", "rows_moved", "replicas_added", "replicas_dropped",
                                              "leaders_changed")]


KA_OK = 0
KA_ERR_RF_MISMATCH, KA_ERR_RF_NOT_POSITIVE, KA_ERR_RF_GT_BROKERS, KA_ERR_UNASSIGNABLE, KA_ERR_HASH_INDEX = 1, 2, 3, 4, 5
KA_ERR_BAD_ARG, KA_ERR_CUDA, KA_ERR_NO_DEVICE, KA_ERR_LIMIT = -1, -2, -3, -4

# every symbol include/kassign.h declares: (restype, argtypes)
_vp, _i32, _i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
SYMBOLS = {
    "ka_ctx_create": (_vp, [_i32]),
    "ka_ctx_destroy": (None, [_vp]),
    "ka_ctx_reset": (_i32, [_vp]),
    "ka_ctx_set_brokers": (_i32, [_vp, _i32, _vp, _vp]),
    "ka_rack_indices": (_i32, [_i32, _vp, _vp, _vp]),
    "ka_java_string_hash": (_i32, [ctypes.c_char_p]),
    "ka_solve": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "ka_solve_dense": (_i32, [_vp, _i32, _vp, _i32, _i32, _vp, _i32, _i32, _vp, _vp, _vp]),
    "ka_solve_dense_json": (_i32, [_vp, _i32, _vp, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _i64, _vp, _vp]),
    "ka_solve_dense_json_changed": (_i32, [_vp, _i32, _vp, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _i64, _vp, _vp]),
    "ka_solve_dense_device": (_i32, [_vp, _i32, _vp, _i32, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "ka_stage_dense_device": (_i32, [_vp, _i32, _vp, _i32, _i32, _vp, _i32, _i32, _vp]),
    "ka_order_device": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "ka_ctx_set_topic_base": (_i32, [_vp, _i32]),
    "ka_staged_slot_chains": (_i32, [_vp]),
    "ka_order_slot_device": (_i32, [_vp, _i32, _vp]),
    "ka_emit_device": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "ka_ctx_export_counter_slot_device": (_i32, [_vp, _i32, _vp, _vp]),
    "ka_ctx_import_counter_slot_device": (_i32, [_vp, _i32, _vp, _vp]),
    "ka_last_status": (_i32, [_vp, _vp]),
    "ka_ctx_set_report_brokers": (_i32, [_vp, _i32, _vp]),
    "ka_plan_last": (_i32, [_vp, _vp, _vp, _vp]),
    "ka_ctx_counter_slots": (_i32, [_vp]),
    "ka_ctx_get_counters": (_i32, [_vp, _vp]),
    "ka_ctx_set_counters": (_i32, [_vp, _vp]),
    "ka_ctx_export_counters_device": (_i32, [_vp, _vp, _vp]),
    "ka_ctx_import_counters_device": (_i32, [_vp, _vp, _vp]),
    "ka_ctx_set_timing": (_i32, [_vp, _i32]),
    "ka_ctx_last_timing": (_i32, [_vp, _vp]),
    "ka_ctx_launch_count": (_i64, [_vp]),
    "ka_version": (ctypes.c_char_p, []),
}

_lib = None


def lib_path():
    return _build.LIB


def load():
    """dlopen csrc/libkassign.so and type every exported entry point."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError("%s is missing — run `python __graft_entry__.py` (build) first; "
                           "kassign has no CPU fallback" % path)
    L = ctypes.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(L, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L
