"""ctypes binding of libcmdiad_b200.so (the C ABI declared in include/cmdiad_b200.h).

There is no CPU fallback anywhere in this package: if the shared library is missing the import of the product path
fails loudly, and on a machine without an sm_100 GPU every compute call raises CmdbError(CMDB_ERR_CUDA).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libcmdiad_b200.so")

CMDB_OK = 0
CMDB_ERR_INVALID = -1
CMDB_ERR_CUDA = -2
CMDB_ERR_STATE = -3
CMDB_ERR_CAPACITY = -4
CMDB_ERR_UNSUPPORTED = -5
CORESET_FP16 = 0
CORESET_FP64 = 1
SCORE_TCGEN05 = 0
SCORE_SIMT = 1
OPT_SCORE_IMPL = 1
OPT_TIMING = 2
OPT_PREFILTER_TERMS = 3
T_STAGES = ("stage_in", "gemm", "refine", "map", "reweight", "out")

c_i64_p = ctypes.POINTER(ctypes.c_int64)
c_i32_p = ctypes.POINTER(ctypes.c_int32)
c_f32_p = ctypes.POINTER(ctypes.c_float)
c_f64_p = ctypes.POINTER(ctypes.c_double)
c_u8_p = ctypes.POINTER(ctypes.c_uint8)


class ScoreOut(ctypes.Structure):
    """struct cmdb_score_out"""
    _fields_ = [("s", c_f32_p), ("s_star", c_f32_p), ("s_idx", c_i64_p), ("min_val", c_f32_p), ("min_idx", c_i64_p),
                ("nn_idx", c_i64_p), ("m_star_knn", c_f32_p), ("w", c_f32_p), ("s_map", c_f32_p),
                ("s_map_pre", c_f32_p), ("s_map_u8", c_u8_p)]


class FusionHead(ctypes.Structure):
    """struct cmdb_fusion_head"""
    _fields_ = [("n_modal", ctypes.c_int), ("s_lambda", ctypes.c_float * 3), ("smap_lambda", ctypes.c_float * 3),
                ("detect_coef", ctypes.c_double * 3), ("detect_offset", ctypes.c_double),
                ("seg_coef", ctypes.c_double * 3), ("seg_offset", ctypes.c_double)]


class FusedOut(ctypes.Structure):
    """struct cmdb_fused_out"""
    _fields_ = [("s", c_f64_p), ("s_map", c_f64_p), ("s_modal", c_f32_p), ("min_val", c_f32_p * 3), ("min_idx", c_i64_p * 3)]


FUSED_KEEP_ON_DEVICE = 1
FUSED_NO_HOST_MAPS = 2


class CmdbError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"cmdiad_b200 error {status}: {message}")
        self.status = status


# every symbol include/cmdiad_b200.h declares: name -> (restype, argtypes)
_VP = ctypes.c_void_p
_I = ctypes.c_int
_I64 = ctypes.c_int64
SYMBOLS = {
    "cmdb_version": (_I, []),
    "cmdb_last_error": (ctypes.c_char_p, []),
    "cmdb_device_count": (_I, [ctypes.POINTER(_I)]),
    "cmdb_bank_create": (_I, [_I, _I, _I64, ctypes.POINTER(_VP)]),
    "cmdb_bank_destroy": (None, [_VP]),
    "cmdb_bank_append": (_I, [_VP, _VP, _I64, _I]),
    "cmdb_bank_rows": (_I, [_VP, c_i64_p]),
    "cmdb_bank_dim": (_I, [_VP, ctypes.POINTER(_I)]),
    "cmdb_bank_set_row_offset": (_I, [_VP, _I64]),
    "cmdb_bank_set_option": (_I, [_VP, _I, _I]),
    "cmdb_bank_stats": (_I, [_VP, c_f64_p, c_f64_p, c_f64_p, c_f64_p]),
    "cmdb_bank_normalize": (_I, [_VP, ctypes.c_float, ctypes.c_float]),
    "cmdb_bank_gather": (_I, [_VP, _VP, _I64]),
    "cmdb_bank_read": (_I, [_VP, _I64, _I64, _VP]),
    "cmdb_bank_finalize": (_I, [_VP]),
    "cmdb_bank_stream": (_I, [_VP, ctypes.POINTER(_VP)]),
    "cmdb_bank_lane_streams": (_I, [_VP, ctypes.POINTER(_VP)]),
    "cmdb_bank_get_timings": (_I, [_VP, c_f32_p]),
    "cmdb_bank_score_stats": (_I, [_VP, _VP]),
    "cmdb_bank_build_knn": (_I, [_VP]),
    "cmdb_coreset_select": (_I, [_VP, _I64, _VP, _VP, _VP, _I, _I, _VP]),
    "cmdb_comm_create": (_I, [_I, _I, _I, ctypes.c_size_t, ctypes.POINTER(_VP)]),
    "cmdb_comm_handle_bytes": (_I, []),
    "cmdb_comm_export": (_I, [_VP, _VP]),
    "cmdb_comm_import": (_I, [_VP, _VP]),
    "cmdb_comm_reset": (_I, [_VP]),
    "cmdb_comm_destroy": (None, [_VP]),
    "cmdb_coreset_mailbox_bytes": (ctypes.c_size_t, [_I, _I]),
    "cmdb_coreset_comm_bytes": (ctypes.c_size_t, [_I, _I, _I64, _I]),
    "cmdb_coreset_select_sharded": (_I, [_VP, _VP, _I64, _I64, _VP, _VP, _VP, _I, _I, _VP, _VP]),
    "cmdb_project": (_I, [_VP, _VP, _VP, _VP, _I, _I64, _I64, _VP]),
    "cmdb_coreset_rownorms": (_I, [_I, _VP, _VP, _I64, _I, _I, _VP]),
    "cmdb_score": (_I, [_VP, _VP, _I, _I, _I, _I, _I, ctypes.POINTER(ScoreOut)]),
    "cmdb_score_batch": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, ctypes.POINTER(ScoreOut)]),
    "cmdb_score_batch_submit": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, ctypes.c_uint, ctypes.POINTER(ctypes.c_int64)]),
    "cmdb_score_batch_wait": (_I, [_VP, ctypes.c_int64, ctypes.POINTER(ScoreOut)]),
    "cmdb_score_shard_min": (_I, [_VP, _VP, _I, _I, _I, _I, _VP]),
    "cmdb_upsample_blur": (_I, [_I, _VP, _I, _I, _I, _VP, _VP, _VP]),
    "cmdb_bank_set_query_norm": (_I, [_VP, ctypes.c_float, ctypes.c_float, _I]),
    "cmdb_bank_build_knn_rows": (_I, [_VP, _I64, _I64]),
    "cmdb_bank_read_knn": (_I, [_VP, _I64, _I64, _VP, _I]),
    "cmdb_bank_set_knn_table": (_I, [_VP, _VP, _I64, _I]),
    "cmdb_score_shard_lookup": (_I, [_VP, _VP, _I, _I, _VP]),
    "cmdb_score_shard_finish_submit": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _I, ctypes.c_uint, ctypes.POINTER(ctypes.c_int64)]),
    "cmdb_score_shard_wait": (_I, [_VP, ctypes.c_int64, ctypes.POINTER(ScoreOut)]),
    "cmdb_bank_attach_comm": (_I, [_VP, _VP]),
    "cmdb_score_shard_round_submit": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _I, _I, _I, ctypes.c_uint, ctypes.POINTER(ctypes.c_int64)]),
    "cmdb_bank_read_device": (_I, [_VP, _I64, _I64, _VP]),
    "cmdb_score_fused_batch_submit": (_I, [ctypes.POINTER(_VP), ctypes.POINTER(_VP), ctypes.POINTER(_I), ctypes.POINTER(_I),
                                           ctypes.POINTER(_I), _I, _I, _I, ctypes.POINTER(FusionHead), ctypes.c_uint,
                                           ctypes.POINTER(ctypes.c_int64)]),
    "cmdb_score_fused_batch_wait": (_I, [_VP, ctypes.c_int64, ctypes.POINTER(FusedOut)]),
    "cmdb_score_fused_batch": (_I, [ctypes.POINTER(_VP), ctypes.POINTER(_VP), ctypes.POINTER(_I), ctypes.POINTER(_I),
                                    ctypes.POINTER(_I), _I, _I, _I, ctypes.POINTER(FusionHead), ctypes.c_uint,
                                    ctypes.POINTER(FusedOut)]),
    "cmdb_eval_reserve": (_I, [_VP, _I64, _I]),
    "cmdb_eval_reset": (_I, [_VP]),
    "cmdb_eval_count": (_I, [_VP, c_i64_p]),
    "cmdb_eval_read": (_I, [_VP, _I64, _I64, _VP, _VP]),
    "cmdb_eval_pixel_metrics": (_I, [_VP, _VP, _I64, _VP, _I, _VP, _VP, _VP, ctypes.POINTER(ctypes.c_uint64), c_i64_p, c_i64_p]),
}
# test hook exported by the library but deliberately not part of the public header
DEBUG_SYMBOLS = {
    "cmdb_debug_exact_min": (_I, [_VP, _VP, _I, _VP, _VP]),
    "cmdb_debug_eval_load": (_I, [_VP, _VP, _I64]),
    "cmdb_coreset_select_debug": (_I, [_VP, _I64, _VP, _VP, _VP, _I, _I, _VP, _VP, _VP, _I]),
    "cmdb_debug_coreset_plan": (_I, [_I, _I64, _I, _I, c_i64_p, ctypes.POINTER(_I)]),
    "cmdb_debug_producer_tiles": (_I, [_I, _I, _I, _I, _I, _I, c_i32_p, _I, ctypes.POINTER(_I)]),
}

_lib = None


def load():
    """Loads the shared library (built in-tree by cmdiad_b200/build.py). Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(f"{SO_PATH} not found: run `python -m cmdiad_b200.build` (or __graft_entry__.build()); "
                          "cmdiad_b200 has no CPU fallback")
    lib = ctypes.CDLL(SO_PATH)
    for name, (res, args) in {**SYMBOLS, **DEBUG_SYMBOLS}.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status):
    if status != CMDB_OK:
        raise CmdbError(status, load().cmdb_last_error().decode("utf-8", "replace"))
