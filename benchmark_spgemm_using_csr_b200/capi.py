"""ctypes binding of the C-ABI in include/bhsparse_b200.h.

Loads benchmark_spgemm_using_csr_b200/lib/libbhsparse_b200.so.  There is NO CPU
fallback: if the library is missing or no sm_100 GPU is visible every compute
entry point raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libbhsparse_b200.so")

SUCCESS = 0
ERR_INVALID = -1
ERR_CUDA = -2
ERR_OVERFLOW = -3
ERR_ALLOC = -4
ERR_NO_DEVICE = -5
DTYPE_F32 = 0
DTYPE_F64 = 1
DTYPE_NONE = 2   # structure only: row pointers and columns, no values
DTYPE_C64 = 4    # complex64: two float32 (re, im) per value (3 is not a type)
OP_N = 0
OP_T = 1
OP_C = 2         # conjugate transpose (complex64 operands only)
NUM_BINS = 24
NUM_MASK_BINS = 9
MASK_BIN_NAMES = ["none", "esc<=32", "w64", "w256", "w1024", "c1024", "c4096", "c16384", "global"]

SYM_BIN_NAMES = ["p=0", "p=1", "esc<=32", "g128", "g256", "g512", "g1024", "g2048", "g4096",
                 "b8192", "b16384", "b32768", "large", "range_s", "range_l"]
NUM_BIN_NAMES = ["c=0", "p=1", "esc<=32", "g64", "g128", "g256", "g512", "g1024", "g2048",
                 "b4096", "b8192", "b16384", "large", "range_s128", "range_s512", "range_l128", "range_l512", "copy_ct"]

# every symbol include/bhsparse_b200.h declares (checked by tests/test_capi_symbols.py)
EXPORTED = [
    "bhb200_create", "bhb200_destroy", "bhb200_set_stream", "bhb200_last_error", "bhb200_device_name",
    "bhb200_sm_count", "bhb200_init_data_f64", "bhb200_init_data_f32", "bhb200_init_data_device", "bhb200_operands_aliased", "bhb200_get_operands_device",
    "bhb200_warmup", "bhb200_spgemm", "bhb200_synchronize", "bhb200_get_nnzC", "bhb200_get_C_f64",
    "bhb200_get_C_f32", "bhb200_get_rowptrC_i64", "bhb200_get_C_range", "bhb200_get_C_device", "bhb200_copy_C_to_device", "bhb200_get_row_products",
    "bhb200_get_stats", "bhb200_set_profiling", "bhb200_free_mem", "bhb200_version",
    "bhb200_update_values_f64", "bhb200_update_values_f32", "bhb200_spgemm_numeric",
    "bhb200_dist_unique_id", "bhb200_dist_init", "bhb200_dist_setup_square", "bhb200_dist_spgemm",
    "bhb200_dist_get_layout", "bhb200_dist_get_block_products", "bhb200_dist_get_global_rowptr_device",
    "bhb200_dist_broadcast_ms", "bhb200_dist_finalize", "bhb200_pattern_plan_probe",
    "bhb200_init_data_op_f64", "bhb200_init_data_op_f32", "bhb200_init_data_device_op",
    "bhb200_set_mask", "bhb200_set_mask_device", "bhb200_clear_mask",
    "bhb200_init_data_structure", "bhb200_get_C_structure",
    "bhb200_init_data_op_c64", "bhb200_update_values_c64", "bhb200_get_C_c64",
]
DIST_ID_BYTES = 128


class Stats(ctypes.Structure):
    _fields_ = [
        ("m", c_int64), ("k", c_int64), ("n", c_int64), ("nnzA", c_int64), ("nnzB", c_int64),
        ("products", c_int64), ("nnzC", c_int64), ("max_row_products", c_int64),
        ("sym_bin_rows", c_int64 * NUM_BINS), ("num_bin_rows", c_int64 * NUM_BINS),
        ("ms_total", c_float), ("ms_count", c_float), ("ms_symbolic", c_float), ("ms_scan", c_float),
        ("ms_numeric", c_float),
        ("kernel_launches", c_int32), ("dtype", c_int32),
        ("bytes_algorithmic", c_int64), ("bytes_compulsory", c_int64), ("workspace_bytes", c_int64),
        ("num_bin_products", c_int64 * NUM_BINS), ("num_bin_nnzC", c_int64 * NUM_BINS),
        ("num_bin_nnzA", c_int64 * NUM_BINS),
        ("ms_sym_bin", c_float * NUM_BINS), ("ms_num_bin", c_float * NUM_BINS),
        ("direct_rows", c_int64), ("direct_retry_rows", c_int64), ("direct_ct_bytes", c_int64),
        ("direct_bin_mask", c_int64),
        ("pattern_mode", c_int64), ("pattern_nDA", c_int64), ("pattern_nDB", c_int64), ("pattern_nD", c_int64),
        ("pattern_acc_len", c_int64), ("spill_bytes", c_int64),
        ("transposed_ops", c_int64), ("ms_transpose", c_float),
        ("masked", c_int64), ("nnzM", c_int64), ("mask_bin_rows", c_int64 * NUM_MASK_BINS),
    ]

    def as_dict(self) -> dict:
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if hasattr(v, "__len__") else v
        return d


class BhsparseError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"bhsparse_b200 error {code}: {msg}")
        self.code = code


_LIB = None


def load(build_if_missing: bool = False):
    """Load the shared library (optionally building it with nvcc first)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        if build_if_missing:
            from . import build as _b
            _b.build()
        else:
            raise ImportError(
                f"{LIB_PATH} not found: run `python -m benchmark_spgemm_using_csr_b200.build` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    ctxp = c_void_p
    i32p = POINTER(c_int32)
    L.bhb200_version.restype = c_char_p
    L.bhb200_create.argtypes = [POINTER(ctxp), c_int]
    L.bhb200_destroy.argtypes = [ctxp]
    L.bhb200_set_stream.argtypes = [ctxp, c_void_p]
    L.bhb200_last_error.argtypes = [ctxp]
    L.bhb200_last_error.restype = c_char_p
    L.bhb200_device_name.argtypes = [ctxp]
    L.bhb200_device_name.restype = c_char_p
    L.bhb200_sm_count.argtypes = [ctxp]
    L.bhb200_init_data_f64.argtypes = [ctxp, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                       c_int, c_void_p, c_void_p, c_void_p]
    L.bhb200_init_data_f32.argtypes = L.bhb200_init_data_f64.argtypes
    L.bhb200_init_data_device.argtypes = [ctxp, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                          c_int, c_void_p, c_void_p, c_void_p]
    L.bhb200_init_data_op_f64.argtypes = [ctxp, c_int, c_int] + L.bhb200_init_data_f64.argtypes[1:]
    L.bhb200_init_data_op_f32.argtypes = L.bhb200_init_data_op_f64.argtypes
    L.bhb200_init_data_op_c64.argtypes = L.bhb200_init_data_op_f64.argtypes
    L.bhb200_init_data_device_op.argtypes = [ctxp, c_int, c_int, c_int] + L.bhb200_init_data_device.argtypes[2:]
    L.bhb200_init_data_structure.argtypes = [ctxp, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                                             c_void_p, c_void_p]
    L.bhb200_get_C_structure.argtypes = [ctxp, c_void_p, c_void_p]
    L.bhb200_operands_aliased.argtypes = [ctxp]
    L.bhb200_get_operands_device.argtypes = [ctxp, POINTER(c_int32)] + [POINTER(c_void_p)] * 6
    L.bhb200_set_mask.argtypes = [ctxp, c_int, c_void_p, c_void_p]
    L.bhb200_set_mask_device.argtypes = [ctxp, c_int, c_void_p, c_void_p]
    L.bhb200_clear_mask.argtypes = [ctxp]
    L.bhb200_warmup.argtypes = [ctxp]
    L.bhb200_spgemm.argtypes = [ctxp]
    L.bhb200_synchronize.argtypes = [ctxp]
    L.bhb200_update_values_f64.argtypes = [ctxp, c_void_p, c_void_p]
    L.bhb200_update_values_f32.argtypes = [ctxp, c_void_p, c_void_p]
    L.bhb200_update_values_c64.argtypes = [ctxp, c_void_p, c_void_p]
    L.bhb200_spgemm_numeric.argtypes = [ctxp]
    L.bhb200_get_nnzC.argtypes = [ctxp]
    L.bhb200_get_nnzC.restype = c_int64
    L.bhb200_get_C_f64.argtypes = [ctxp, c_void_p, c_void_p, c_void_p]
    L.bhb200_get_C_f32.argtypes = [ctxp, c_void_p, c_void_p, c_void_p]
    L.bhb200_get_C_c64.argtypes = [ctxp, c_void_p, c_void_p, c_void_p]
    L.bhb200_get_rowptrC_i64.argtypes = [ctxp, c_void_p]
    L.bhb200_get_C_range.argtypes = [ctxp, c_int64, c_int64, c_void_p, c_void_p]
    L.bhb200_get_C_device.argtypes = [ctxp, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p)]
    L.bhb200_copy_C_to_device.argtypes = [ctxp, c_void_p, c_void_p, c_void_p]
    L.bhb200_get_row_products.argtypes = [ctxp, c_void_p]
    L.bhb200_get_stats.argtypes = [ctxp, POINTER(Stats)]
    L.bhb200_set_profiling.argtypes = [ctxp, c_int]
    L.bhb200_free_mem.argtypes = [ctxp]
    L.bhb200_dist_unique_id.argtypes = [c_void_p]
    L.bhb200_dist_init.argtypes = [ctxp, c_int, c_int, c_void_p]
    L.bhb200_dist_setup_square.argtypes = [ctxp, c_int, c_int, c_int, c_int64, c_void_p, c_void_p, c_void_p]
    L.bhb200_dist_spgemm.argtypes = [ctxp]
    L.bhb200_dist_get_layout.argtypes = [ctxp] + [POINTER(c_int64)] * 5
    L.bhb200_dist_get_block_products.argtypes = [ctxp, POINTER(c_int64)]
    L.bhb200_dist_get_global_rowptr_device.argtypes = [ctxp, POINTER(c_void_p)]
    L.bhb200_dist_broadcast_ms.argtypes = [ctxp, POINTER(c_float)]
    L.bhb200_dist_finalize.argtypes = [ctxp]
    L.bhb200_pattern_plan_probe.argtypes = [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]
    for name in EXPORTED:
        f = getattr(L, name)
        if f.restype is c_int:  # default
            f.restype = c_int
    _LIB = L
    return L


def check(lib, ctx, code: int):
    if code != SUCCESS:
        msg = lib.bhb200_last_error(ctx)
        raise BhsparseError(code, msg.decode() if msg else "")
