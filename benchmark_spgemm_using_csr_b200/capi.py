"""ctypes binding of the C-ABI in include/bhsparse_b200.h, and `Context`, the Python owner of one bhb200_ctx.

Loads benchmark_spgemm_using_csr_b200/lib/libbhsparse_b200.so.  There is NO CPU
fallback: if the library is missing or no sm_100 GPU is visible every compute
entry point raises.  torch is imported only by the methods that take or return device tensors.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_void_p

import numpy as np

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
DTYPE_C128 = 5   # complex128: two float64 (re, im) per value, 16-byte aligned
OP_N = 0
OP_T = 1
OP_C = 2         # conjugate transpose (complex operands only)
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
    "bhb200_init_data_op_c128", "bhb200_update_values_c128", "bhb200_get_C_c128",
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
    L.bhb200_init_data_op_c128.argtypes = L.bhb200_init_data_op_f64.argtypes
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
    L.bhb200_update_values_c128.argtypes = [ctxp, c_void_p, c_void_p]
    L.bhb200_spgemm_numeric.argtypes = [ctxp]
    L.bhb200_get_nnzC.argtypes = [ctxp]
    L.bhb200_get_nnzC.restype = c_int64
    L.bhb200_get_C_f64.argtypes = [ctxp, c_void_p, c_void_p, c_void_p]
    L.bhb200_get_C_f32.argtypes = [ctxp, c_void_p, c_void_p, c_void_p]
    L.bhb200_get_C_c64.argtypes = [ctxp, c_void_p, c_void_p, c_void_p]
    L.bhb200_get_C_c128.argtypes = [ctxp, c_void_p, c_void_p, c_void_p]
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


# BHB200_DTYPE_* of a valued product -> (suffix of bhb200_init_data_op_*, bhb200_update_values_* and
# bhb200_get_C_*; numpy and torch dtype name)
VALUE_TYPES = {DTYPE_F32: ("f32", "float32"), DTYPE_F64: ("f64", "float64"), DTYPE_C64: ("c64", "complex64"),
               DTYPE_C128: ("c128", "complex128")}
_DTYPE_OF_NAME = {name: dt for dt, (_, name) in VALUE_TYPES.items()}


def dtype_of(x) -> int:
    """BHB200_DTYPE_* of a numpy or torch value array, dtype or dtype name.  Other value types raise, never
    converted."""
    name = str(getattr(x, "dtype", x)).removeprefix("torch.")
    if name not in _DTYPE_OF_NAME:
        raise BhsparseError(ERR_INVALID, f"{name} values are not supported")
    return _DTYPE_OF_NAME[name]


def op_shape(rows: int, cols: int, op: int):
    """Shape of op(X) for X of shape (rows, cols), and of X for op(X) of that shape."""
    return (cols, rows) if op != OP_N else (rows, cols)


def op_dims(A, B, opA: int = OP_N, opB: int = OP_N):
    """(m, k, n) of C = op(A)*op(B) for A and B as stored (anything with .rows and .cols)."""
    m, k = op_shape(A.rows, A.cols, opA)
    return m, k, op_shape(B.rows, B.cols, opB)[1]


class DevicePtr:
    """A borrowed device pointer as a __cuda_array_interface__ object (typestr e.g. "<i4"), for torch.as_tensor."""

    def __init__(self, ptr: int, numel: int, typestr: str):
        self.__cuda_array_interface__ = {"shape": (numel,), "typestr": typestr, "data": (ptr, False), "version": 2}


def device_view(ptr: int, numel: int, dtype: str, device):
    """A torch tensor over `numel` elements of device memory at `ptr` that the library owns: no copy, valid until
    the owning context changes or frees it."""
    import torch
    if numel == 0:
        return torch.empty(0, dtype=getattr(torch, dtype), device=device)
    return torch.as_tensor(DevicePtr(ptr, numel, np.dtype(dtype).str), device=device)


def _ptr(a):
    """Address of a numpy array, or NULL for None."""
    return None if a is None else c_void_p(a.ctypes.data)


def _dptr(t):
    """Address of a torch tensor, or NULL for None."""
    return None if t is None else c_void_p(t.data_ptr())


class Context:
    """One bhb200_ctx.  Every call raises BhsparseError on a nonzero return.  Operands, values and device masks
    handed to it stay referenced until the next init or close, so borrowed device arrays outlive their use.

    m, n: the shape of C; dtype: the BHB200_DTYPE_* of the operands."""

    def __init__(self, device: int = 0):
        self.lib = load()
        self.ctx = c_void_p()
        self.device = device
        self.m = self.n = 0
        self.dtype = DTYPE_F64
        self._keep = []
        self._check(self.lib.bhb200_create(ctypes.byref(self.ctx), device))

    def close(self):
        if self.ctx:
            self.lib.bhb200_destroy(self.ctx)
            self.ctx = c_void_p()
        self._keep = []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, code: int):
        check(self.lib, self.ctx, code)

    # -- operands ---------------------------------------------------------------------------------------
    def init(self, A, B, opA: int = OP_N, opB: int = OP_N, dtype: int | None = None, same: bool = False):
        """Host CSR operands as stored; C = op(A)*op(B).  dtype None takes the value type from A.val, DTYPE_NONE
        passes no values.  same=True passes A's arrays for B (the library uploads them once); otherwise B's values
        are a copy of their own."""
        m, k, n = op_dims(A, B, opA, opB)
        dt = dtype_of(A.val) if dtype is None else dtype
        a = [np.ascontiguousarray(A.rowptr, np.int32), np.ascontiguousarray(A.col, np.int32)]
        b = a if same else [np.ascontiguousarray(B.rowptr, np.int32), np.ascontiguousarray(B.col, np.int32)]
        if dt == DTYPE_NONE:
            self._keep = [a, b]
            self._check(self.lib.bhb200_init_data_structure(self.ctx, opA, opB, m, k, n, A.nnz, *map(_ptr, a), B.nnz,
                                                            *map(_ptr, b)))
        else:
            suffix, name = VALUE_TYPES[dt]
            va = np.ascontiguousarray(A.val, name)
            vb = va if same else np.array(B.val, name)
            self._keep = [a, b, va, vb]
            fn = getattr(self.lib, "bhb200_init_data_op_" + suffix)
            self._check(fn(self.ctx, opA, opB, m, k, n, A.nnz, _ptr(va), *map(_ptr, a), B.nnz, _ptr(vb), *map(_ptr, b)))
        self.m, self.n, self.dtype = m, n, dt

    def init_device(self, A, B, m: int, k: int, n: int, opA: int = OP_N, opB: int = OP_N, dtype: int | None = None):
        """Borrowed device operands: A, B = (rowptr, col, val) torch tensors as stored; op(A) is m x k, op(B) k x n.
        dtype None takes the value type from A's values.  A val of None is passed as a NULL value pointer (for
        DTYPE_NONE)."""
        dt = dtype_of(A[2]) if dtype is None else dtype
        self._keep = [A, B]
        self._check(self.lib.bhb200_init_data_device_op(self.ctx, dt, opA, opB, m, k, n, int(A[1].numel()), _dptr(A[2]),
                                                        _dptr(A[0]), _dptr(A[1]), int(B[1].numel()), _dptr(B[2]),
                                                        _dptr(B[0]), _dptr(B[1])))
        self.m, self.n, self.dtype = m, n, dt

    def set_mask(self, rowptr, col):
        """C = M .* (op(A)*op(B)) on the pattern of M, host arrays (copied by the library)."""
        rp, c = np.ascontiguousarray(rowptr, np.int32), np.ascontiguousarray(col, np.int32)
        self._check(self.lib.bhb200_set_mask(self.ctx, int(c.size), _ptr(rp), _ptr(c) if c.size else None))

    def set_mask_device(self, rowptr, col):
        """The mask from borrowed int32 device tensors."""
        self._keep.append((rowptr, col))
        self._check(self.lib.bhb200_set_mask_device(self.ctx, int(col.numel()), _dptr(rowptr), _dptr(col)))

    def clear_mask(self):
        self._check(self.lib.bhb200_clear_mask(self.ctx))

    # -- products ---------------------------------------------------------------------------------------
    def spgemm(self) -> int:
        """The product; returns nnz(C)."""
        self._check(self.lib.bhb200_spgemm(self.ctx))
        return int(self.lib.bhb200_get_nnzC(self.ctx))

    def update_values(self, va, vb):
        """New host values of A and B as stored (None: unchanged), same patterns."""
        name = VALUE_TYPES[self.dtype][1]
        va, vb = (None if v is None else np.ascontiguousarray(v, name) for v in (va, vb))
        self._keep.append((va, vb))
        fn = getattr(self.lib, "bhb200_update_values_" + VALUE_TYPES[self.dtype][0])
        self._check(fn(self.ctx, _ptr(va), _ptr(vb)))

    def spgemm_numeric(self):
        self._check(self.lib.bhb200_spgemm_numeric(self.ctx))

    # -- results ----------------------------------------------------------------------------------------
    def rowptr64_host(self) -> np.ndarray:
        out = np.empty(self.m + 1, dtype=np.int64)
        self._check(self.lib.bhb200_get_rowptrC_i64(self.ctx, _ptr(out)))
        return out

    def get_C_range(self, first: int, count: int):
        """Entries [first, first+count) of C as host arrays (col int32, val); val is None for structure-only."""
        col = np.empty(max(count, 0), dtype=np.int32)
        val = None if self.dtype == DTYPE_NONE else np.empty(max(count, 0), dtype=VALUE_TYPES[self.dtype][1])
        self._check(self.lib.bhb200_get_C_range(self.ctx, int(first), int(count), _ptr(col), _ptr(val)))
        return col, val

    def C(self):
        """C on the host: (rowptr int64, col int32, val), val None for structure-only; any nnz(C)."""
        rp = self.rowptr64_host()
        return (rp, *self.get_C_range(0, int(rp[-1])))

    def C_device(self):
        """Copies of C on the device as torch tensors (rowptr int64, col int32, val); val None for structure-only.
        The copy is complete when this returns, so any stream may use them."""
        import torch
        nnz = int(self.lib.bhb200_get_nnzC(self.ctx))
        dev = torch.device("cuda", self.device)
        rowptr = torch.empty(self.m + 1, dtype=torch.int64, device=dev)
        col = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
        val = None if self.dtype == DTYPE_NONE else \
            torch.empty(max(nnz, 1), dtype=getattr(torch, VALUE_TYPES[self.dtype][1]), device=dev)
        self._check(self.lib.bhb200_copy_C_to_device(self.ctx, _dptr(rowptr), _dptr(col), _dptr(val)))
        return rowptr, col[:nnz], None if val is None else val[:nnz]

    def operands(self):
        """((m, k, n), op(A), op(B)) as the library holds them: (rowptr, col, val) views of its device memory
        (device_view), val None for structure-only."""
        dims = (c_int32 * 6)()
        ptrs = [c_void_p() for _ in range(6)]
        self._check(self.lib.bhb200_get_operands_device(self.ctx, dims, *(ctypes.byref(p) for p in ptrs)))
        self._check(self.lib.bhb200_synchronize(self.ctx))
        m, k, n, nnzA, nnzB, dt = (int(x) for x in dims)
        dev = f"cuda:{self.device}"

        def csr(rows, nnz, rp, col, val):
            return (device_view(rp.value, rows + 1, "int32", dev), device_view(col.value, nnz, "int32", dev),
                    None if dt == DTYPE_NONE else device_view(val.value, nnz, VALUE_TYPES[dt][1], dev))
        return (m, k, n), csr(m, nnzA, *ptrs[:3]), csr(k, nnzB, *ptrs[3:])

    def stats(self) -> dict:
        st = Stats()
        self._check(self.lib.bhb200_get_stats(self.ctx, ctypes.byref(st)))
        return st.as_dict()

    def error(self) -> str:
        return self.lib.bhb200_last_error(self.ctx).decode()

    def aliased(self) -> int:
        """1 if A and B came from the same arrays and were uploaded once."""
        return int(self.lib.bhb200_operands_aliased(self.ctx))

    def set_stream(self, cuda_stream_ptr: int):
        self._check(self.lib.bhb200_set_stream(self.ctx, c_void_p(cuda_stream_ptr)))

    def set_profiling(self, on: bool):
        self._check(self.lib.bhb200_set_profiling(self.ctx, 1 if on else 0))
