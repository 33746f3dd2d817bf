"""Python mirror of the reference's `bhsparse` class (SpGEMM_cuda/bhsparse.h:17-34)
over the C-ABI: same method names, argument order (val, rowptr, colidx) and
`int` error convention (0 == BHSPARSE_SUCCESS, common.h:26), so that the parity
tests read like the reference driver (main.cu:104-135).

    bh = bhsparse()
    bh.initPlatform(platforms)          # platforms[BHSPARSE_CUDA] = True
    bh.initData(m, k, n, nnzA, valA, rowptrA, colA, nnzB, valB, rowptrB, colB, rowptrC)
    bh.warmup(); bh.spgemm()
    nnzC = bh.get_nnzC(); bh.get_C(colC, valC)
    bh.free_mem(); bh.freePlatform()

Host arrays are numpy (or anything exposing a writable buffer of the right
dtype); the value dtype (float32/float64/complex64/complex128) is taken from valA -- the reference
needs a recompile for that (common.h:31, README.md:84-86).  A complex valB of another dtype than
valA, or a complex and a real operand, is refused (ERR_INVALID), never converted.  With valA and valB both
None the product is structure-only (BHB200_DTYPE_NONE): C has row pointers and
columns, and get_C takes None for the values.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import capi

BHSPARSE_SUCCESS = 0
NUM_PLATFORMS = 9       # common.h:33
BHSPARSE_CUDA = 1       # common.h:36


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _suffix(dt) -> str | None:
    """init_data_op / update_values / get_C entry-point suffix of a value dtype, None if unsupported"""
    try:
        return capi.VALUE_TYPES[capi.dtype_of(dt)][0]
    except capi.BhsparseError:
        return None


def _op(trans) -> int:
    """transA / transB: False / "N", True / "T", or "C" (conjugate transpose, complex values only)"""
    if trans == "C":
        return capi.OP_C
    return capi.OP_T if trans in (True, "T") else capi.OP_N


class bhsparse:
    def __init__(self, device: int = 0, verbose: bool = False):
        self._lib = None
        self._ctx = ctypes.c_void_p(None)
        self._device = device
        self._verbose = verbose
        self._rowptrC = None
        self._dtype = None
        self._structure = False   # structure-only operands (no values)
        self._m = 0

    # -- platform (bhsparse.h:96-148) ---------------------------------------
    def initPlatform(self, spgemm_platform) -> int:
        if len(spgemm_platform) < NUM_PLATFORMS or not spgemm_platform[BHSPARSE_CUDA]:
            return capi.ERR_INVALID          # only the CUDA platform exists here
        self._lib = capi.load()
        ctx = ctypes.c_void_p(None)
        err = self._lib.bhb200_create(ctypes.byref(ctx), self._device)
        if err == BHSPARSE_SUCCESS:
            self._ctx = ctx
            if self._verbose:               # bhsparse_cuda.h:108-110
                print(f"Device [{self._device}] {self._lib.bhb200_device_name(ctx).decode()}. "
                      f"{self._lib.bhb200_sm_count(ctx)} SMs.")
        return err

    def freePlatform(self) -> int:
        if not self._ctx:
            return BHSPARSE_SUCCESS
        err = self._lib.bhb200_destroy(self._ctx)
        self._ctx = ctypes.c_void_p(None)
        return err

    # -- data (bhsparse.h:180-258) -------------------------------------------
    def initData(self, m, k, n, nnzA, csrValA, csrRowPtrA, csrColIndA,
                 nnzB, csrValB, csrRowPtrB, csrColIndB, csrRowPtrC, transA=False, transB=False) -> int:
        """C = op(A)*op(B): m, k, n are the dimensions of op(A) (m x k) and op(B) (k x n); with
        transA / transB the arrays hold A / B as stored, i.e. k x m / n x k (bhb200_init_data_op_*).
        transA / transB = "C": conjugate transpose (complex64 or complex128 values).
        csrValA and csrValB both None: structure-only product (bhb200_init_data_structure)."""
        if not self._ctx:
            return capi.ERR_INVALID
        structure = csrValA is None and csrValB is None
        if structure:
            dt = None
        elif csrValA is None or csrValB is None:
            return capi.ERR_INVALID
        else:
            valA = np.ascontiguousarray(csrValA)
            dt = valA.dtype
            if _suffix(dt) is None:
                return capi.ERR_INVALID
            dtB = np.asarray(csrValB).dtype
            if dtB != dt and (dt.kind == "c" or dtB.kind == "c"):   # (no mixed complex operands: never converted)
                return capi.ERR_INVALID
            fn = getattr(self._lib, "bhb200_init_data_op_" + _suffix(dt))
            valB = np.ascontiguousarray(csrValB, dtype=dt)
        rpA = np.ascontiguousarray(csrRowPtrA, dtype=np.int32)
        cA = np.ascontiguousarray(csrColIndA, dtype=np.int32)
        rpB = np.ascontiguousarray(csrRowPtrB, dtype=np.int32)
        cB = np.ascontiguousarray(csrColIndB, dtype=np.int32)
        opA, opB = _op(transA), _op(transB)
        rows_a = capi.op_shape(m, k, opA)[0]   # rows of A / B as stored
        rows_b = capi.op_shape(k, n, opB)[0]
        if rpA.size != rows_a + 1 or rpB.size != rows_b + 1 or cA.size < nnzA or cB.size < nnzB:
            return capi.ERR_INVALID
        if csrRowPtrC is not None and (csrRowPtrC.dtype != np.int32 or csrRowPtrC.size < m + 1):
            return capi.ERR_INVALID
        self._rowptrC = csrRowPtrC           # caller-owned, written by get_C (main.cu:100)
        self._dtype = dt
        self._structure = structure
        self._m = m
        # (the same host arrays for A and B stay the same objects here, so the library can upload them once)
        if structure:
            return self._lib.bhb200_init_data_structure(self._ctx, opA, opB, m, k, n, nnzA, _ptr(rpA), _ptr(cA), nnzB,
                                                        _ptr(rpB), _ptr(cB))
        return fn(self._ctx, opA, opB, m, k, n, nnzA, _ptr(valA), _ptr(rpA), _ptr(cA), nnzB, _ptr(valB), _ptr(rpB), _ptr(cB))

    def aliased_operands(self) -> bool:
        """True if initData got the same host arrays for A and B and uploaded them once."""
        return bool(self._ctx) and bool(self._lib.bhb200_operands_aliased(self._ctx))

    def warmup(self) -> int:
        return self._lib.bhb200_warmup(self._ctx) if self._ctx else capi.ERR_INVALID

    # -- the hot path (bhsparse.h:260-339) -------------------------------------
    def spgemm(self) -> int:
        if not self._ctx:
            return capi.ERR_INVALID
        err = self._lib.bhb200_spgemm(self._ctx)
        # create_C leaves rowptrC in the caller's array at the end of spgemm() (bhsparse_cuda.h:2787-2808)
        if err == BHSPARSE_SUCCESS and self._rowptrC is not None and 0 <= self.get_nnzC() <= 0x7fffffff:
            err = self._lib.bhb200_get_C_structure(self._ctx, ctypes.c_void_p(self._rowptrC.ctypes.data), None)
        if err == BHSPARSE_SUCCESS and self._verbose:
            st = self.stats()
            t = st["ms_total"]
            gf = 2.0 * st["products"] / (t * 1.0e6) if t > 0 else 0.0
            print(f"STAGE 1 time: {st['ms_count']:.4f} ms.\nSTAGE 2 time: {st['ms_symbolic']:.4f} ms.\n"
                  f"STAGE 3 time: {st['ms_scan']:.4f} ms.\nSTAGE 4 time: {st['ms_numeric']:.4f} ms.\n"
                  f"[ CUDA ] SpGEMM time: {t:.4f} ms. Gflops = {gf:.4f}")    # bhsparse.h:286-289
        return err

    def get_nnzC(self) -> int:
        return int(self._lib.bhb200_get_nnzC(self._ctx)) if self._ctx else -1

    def get_C(self, csrColIndC, csrValC) -> int:
        """Columns (and values) of C; csrValC None skips the values, and must be None for a structure-only product."""
        if not self._ctx:
            return capi.ERR_INVALID
        if csrValC is not None and (self._structure or csrValC.dtype != self._dtype):
            return capi.ERR_INVALID
        if csrColIndC is not None and csrColIndC.dtype != np.int32:
            return capi.ERR_INVALID
        rp = ctypes.c_void_p(self._rowptrC.ctypes.data) if self._rowptrC is not None else None
        cp = ctypes.c_void_p(csrColIndC.ctypes.data) if csrColIndC is not None else None
        if csrValC is None:
            return self._lib.bhb200_get_C_structure(self._ctx, rp, cp)
        fn = getattr(self._lib, "bhb200_get_C_" + _suffix(self._dtype))
        return fn(self._ctx, rp, cp, ctypes.c_void_p(csrValC.ctypes.data))

    def free_mem(self) -> int:
        return self._lib.bhb200_free_mem(self._ctx) if self._ctx else BHSPARSE_SUCCESS

    # -- additions (no reference counterpart) --------------------------------------
    def update_values(self, csrValA=None, csrValB=None) -> int:
        """New values for A and/or B, same patterns (include/bhsparse_b200.h: bhb200_update_values_*)."""
        if not self._ctx:
            return capi.ERR_INVALID
        for v in (csrValA, csrValB):
            if v is not None and (v.dtype != self._dtype or not v.flags.c_contiguous):
                return capi.ERR_INVALID
        fn = getattr(self._lib, "bhb200_update_values_" + _suffix(self._dtype))
        ap = ctypes.c_void_p(csrValA.ctypes.data) if csrValA is not None else None
        bp = ctypes.c_void_p(csrValB.ctypes.data) if csrValB is not None else None
        return fn(self._ctx, ap, bp)

    def spgemm_numeric(self) -> int:
        """Values of C again after update_values; structure of C reused (bhb200_spgemm_numeric)."""
        return self._lib.bhb200_spgemm_numeric(self._ctx) if self._ctx else capi.ERR_INVALID

    def set_mask(self, csrRowPtrM, csrColIndM) -> int:
        """Masked products C = M .* (op(A)*op(B)) on the pattern of M (bhb200_set_mask; host arrays,
        copied).  Call after initData; initData clears it."""
        if not self._ctx:
            return capi.ERR_INVALID
        rp = np.ascontiguousarray(csrRowPtrM, dtype=np.int32)
        col = np.ascontiguousarray(csrColIndM, dtype=np.int32)
        if rp.size != self._m + 1:
            return capi.ERR_INVALID
        return self._lib.bhb200_set_mask(self._ctx, int(col.size), _ptr(rp), _ptr(col) if col.size else None)

    def clear_mask(self) -> int:
        return self._lib.bhb200_clear_mask(self._ctx) if self._ctx else capi.ERR_INVALID

    def get_rowptrC_i64(self) -> np.ndarray:
        out = np.empty(self._m + 1, dtype=np.int64)
        capi.check(self._lib, self._ctx, self._lib.bhb200_get_rowptrC_i64(self._ctx, ctypes.c_void_p(out.ctypes.data)))
        return out

    def get_C_range(self, first: int, count: int):
        """Entries [first, first+count) of (colC, valC): piecewise access for results beyond INT32_MAX.
        valC is None for a structure-only product."""
        col = np.empty(max(count, 0), dtype=np.int32)
        val = None if self._structure else np.empty(max(count, 0), dtype=self._dtype)
        capi.check(self._lib, self._ctx, self._lib.bhb200_get_C_range(
            self._ctx, int(first), int(count), ctypes.c_void_p(col.ctypes.data),
            ctypes.c_void_p(val.ctypes.data) if val is not None else None))
        return col, val

    def get_row_products(self) -> np.ndarray:
        out = np.empty(max(self._m, 1), dtype=np.int32)
        capi.check(self._lib, self._ctx, self._lib.bhb200_get_row_products(self._ctx, ctypes.c_void_p(out.ctypes.data)))
        return out[:self._m]

    def stats(self) -> dict:
        st = capi.Stats()
        capi.check(self._lib, self._ctx, self._lib.bhb200_get_stats(self._ctx, ctypes.byref(st)))
        return st.as_dict()

    def last_error(self) -> str:
        return self._lib.bhb200_last_error(self._ctx).decode() if self._ctx else ""

    def __del__(self):
        try:
            if self._ctx:
                self.freePlatform()
        except Exception:
            pass


def spgemm(A, B, device: int = 0, return_stats: bool = False, return_row_products: bool = False,
           transA: bool = False, transB: bool = False, mask=None, structure_only: bool = False):
    """Convenience driver following main.cu:104-135: C = op(A)*op(B) for two
    generators.CSR operands (op = transpose with transA / transB); returns
    (rowptrC int32, colC int32, valC).  Values float32, float64, complex64 or complex128
    (transA / transB may then be "C", the conjugate transpose); complex operands of two types, or a complex and a
    real one, are refused.  mask: a generators.CSR or (rowptr, col)
    whose pattern restricts C (masked product, bhb200_set_mask).  structure_only:
    the pattern of C alone, from the operands' patterns (valC is None)."""
    platforms = [False] * NUM_PLATFORMS
    platforms[BHSPARSE_CUDA] = True
    bh = bhsparse(device)
    if not structure_only:
        ta, tb = np.asarray(A.val).dtype, np.asarray(B.val).dtype
        if ta != tb and (ta.kind == "c" or tb.kind == "c"):
            raise capi.BhsparseError(capi.ERR_INVALID, f"mixed value types are not supported: {ta} A with {tb} B")
    m, k, n = capi.op_dims(A, B, _op(transA), _op(transB))
    rowptrC = np.zeros(m + 1, dtype=np.int32)

    def ok(err, what):
        if err != BHSPARSE_SUCCESS:
            msg = bh.last_error()
            bh.freePlatform()
            raise capi.BhsparseError(err, f"{what}: {msg}")

    ok(bh.initPlatform(platforms), "initPlatform")
    ok(bh.initData(m, k, n, A.nnz, None if structure_only else A.val, A.rowptr, A.col,
                   B.nnz, None if structure_only else B.val, B.rowptr, B.col, rowptrC, transA, transB), "initData")
    if mask is not None:
        rpM, colM = (mask.rowptr, mask.col) if hasattr(mask, "rowptr") else mask
        ok(bh.set_mask(rpM, colM), "set_mask")
    ok(bh.spgemm(), "spgemm")
    nnzC = bh.get_nnzC()
    colC = np.empty(max(nnzC, 0), dtype=np.int32)
    valC = None if structure_only else np.empty(max(nnzC, 0), dtype=A.val.dtype)
    ok(bh.get_C(colC, valC), "get_C")
    st = bh.stats() if return_stats else None
    prods = bh.get_row_products() if return_row_products else None
    ok(bh.free_mem(), "free_mem")
    ok(bh.freePlatform(), "freePlatform")
    out = (rowptrC, colC, valC)
    if return_stats:
        out += (st,)
    if return_row_products:
        out += (prods,)
    return out
