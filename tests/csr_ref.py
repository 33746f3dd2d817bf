"""Host references on CSR operands shared by the GPU tests: operands as stored for op, the oracle product with ops,
restriction to a mask's pattern, and the lower triangle of a symmetrized graph."""
import numpy as np

import oracle
from benchmark_spgemm_using_csr_b200 import capi
from benchmark_spgemm_using_csr_b200.generators import CSR, int_values, transpose


def stored(X: CSR, op) -> CSR:
    """The operand to hand to the library so that op(stored) = X: X, X^T, or X^H for OP_C.  Each op is its own
    inverse, so this is also op(X) of a stored X."""
    if op == capi.OP_N:
        return X
    t = transpose(X)
    return CSR(t.rows, t.cols, t.rowptr, t.col, np.conj(t.val)) if op == capi.OP_C else t


def product(A: CSR, B: CSR, opA=capi.OP_N, opB=capi.OP_N):
    """The oracle's op(A)*op(B) for A and B as stored: (rowptr, col, val)."""
    a, b = stored(A, opA), stored(B, opB)
    return oracle.spgemm(a.rows, a.cols, b.cols, a.rowptr, a.col, a.val, b.rowptr, b.col, b.val)


def keys(rowptr, col, n):
    """row * n + col of every entry, int64"""
    rows = np.repeat(np.arange(len(rowptr) - 1, dtype=np.int64), np.diff(np.asarray(rowptr, dtype=np.int64)))
    return rows * n + col.astype(np.int64)


def restrict(C, m, n, rpM, colM):
    """C = (rowptr, col, val) of shape m x n restricted to the pattern of M: (rowptr int64, col, val)."""
    rp, col, val = C
    keep = np.isin(keys(rp, col, n), keys(rpM, colM, n))
    rows = np.repeat(np.arange(m, dtype=np.int64), np.diff(np.asarray(rp, dtype=np.int64)))
    rowptr = np.zeros(m + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows[keep], minlength=m), out=rowptr[1:])
    return rowptr, col[keep], val[keep]


def lower_triangle(A: CSR) -> CSR:
    """The entries of A strictly below the diagonal."""
    rows = np.repeat(np.arange(A.rows, dtype=np.int64), np.diff(A.rowptr.astype(np.int64)))
    keep = A.col < rows
    rowptr = np.zeros(A.rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows[keep], minlength=A.rows), out=rowptr[1:])
    return CSR(A.rows, A.cols, rowptr.astype(np.int32), A.col[keep].astype(np.int32), A.val[keep])


def symmetrize(A: CSR) -> CSR:
    """The pattern of A + A^T (square A), with integer values."""
    k = np.union1d(keys(A.rowptr, A.col, A.cols), (A.col.astype(np.int64) * A.cols +
                                                   np.repeat(np.arange(A.rows), np.diff(A.rowptr.astype(np.int64)))))
    rowptr = np.zeros(A.rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(k // A.cols, minlength=A.rows), out=rowptr[1:])
    return CSR(A.rows, A.cols, rowptr.astype(np.int32), (k % A.cols).astype(np.int32), int_values(k.size, 3))
