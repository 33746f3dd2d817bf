"""The exact reference of complex128 products through the real embedding in f64, and complex128 value generators.

The embedding is that of tests/complex_ref.py (see its docstring), with f64 operands: A_e (2m x 2k) has, in row i,
ar_it at column 2t and -ai_it at 2t+1, and in row m+i, ai_it at 2t and ar_it at 2t+1; B_e (2k x n) has br_t. in
row 2t and bi_t. in row 2t+1.  Rows i and m+i of A_e*B_e are Re and Im of row i of A*B with 2p products per entry,
so the quad-precision reference of tests/exact_ref.c and its f64 bound (p -> 2p) check every component.
complex_ref.embed works in f32 (complex64 values) and stays as it is; this module is its f64 counterpart."""
import numpy as np

import exact_ref as xr
from benchmark_spgemm_using_csr_b200.generators import CSR
from complex_ref import conj_transpose  # noqa: F401 (X^H on the host does not depend on the value type)

C128, F64 = np.complex128, np.float64


def embed(A: CSR, B: CSR):
    """(A_e, B_e) as float64 CSRs, see the module docstring."""
    a = np.asarray(A.val, C128)
    b = np.asarray(B.val, C128)
    lens = np.diff(A.rowptr.astype(np.int64))
    rp = np.zeros(2 * A.rows + 1, np.int64)
    rp[1:] = np.cumsum(np.concatenate([2 * lens, 2 * lens]))
    col = np.stack([2 * A.col.astype(np.int64), 2 * A.col.astype(np.int64) + 1], axis=1).reshape(-1)
    re = np.stack([a.real, -a.imag], axis=1).reshape(-1)
    im = np.stack([a.imag, a.real], axis=1).reshape(-1)
    Ae = CSR(2 * A.rows, 2 * A.cols, rp.astype(np.int32), np.concatenate([col, col]).astype(np.int32),
             np.concatenate([re, im]).astype(F64))
    blen = np.diff(B.rowptr.astype(np.int64))
    brp = np.zeros(2 * B.rows + 1, np.int64)
    brp[1::2] = blen
    brp[2::2] = blen
    brp = np.cumsum(brp)
    src = np.repeat(np.arange(B.rows), blen)
    start = np.repeat(brp[0:-1:2], blen) + (np.arange(B.nnz) - np.repeat(B.rowptr[:-1].astype(np.int64), blen))
    bcol = np.empty(2 * B.nnz, np.int32)
    bval = np.empty(2 * B.nnz, F64)
    bcol[start], bcol[start + blen[src]] = B.col, B.col
    bval[start], bval[start + blen[src]] = b.real, b.imag
    return Ae, CSR(2 * B.rows, B.cols, brp.astype(np.int32), bcol, bval)


def product(lib, A: CSR, B: CSR):
    """(Re, Im): the exact references of the two components of A*B (complex128 values), each a dict of
    exact_ref.product with C's structure, dtype float64 and p = 2 x the products of the entry."""
    ref = xr.product(lib, *embed(A, B))
    rp, m = ref["rowptr"], A.rows
    half = int(rp[m])
    out = []
    for sl, base in ((slice(0, half), 0), (slice(half, None), half)):
        d = {k: v[sl] for k, v in ref.items() if isinstance(v, np.ndarray) and k != "rowptr"}
        d["rowptr"] = (rp[:m + 1] if base == 0 else rp[m:] - base).astype(np.int64)
        d["dtype"] = F64
        out.append(d)
    return out


# complex128 values: real parts from the f64 generators of exact_ref with `seed`, imaginary parts with seed + 1000
def tier1(nnz, q, seed):
    return (xr.tier1(nnz, q, seed, F64) + 1j * xr.tier1(nnz, q, seed + 1000, F64)).astype(C128)


def tier2(nnz, seed):
    return (xr.tier2(nnz, seed, F64) + 1j * xr.tier2(nnz, seed + 1000, F64)).astype(C128)


def tier3(nnz, seed):
    """specials in either component: +-inf, NaN, zeros and subnormal products (inf * 0 is NaN)"""
    out = np.empty(nnz, C128)
    out.real, out.imag = xr.tier3(nnz, seed, F64), xr.tier3(nnz, seed + 1000, F64)
    return out


def paired(A: CSR, B: CSR, seed):
    """exact_ref.paired per component: the same structure and scale factors for both, so C2 cancels far below the
    sum of the product magnitudes."""
    Ar, Br = xr.paired(CSR(A.rows, A.cols, A.rowptr, A.col, A.val.real.astype(F64)),
                       CSR(B.rows, B.cols, B.rowptr, B.col, B.val.real.astype(F64)), seed)
    Ai, Bi = xr.paired(CSR(A.rows, A.cols, A.rowptr, A.col, A.val.imag.astype(F64)),
                       CSR(B.rows, B.cols, B.rowptr, B.col, B.val.imag.astype(F64)), seed)
    return (CSR(Ar.rows, Ar.cols, Ar.rowptr, Ar.col, (Ar.val + 1j * Ai.val).astype(C128)),
            CSR(Br.rows, Br.cols, Br.rowptr, Br.col, (Br.val + 1j * Bi.val).astype(C128)))
