"""The exact reference of complex64 products through the real embedding, and complex value generators.

Each component of a complex product entry is a real sum of 2p real products (the value contract of
include/bhsparse_b200.h):
    Re c_ij = sum_t ar_it*br_tj + (-ai_it)*bi_tj,     Im c_ij = sum_t ar_it*bi_tj + ai_it*br_tj.
`embed` writes them as one real product: A_e (2m x 2k) has, in row i, ar_it at column 2t and -ai_it at 2t+1, and in
row m+i, ai_it at 2t and ar_it at 2t+1; B_e (2k x n) has br_t. in row 2t and bi_t. in row 2t+1.  Rows i and m+i of
A_e*B_e are Re and Im of row i of A*B, with the structure of A*B and 2p products per entry, so the quad-precision
reference of tests/exact_ref.c and its bound (p -> 2p) check every component."""
import numpy as np

import exact_ref as xr
from benchmark_spgemm_using_csr_b200.generators import CSR


def conj_transpose(X: CSR) -> CSR:
    """X^H on the host (stable: rows of X^H in increasing column order)."""
    rows = np.repeat(np.arange(X.rows, dtype=np.int64), np.diff(X.rowptr.astype(np.int64)))
    perm = np.argsort(X.col, kind="stable")
    rowptr = np.zeros(X.cols + 1, dtype=np.int64)
    np.cumsum(np.bincount(X.col, minlength=X.cols), out=rowptr[1:])
    return CSR(X.cols, X.rows, rowptr.astype(np.int32), rows[perm].astype(np.int32), np.conj(X.val[perm]))


def embed(A: CSR, B: CSR):
    """(A_e, B_e) as float32 CSRs, see the module docstring."""
    a = np.asarray(A.val, np.complex64)
    b = np.asarray(B.val, np.complex64)
    lens = np.diff(A.rowptr.astype(np.int64))
    rp = np.zeros(2 * A.rows + 1, np.int64)
    rp[1:] = np.cumsum(np.concatenate([2 * lens, 2 * lens]))
    col = np.stack([2 * A.col.astype(np.int64), 2 * A.col.astype(np.int64) + 1], axis=1).reshape(-1)
    re = np.stack([a.real, -a.imag], axis=1).reshape(-1)
    im = np.stack([a.imag, a.real], axis=1).reshape(-1)
    Ae = CSR(2 * A.rows, 2 * A.cols, rp.astype(np.int32), np.concatenate([col, col]).astype(np.int32),
             np.concatenate([re, im]).astype(np.float32))
    blen = np.diff(B.rowptr.astype(np.int64))
    brp = np.zeros(2 * B.rows + 1, np.int64)
    brp[1::2] = blen
    brp[2::2] = blen
    brp = np.cumsum(brp)
    src = np.repeat(np.arange(B.rows), blen)
    start = np.repeat(brp[0:-1:2], blen) + (np.arange(B.nnz) - np.repeat(B.rowptr[:-1].astype(np.int64), blen))
    bcol = np.empty(2 * B.nnz, np.int32)
    bval = np.empty(2 * B.nnz, np.float32)
    bcol[start], bcol[start + blen[src]] = B.col, B.col
    bval[start], bval[start + blen[src]] = b.real, b.imag
    return Ae, CSR(2 * B.rows, B.cols, brp.astype(np.int32), bcol, bval)


def _split(ref, m):
    """rows [0, m) and [m, 2m) of the embedded exact product as two references with C's row pointers"""
    rp = ref["rowptr"]
    half = int(rp[m])
    out = []
    for sl, base in ((slice(0, half), 0), (slice(half, None), half)):
        d = {k: v[sl] for k, v in ref.items() if isinstance(v, np.ndarray) and k != "rowptr"}
        d["rowptr"] = (rp[:m + 1] if base == 0 else rp[m:] - base).astype(np.int64)
        d["dtype"] = np.float32
        out.append(d)
    return out


def product(lib, A: CSR, B: CSR):
    """(Re, Im): the exact references of the two components of A*B (complex64 values), each a dict of
    exact_ref.product with C's structure and p = 2 x the products of the entry."""
    return _split(xr.product(lib, *embed(A, B)), A.rows)


# complex64 values: real parts from the real generators of exact_ref with `seed`, imaginary parts with seed + 1000
def tier1(nnz, q, seed):
    return (xr.tier1(nnz, q, seed, np.float32) + 1j * xr.tier1(nnz, q, seed + 1000, np.float32)).astype(np.complex64)


def tier2(nnz, seed):
    return (xr.tier2(nnz, seed, np.float32) + 1j * xr.tier2(nnz, seed + 1000, np.float32)).astype(np.complex64)


def tier3(nnz, seed):
    """specials in either component: +-inf, NaN, zeros and subnormal products (inf * 0 is NaN)"""
    re, im = xr.tier3(nnz, seed, np.float32), xr.tier3(nnz, seed + 1000, np.float32)
    out = np.empty(nnz, np.complex64)
    out.real, out.imag = re, im
    return out


def paired(A: CSR, B: CSR, seed):
    """exact_ref.paired for complex values: the same structure and scale factors for both components, so
    C2 = -sum_t a_it * b_tj * d_t cancels far below the sum of the product magnitudes."""
    Ar, Br = xr.paired(CSR(A.rows, A.cols, A.rowptr, A.col, A.val.real.astype(np.float64)),
                       CSR(B.rows, B.cols, B.rowptr, B.col, B.val.real.astype(np.float64)), seed)
    Ai, Bi = xr.paired(CSR(A.rows, A.cols, A.rowptr, A.col, A.val.imag.astype(np.float64)),
                       CSR(B.rows, B.cols, B.rowptr, B.col, B.val.imag.astype(np.float64)), seed)
    return (CSR(Ar.rows, Ar.cols, Ar.rowptr, Ar.col, (Ar.val + 1j * Ai.val).astype(np.complex64)),
            CSR(Br.rows, Br.cols, Br.rowptr, Br.col, (Br.val + 1j * Bi.val).astype(np.complex64)))
