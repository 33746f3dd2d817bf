"""The quad-precision reference of tests/exact_ref.c, the library's error bound, and the value generators of
tests/test_values_gpu.py.

The value contract (DESIGN.md §2, include/bhsparse_b200.h): for an entry C_ij with p products a_ik*b_kj,
s = sum |a_ik*b_kj| (exact), unit roundoff u and smallest normal number lam of the value type,
    |c_hat - c| <= gamma(p)*s + 2*p*lam,   gamma(p) = p*u / (1 - p*u),
for finite inputs whose exact partial sums cannot overflow.  Integer inputs inside the bit budget of
`tier1_bits` are summed exactly in every order, so there the values must be equal."""
import ctypes
import os
import shutil
import subprocess

import numpy as np

from benchmark_spgemm_using_csr_b200.generators import CSR

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCE = os.path.join(HERE, "exact_ref.c")

FINITE, NAN, PINF, NINF = 0, 1, 2, 3

# (significand bits t, unit roundoff u = 2^-t, smallest normal lam)
FORMAT = {np.float64: (53, 2.0 ** -53, 2.0 ** -1022), np.float32: (24, 2.0 ** -24, 2.0 ** -126)}


def compile_lib(tmpdir) -> ctypes.CDLL:
    """gcc -O2 -fopenmp exact_ref.c into tmpdir; None if there is no gcc."""
    gcc = shutil.which("gcc")
    if gcc is None:
        return None
    out = os.path.join(str(tmpdir), "libexact_ref.so")
    r = subprocess.run([gcc, "-O2", "-fopenmp", "-fPIC", "-shared", SOURCE, "-o", out], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lib = ctypes.CDLL(out)
    lib.exact_symbolic.restype = ctypes.c_int64
    lib.exact_numeric.restype = ctypes.c_int
    return lib


def _p(a):
    return ctypes.c_void_p(a.ctypes.data)


def product(lib, A: CSR, B: CSR) -> dict:
    """The exact product of A (m x k) and B (k x n): rowptr, col, hi, lo, s, p, cls per entry of C.
    The value type is A's (float32 or float64)."""
    f32 = A.val.dtype == np.float32
    rpA, cA = np.ascontiguousarray(A.rowptr, np.int32), np.ascontiguousarray(A.col, np.int32)
    rpB, cB = np.ascontiguousarray(B.rowptr, np.int32), np.ascontiguousarray(B.col, np.int32)
    vA = np.ascontiguousarray(A.val, np.float64)
    vB = np.ascontiguousarray(B.val.astype(A.val.dtype), np.float64)
    rowptr = np.zeros(A.rows + 1, dtype=np.int64)
    nnz = lib.exact_symbolic(A.rows, B.cols, _p(rpA), _p(cA), _p(rpB), _p(cB), _p(rowptr))
    assert nnz >= 0, "exact_symbolic: out of memory"
    col = np.empty(nnz, np.int32)
    hi, lo, s = (np.empty(nnz, np.float64) for _ in range(3))
    p = np.empty(nnz, np.int64)
    cls = np.empty(nnz, np.int8)
    rc = lib.exact_numeric(A.rows, B.cols, int(f32), _p(rpA), _p(cA), _p(vA), _p(rpB), _p(cB), _p(vB), _p(rowptr),
                           _p(col), _p(hi), _p(lo), _p(s), _p(p), _p(cls))
    assert rc == 0, "exact_numeric: out of memory"
    return dict(rowptr=rowptr, col=col, hi=hi, lo=lo, s=s, p=p, cls=cls, dtype=A.val.dtype.type)


def bound(p, s, dtype):
    """gamma(p)*s + 2*p*lam: the largest error the library allows in an entry of p products with sum s of their
    magnitudes."""
    _, u, lam = FORMAT[dtype]
    p = np.asarray(p, dtype=np.float64)
    return p * u / (1.0 - p * u) * np.asarray(s, dtype=np.float64) + 2.0 * p * lam


def tier1_bits(p_max: int, dtype) -> int:
    """q such that integers in [-2^q, 2^q] are summed exactly in every order by entries of at most p_max products:
    p_max * 2^(2q) <= 2^(t-1)."""
    t = FORMAT[dtype][0]
    return (t - 1 - int(np.ceil(np.log2(max(p_max, 1))))) // 2


def row_index(rowptr):
    rowptr = np.asarray(rowptr, dtype=np.int64)
    return np.repeat(np.arange(rowptr.size - 1, dtype=np.int64), np.diff(rowptr))


# ---- value generators --------------------------------------------------------------------------------
def tier1(nnz, q, seed, dtype, zeros=0.01):
    """Nonzero integers in [-2^q, 2^q], and a fraction `zeros` of explicit zeros."""
    rng = np.random.default_rng(seed)
    v = rng.integers(1, 2 ** q + 1, size=nnz) * rng.choice([-1, 1], size=nnz)
    v[rng.random(nnz) < zeros] = 0
    return v.astype(dtype)


def tier2(nnz, seed, dtype):
    """+-(1 + f) * 2^e: every significand bit random, e in [-4, 4]."""
    rng = np.random.default_rng(seed)
    t = FORMAT[dtype][0]
    frac = rng.integers(0, 2 ** (t - 1), size=nnz, dtype=np.int64).astype(np.float64) / 2.0 ** (t - 1)
    v = (1.0 + frac) * np.exp2(rng.integers(-4, 5, size=nnz)) * rng.choice([-1.0, 1.0], size=nnz)
    return v.astype(dtype)


def tier3(nnz, seed, dtype, rate=0.002):
    """Tier-2 values with specials sprinkled in at `rate` each: +-inf, NaN, stored zeros (which meet an inf in
    some products: inf * 0 is NaN), and values whose products with each other are subnormal."""
    rng = np.random.default_rng(seed)
    v = tier2(nnz, seed + 1, dtype).astype(np.float64)
    tiny = 2.0 ** -70 if dtype == np.float32 else 2.0 ** -530
    pick = rng.random(nnz)
    v[pick < rate] = np.inf
    v[(pick >= rate) & (pick < 2 * rate)] = -np.inf
    v[(pick >= 2 * rate) & (pick < 3 * rate)] = np.nan
    v[(pick >= 3 * rate) & (pick < 8 * rate)] = 0.0
    sub = (pick >= 8 * rate) & (pick < 40 * rate)
    v[sub] = np.sign(v[sub]) * np.abs(v[sub]) * tiny
    return v.astype(dtype)


def paired(A: CSR, B: CSR, seed):
    """Operands whose product cancels: B2 has rows 2t, 2t+1 = row t of B and row t of B scaled by (1 + d_t),
    A2 has the entries (a, -a) in columns (2t, 2t+1) for every entry a in column t of A.  C2 has the pattern of
    A*B, and C2_ij = -sum_t a_it * b_tj * d_t, so |C2_ij| is about 2^-10 of the sum of its product magnitudes."""
    rng = np.random.default_rng(seed)
    d = np.exp2(-rng.integers(8, 13, size=B.rows)) * (1.0 + rng.integers(0, 2 ** 20, size=B.rows) / 2.0 ** 20)
    lens = np.diff(B.rowptr.astype(np.int64))
    rp = np.zeros(2 * B.rows + 1, np.int64)
    rp[1::2] = lens
    rp[2::2] = lens
    rp = np.cumsum(rp)
    src = np.repeat(np.arange(B.rows), lens)
    col = np.empty(2 * B.nnz, np.int32)
    val = np.empty(2 * B.nnz, np.float64)
    start = np.repeat(rp[0:-1:2], lens) + (np.arange(B.nnz) - np.repeat(B.rowptr[:-1].astype(np.int64), lens))
    col[start] = B.col
    col[start + lens[src]] = B.col
    val[start] = B.val
    val[start + lens[src]] = B.val * (1.0 + d[src])
    B2 = CSR(2 * B.rows, B.cols, rp.astype(np.int32), col, val.astype(B.val.dtype))
    ac = np.stack([2 * A.col.astype(np.int64), 2 * A.col.astype(np.int64) + 1], axis=1).reshape(-1)
    av = np.stack([A.val, -A.val], axis=1).reshape(-1)
    A2 = CSR(A.rows, 2 * A.cols, (2 * A.rowptr.astype(np.int64)).astype(np.int32), ac.astype(np.int32), av)
    return A2, B2
