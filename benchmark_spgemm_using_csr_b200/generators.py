"""Synthetic CSR workloads for the SpGEMM path (host side, numpy).

These replace the CUSP gallery calls of the reference driver
(SpGEMM_cuda/main.cu:30-53: poisson5pt/9pt/7pt/27pt) and add the R-MAT and
uniform-random rectangular workloads BASELINE.json names.  Patterns follow the
CUSP gallery convention as far as the reference exposes it: regular grid, x the
fastest-varying index, out-of-grid neighbours dropped; the nnz counts match the
stock sizes (326 656 / 586 756 / 912 951 / 3 442 951, SURVEY.md Appendix C).

Values mirror main.cu:79-94 (`rand() % 9 + 1`) but from a fixed-seed
counter-based generator so that runs are reproducible.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

__all__ = [
    "CSR", "poisson5pt", "poisson9pt", "poisson7pt", "poisson27pt", "rmat",
    "uniform_rect", "random_csr", "banded_random", "diagonals", "rmat_counter", "rmat_counter_torch", "int_values", "real_values", "transpose_pattern", "transpose",
]


@dataclass
class CSR:
    """Host CSR triple in the reference's layout (bhsparse.h:22-25): int32
    row pointers / column indices (0-based, ascending, duplicate-free per row)
    and float32/float64 values."""
    rows: int
    cols: int
    rowptr: np.ndarray
    col: np.ndarray
    val: np.ndarray

    @property
    def nnz(self) -> int:
        return int(self.rowptr[-1])

    def astype(self, dt) -> "CSR":
        return CSR(self.rows, self.cols, self.rowptr, self.col, self.val.astype(dt))

    def row_slice(self, r0: int, r1: int) -> "CSR":
        """Rows [r0, r1) as an independent CSR (used by the row-block partition)."""
        s, e = int(self.rowptr[r0]), int(self.rowptr[r1])
        rp = (self.rowptr[r0:r1 + 1] - s).astype(np.int32)
        return CSR(r1 - r0, self.cols, rp, self.col[s:e], self.val[s:e])


def _splitmix64(x: np.ndarray) -> np.ndarray:
    x = (x + np.uint64(0x9E3779B97F4A7C15)).astype(np.uint64)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def int_values(nnz: int, seed: int, dtype=np.float64) -> np.ndarray:
    """Integers 1..9 (exactly representable -> order-independent sums), the
    deterministic counterpart of main.cu:82,93."""
    with np.errstate(over="ignore"):
        h = _splitmix64(np.arange(nnz, dtype=np.uint64) + np.uint64(seed) * np.uint64(0x632BE59BD9B4E019))
    return ((h % np.uint64(9)) + np.uint64(1)).astype(dtype)


def real_values(nnz: int, seed: int, dtype=np.float64) -> np.ndarray:
    """Uniform reals in (0,1] -- exercises the tolerance path."""
    with np.errstate(over="ignore"):
        h = _splitmix64(np.arange(nnz, dtype=np.uint64) + np.uint64(seed) * np.uint64(0x632BE59BD9B4E019))
    return (((h >> np.uint64(11)).astype(np.float64) + 1.0) * (1.0 / 9007199254740992.0)).astype(dtype)


def _values(nnz, seed, dtype, kind):
    if kind == "int":
        return int_values(nnz, seed, dtype)
    if kind == "real":
        return real_values(nnz, seed, dtype)
    if kind == "ones":
        return np.ones(nnz, dtype=dtype)
    raise ValueError(kind)


def _stencil(dims, offsets, seed, dtype, values):
    """Generic box/axis stencil on a regular grid; dims = (nx[,ny[,nz]])."""
    nd = len(dims)
    N = int(np.prod(dims))
    idx = np.arange(N, dtype=np.int64)
    coords = []
    rem = idx
    for d in dims:                      # x fastest
        coords.append(rem % d)
        rem = rem // d
    strides = [int(np.prod(dims[:i])) for i in range(nd)]
    # ascending column offset order
    offs = sorted(offsets, key=lambda o: sum(o[i] * strides[i] for i in range(nd)))
    counts = np.zeros(N, dtype=np.int64)
    masks = []
    for o in offs:
        ok = np.ones(N, dtype=bool)
        for i in range(nd):
            if o[i] < 0:
                ok &= coords[i] >= -o[i]
            elif o[i] > 0:
                ok &= coords[i] < dims[i] - o[i]
        masks.append(ok)
        counts += ok
    rowptr = np.zeros(N + 1, dtype=np.int64)
    np.cumsum(counts, out=rowptr[1:])
    nnz = int(rowptr[-1])
    if nnz > np.iinfo(np.int32).max:
        raise OverflowError("nnz exceeds int32")
    col = np.empty(nnz, dtype=np.int32)
    cursor = rowptr[:-1].copy()
    for o, ok in zip(offs, masks):
        delta = sum(o[i] * strides[i] for i in range(nd))
        pos = cursor[ok]
        col[pos] = (idx[ok] + delta).astype(np.int32)
        cursor[ok] += 1
    return CSR(N, N, rowptr.astype(np.int32), col, _values(nnz, seed, dtype, values))


def poisson5pt(nx, ny, seed=2, dtype=np.float64, values="int"):
    """2-D 5-point stencil (main.cu:32-33)."""
    offs = [(0, 0), (-1, 0), (1, 0), (0, -1), (0, 1)]
    return _stencil((nx, ny), offs, seed, dtype, values)


def poisson9pt(nx, ny, seed=2, dtype=np.float64, values="int"):
    """2-D 9-point stencil (main.cu:38-39)."""
    offs = [(dx, dy) for dy in (-1, 0, 1) for dx in (-1, 0, 1)]
    return _stencil((nx, ny), offs, seed, dtype, values)


def poisson7pt(nx, ny, nz, seed=2, dtype=np.float64, values="int"):
    """3-D 7-point stencil (main.cu:44-45)."""
    offs = [(0, 0, 0), (-1, 0, 0), (1, 0, 0), (0, -1, 0), (0, 1, 0), (0, 0, -1), (0, 0, 1)]
    return _stencil((nx, ny, nz), offs, seed, dtype, values)


def poisson27pt(nx, ny, nz, seed=2, dtype=np.float64, values="int"):
    """3-D 27-point stencil (main.cu:50-51)."""
    offs = [(dx, dy, dz) for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)]
    return _stencil((nx, ny, nz), offs, seed, dtype, values)


def _from_coo_dedup(rows, cols, r, c, seed, dtype, values):
    key = (r.astype(np.int64) << np.int64(32)) | c.astype(np.int64)
    key = np.unique(key)                     # sorted + duplicate-free
    r = (key >> np.int64(32)).astype(np.int64)
    c = (key & np.int64(0xFFFFFFFF)).astype(np.int32)
    nnz = key.size
    if nnz > np.iinfo(np.int32).max:
        raise OverflowError("nnz exceeds int32")
    rowptr = np.zeros(rows + 1, dtype=np.int64)
    counts = np.bincount(r, minlength=rows)
    np.cumsum(counts, out=rowptr[1:])
    return CSR(rows, cols, rowptr.astype(np.int32), c, _values(nnz, seed, dtype, values))


def rmat(scale, edge_factor=16, a=0.45, b=0.15, c=0.15, d=0.25, seed=1, value_seed=2,
         dtype=np.float64, values="int"):
    """R-MAT power-law matrix, n = 2**scale, edge_factor*n generated edges,
    duplicates merged, columns sorted.  Default quadrant probabilities are the
    "mild" (.45,.15,.15,.25) set SURVEY.md Appendix B sizes (Graph500's
    (.57,.19,.19,.05) gives 1.46e11 products at scale 22)."""
    if abs(a + b + c + d - 1.0) > 1e-9:
        raise ValueError("a+b+c+d must be 1")
    n = 1 << scale
    E = edge_factor * n
    rng = np.random.Generator(np.random.PCG64(seed))
    r = np.zeros(E, dtype=np.int64)
    cc = np.zeros(E, dtype=np.int64)
    for _ in range(scale):
        u = rng.random(E)
        # quadrants: a=(0,0) b=(0,1) c=(1,0) d=(1,1)
        rbit = u >= a + b
        cbit = ((u >= a) & (u < a + b)) | (u >= a + b + c)
        r = (r << 1) | rbit
        cc = (cc << 1) | cbit
    return _from_coo_dedup(n, n, r, cc, value_seed, dtype, values)


def uniform_rect(rows, cols, per_row=8, seed=1, value_seed=2, dtype=np.float32, values="int"):
    """`rows` x `cols` with exactly `per_row` distinct, uniformly drawn, sorted
    columns in every row (BASELINE.json config 4)."""
    if per_row > cols:
        raise ValueError("per_row > cols")
    rng = np.random.Generator(np.random.PCG64(seed))
    # sorted sample from [0, cols-per_row] plus 0..per_row-1 -> strictly increasing
    base = rng.integers(0, cols - per_row + 1, size=(rows, per_row), dtype=np.int64)
    base.sort(axis=1)
    base += np.arange(per_row, dtype=np.int64)[None, :]
    nnz = rows * per_row
    if nnz > np.iinfo(np.int32).max:
        raise OverflowError("nnz exceeds int32")
    rowptr = (np.arange(rows + 1, dtype=np.int64) * per_row).astype(np.int32)
    return CSR(rows, cols, rowptr, base.reshape(-1).astype(np.int32), _values(nnz, value_seed, dtype, values))


def random_csr(rows, cols, row_nnz, seed=1, value_seed=2, dtype=np.float64, values="int"):
    """Test helper: row i gets row_nnz[i] distinct sorted uniform columns
    (row_nnz may be a scalar).  Used to hit chosen bin boundaries."""
    rng = np.random.Generator(np.random.PCG64(seed))
    row_nnz = np.broadcast_to(np.asarray(row_nnz, dtype=np.int64), (rows,)).copy()
    row_nnz = np.minimum(row_nnz, cols)
    rowptr = np.zeros(rows + 1, dtype=np.int64)
    np.cumsum(row_nnz, out=rowptr[1:])
    nnz = int(rowptr[-1])
    col = np.empty(nnz, dtype=np.int32)
    for i in range(rows):
        k = int(row_nnz[i])
        if k == 0:
            continue
        if k * 4 >= cols:
            sel = np.sort(rng.permutation(cols)[:k])
        else:
            sel = rng.integers(0, cols - k + 1, size=k, dtype=np.int64)
            sel.sort()
            sel += np.arange(k, dtype=np.int64)
        col[rowptr[i]:rowptr[i + 1]] = sel
    return CSR(rows, cols, rowptr.astype(np.int32), col, _values(nnz, value_seed, dtype, values))


def banded_random(n, half_bw, row_nnz, seed=1, value_seed=2, dtype=np.float64, values="int"):
    """n x n matrix whose row i has `row_nnz` distinct sorted columns drawn from the
    band [i-half_bw, i+half_bw] (clipped): narrow column span per row, like FEM or
    stencil matrices, but irregular inside the band."""
    rng = np.random.Generator(np.random.PCG64(seed))
    rowptr = np.zeros(n + 1, dtype=np.int64)
    cols = []
    for i in range(n):
        lo, hi = max(0, i - half_bw), min(n - 1, i + half_bw)
        k = min(int(row_nnz), hi - lo + 1)
        sel = np.sort(rng.choice(hi - lo + 1, size=k, replace=False)) + lo
        cols.append(sel)
        rowptr[i + 1] = rowptr[i] + k
    col = np.concatenate(cols).astype(np.int32) if cols else np.zeros(0, np.int32)
    return CSR(n, n, rowptr.astype(np.int32), col, _values(col.size, value_seed, dtype, values))


def transpose_pattern(A: CSR, value_seed=3, values="int") -> CSR:
    """A^T with fresh values (test helper for rectangular chains)."""
    r = np.repeat(np.arange(A.rows, dtype=np.int64), np.diff(A.rowptr))
    return _from_coo_dedup(A.cols, A.rows, A.col.astype(np.int64), r, value_seed, A.val.dtype, values)


def transpose(X: CSR) -> CSR:
    """X^T by a stable argsort of the columns: the entries of a row of X^T in the stored order of X."""
    rows = np.repeat(np.arange(X.rows, dtype=np.int64), np.diff(X.rowptr.astype(np.int64)))
    perm = np.argsort(X.col, kind="stable")
    rowptr = np.zeros(X.cols + 1, dtype=np.int64)
    np.cumsum(np.bincount(X.col, minlength=X.cols), out=rowptr[1:])
    return CSR(X.cols, X.rows, rowptr.astype(np.int32), rows[perm].astype(np.int32), X.val[perm])


def diagonals(rows, cols, offsets, keep=1.0, seed=1, value_seed=2, dtype=np.float64, values="int") -> CSR:
    """Entries at (i, i + d) for every offset d in `offsets` that lands inside the matrix
    (DIA-like: stencils, banded and Toeplitz-structured matrices); with keep < 1 each entry
    survives with that probability, so rows hold irregular subsets of the diagonals."""
    offs = np.unique(np.asarray(offsets, dtype=np.int64))
    i = np.repeat(np.arange(rows, dtype=np.int64), offs.size)
    c = i + np.tile(offs, rows)
    ok = (c >= 0) & (c < cols)
    if keep < 1.0:
        rng = np.random.Generator(np.random.PCG64(seed))
        ok &= rng.random(ok.size) < keep
    return _from_coo_dedup(rows, cols, i[ok], c[ok], value_seed, dtype, values)


# ---- counter-based R-MAT: the same matrix from numpy (host) and torch (device) -----------------
# bench.py builds config 5 (scale 24: 2.7e8 edges) on the GPU in seconds; numpy's PCG stream above
# cannot be reproduced there, so this generator draws every (edge, level) decision from a
# SplitMix64 hash of its counter.  Bit-identical across the two back ends (tests/test_generators.py).
_SM_GAMMA = 0x9E3779B97F4A7C15
_SM_M1 = 0xBF58476D1CE4E5B9
_SM_M2 = 0x94D049BB133111EB
_VAL_MUL = 0x632BE59BD9B4E019


def _rmat_thresholds(a, b, c, d):
    if abs(a + b + c + d - 1.0) > 1e-9:
        raise ValueError("a+b+c+d must be 1")
    s = float(1 << 32)
    return int(a * s), int((a + b) * s), int((a + b + c) * s)


def rmat_counter(scale, edge_factor=16, a=0.45, b=0.15, c=0.15, d=0.25, seed=1, value_seed=2, dtype=np.float64) -> CSR:
    """R-MAT like rmat(), decisions from SplitMix64(edge * 64 + level + seed * 2^40) >> 32."""
    n = 1 << scale
    E = edge_factor * n
    ta, tb, tc = _rmat_thresholds(a, b, c, d)
    e = np.arange(E, dtype=np.uint64) * np.uint64(64) + (np.uint64(seed) << np.uint64(40))
    r = np.zeros(E, dtype=np.int64)
    cc = np.zeros(E, dtype=np.int64)
    with np.errstate(over="ignore"):
        for level in range(scale):
            u = (_splitmix64(e + np.uint64(level)) >> np.uint64(32)).astype(np.int64)
            rbit = u >= tb
            cbit = ((u >= ta) & (u < tb)) | (u >= tc)
            r = (r << 1) | rbit
            cc = (cc << 1) | cbit
    return _from_coo_dedup(n, n, r, cc, value_seed, dtype, "int")


def _i64(x: int) -> int:
    """The two's-complement int64 holding the uint64 bit pattern x."""
    x &= (1 << 64) - 1
    return x - (1 << 64) if x >= (1 << 63) else x


def rmat_counter_torch(scale, edge_factor=16, a=0.45, b=0.15, c=0.15, d=0.25, seed=1, value_seed=2, dtype=None,
                       device="cuda"):
    """rmat_counter() on a torch device.  Returns (rowptr int32, col int32, val) tensors there.
    int64 arithmetic wraps like uint64; logical shifts are arithmetic shifts + a mask."""
    import torch
    dtype = dtype or torch.float64
    n = 1 << scale
    E = edge_factor * n
    ta, tb, tc = _rmat_thresholds(a, b, c, d)

    def lsr(x, s):
        return (x >> s) & ((1 << (64 - s)) - 1)

    def splitmix(x):
        x = x + _i64(_SM_GAMMA)
        x = (x ^ lsr(x, 30)) * _i64(_SM_M1)
        x = (x ^ lsr(x, 27)) * _i64(_SM_M2)
        return x ^ lsr(x, 31)

    e = torch.arange(E, dtype=torch.int64, device=device) * 64 + _i64(seed << 40)
    r = torch.zeros(E, dtype=torch.int64, device=device)
    cc = torch.zeros(E, dtype=torch.int64, device=device)
    for level in range(scale):
        u = lsr(splitmix(e + level), 32)
        rbit = (u >= tb).to(torch.int64)
        cbit = (((u >= ta) & (u < tb)) | (u >= tc)).to(torch.int64)
        r = (r << 1) | rbit
        cc = (cc << 1) | cbit
        del u, rbit, cbit
    del e
    key = (r << 32) | cc
    del r, cc
    key = torch.unique(key)                                   # sorted, duplicate-free
    rows = key >> 32
    col = (key & 0xFFFFFFFF).to(torch.int32)
    del key
    nnz = int(col.numel())
    if nnz > np.iinfo(np.int32).max:
        raise OverflowError("nnz exceeds int32")
    counts = torch.bincount(rows, minlength=n)
    del rows
    rowptr = torch.zeros(n + 1, dtype=torch.int64, device=device)
    torch.cumsum(counts, 0, out=rowptr[1:])
    h = splitmix(torch.arange(nnz, dtype=torch.int64, device=device) + _i64(value_seed * _VAL_MUL))
    hi, lo = lsr(h, 32), h & 0xFFFFFFFF
    val = (((hi * 4 + lo) % 9) + 1).to(dtype)                 # uint64 h mod 9 (2^32 mod 9 = 4)
    return rowptr.to(torch.int32), col, val
