"""MatrixMarket (.mtx) coordinate reader -> CSR, the front end the reference
driver uses for `-spgemm A.mtx [B.mtx]` (SpGEMM_cuda/main.cu:56-64 via
cusp::io::read_matrix_market_file, then ref_spgemm::csr_sort_indices,
ref_spgemm.h:37-62).  Handles real/integer/pattern fields and
general/symmetric/skew-symmetric symmetry like the hand-rolled reader of the
OpenCL driver (SpGEMM_opencl/main.cpp:55-208), and complex fields (hermitian files
mirror the conjugate).  Duplicate entries are summed, columns come out sorted ascending.
A complex file needs a complex dtype: its imaginary parts are never dropped.
"""
from __future__ import annotations

import numpy as np

from .generators import CSR


def read_mtx(path: str, dtype=np.float64) -> CSR:
    with open(path, "r") as f:
        header = f.readline().split()
        if len(header) < 5 or header[0] != "%%MatrixMarket" or header[1].lower() != "matrix":
            raise ValueError("not a MatrixMarket matrix file")
        fmt, field, symm = header[2].lower(), header[3].lower(), header[4].lower()
        if fmt != "coordinate":
            raise ValueError("only coordinate format is supported")
        if field not in ("real", "integer", "pattern", "double", "complex"):
            raise ValueError(f"unsupported field {field}")
        if field == "complex" and not np.issubdtype(np.dtype(dtype), np.complexfloating):
            raise ValueError(f"complex matrix read into the real dtype {np.dtype(dtype)}: pass dtype=np.complex64")
        line = f.readline()
        while line.startswith("%") or not line.strip():
            line = f.readline()
        rows, cols, nnz = (int(x) for x in line.split()[:3])
        data = np.loadtxt(f, ndmin=2) if nnz else np.zeros((0, 4))
    if data.shape[0] != nnz:
        raise ValueError("entry count does not match the size line")
    r = data[:, 0].astype(np.int64) - 1
    c = data[:, 1].astype(np.int64) - 1
    if field == "pattern":
        v = np.ones(nnz)
    elif field == "complex":
        v = data[:, 2] + 1j * data[:, 3]
    else:
        v = data[:, 2].astype(np.float64)
    if symm in ("symmetric", "skew-symmetric", "hermitian"):
        off = r != c
        mirror = -v[off] if symm == "skew-symmetric" else np.conj(v[off]) if symm == "hermitian" else v[off]
        r, c, v = (np.concatenate([r, c[off]]), np.concatenate([c, r[off]]), np.concatenate([v, mirror]))
    elif symm != "general":
        raise ValueError(f"unsupported symmetry {symm}")
    if r.size and (r.min() < 0 or r.max() >= rows or c.min() < 0 or c.max() >= cols):
        raise ValueError("index out of range")
    key = r * np.int64(cols) + c
    order = np.argsort(key, kind="stable")
    key, v = key[order], v[order]
    uniq, start = np.unique(key, return_index=True)
    vals = np.add.reduceat(v, start) if key.size else v
    rr = uniq // cols
    cc = (uniq % cols).astype(np.int32)
    rowptr = np.zeros(rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(rr, minlength=rows), out=rowptr[1:])
    return CSR(rows, cols, rowptr.astype(np.int32), cc, vals.astype(dtype))
