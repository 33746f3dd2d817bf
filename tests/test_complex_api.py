"""complex64 products without a GPU: the header and the Python binding agree on the new type, op and entry points;
C99 and C++ callers compile and link; the Matrix Market reader handles complex files like scipy; and the embedding
reference of tests/complex_ref.py gives the exact complex product (checked against complex Fractions), including
conjugate-transposed operands."""
import math
import os
import re
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import complex_ref as cr
import exact_ref as xr
from benchmark_spgemm_using_csr_b200 import capi, generators as gen, mtx
from benchmark_spgemm_using_csr_b200.generators import CSR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "bhsparse_b200.h")


def test_header_and_binding_agree():
    h = open(HEADER).read()
    assert re.search(r"^#define BHB200_DTYPE_C64 4$", h, re.M)
    assert re.search(r"^#define BHB200_OP_C 2$", h, re.M)
    assert not re.search(r"^#define BHB200_\w+ 3$", h, re.M), "dtype 3 stays invalid"
    assert capi.DTYPE_C64 == 4 and capi.OP_C == 2
    for name in ("bhb200_init_data_op_c64", "bhb200_update_values_c64", "bhb200_get_C_c64"):
        assert name in capi.EXPORTED and re.search(rf"\b{name}\(", h)


C_CALLER = r'''
#include <stddef.h>
#include "bhsparse_b200.h"

int main(void)
{
    bhb200_ctx *ctx = NULL;
    /* A = [[1+2i, 3], [0, -1i]] as interleaved (re, im) floats; C = A * A^H */
    int32_t rowptr[3] = {0, 2, 3}, col[3] = {0, 1, 1};
    float val[6] = {1.f, 2.f, 3.f, 0.f, 0.f, -1.f};
    int32_t rowptrC[3], colC[4];
    float valC[8];
    int rc;
    if (bhb200_create(&ctx, 0) != BHB200_SUCCESS) return 0;   /* no device: nothing to run */
    rc = bhb200_init_data_op_c64(ctx, BHB200_OP_N, BHB200_OP_C, 2, 2, 2, 3, val, rowptr, col, 3, val, rowptr, col);
    if (rc == BHB200_SUCCESS) rc = bhb200_spgemm(ctx);
    if (rc == BHB200_SUCCESS) rc = bhb200_update_values_c64(ctx, val, val);
    if (rc == BHB200_SUCCESS) rc = bhb200_spgemm_numeric(ctx);
    if (rc == BHB200_SUCCESS) rc = bhb200_get_C_c64(ctx, rowptrC, colC, valC);
    if (rc == BHB200_SUCCESS) rc = bhb200_init_data_device(ctx, BHB200_DTYPE_C64, 0, 0, 0, 0, NULL, rowptr, NULL, 0, NULL,
                                                           rowptr, NULL);
    bhb200_destroy(ctx);
    return rc == BHB200_SUCCESS ? 0 : 1;
}
'''

CXX_CALLER = r'''
#include "bhsparse.h"

int main()
{
    bool platforms[NUM_PLATFORMS] = {false};
    platforms[BHSPARSE_CUDA] = true;
    bhsparse bh;
    bh.set_verbose(false);
    if (bh.initPlatform(platforms) != BHSPARSE_SUCCESS) return 0;   /* no device: nothing to run */
    index_type rowptr[3] = {0, 2, 3}, col[3] = {0, 1, 1};
    value_type val[3] = {value_type(1.f, 2.f), value_type(3.f, 0.f), value_type(0.f, -1.f)};
    index_type rowptrC[3], colC[4];
    value_type valC[4];
    int rc = bh.initData(2, 2, 2, 3, val, rowptr, col, 3, val, rowptr, col, rowptrC);
    if (rc == BHSPARSE_SUCCESS) rc = bh.spgemm();
    if (rc == BHSPARSE_SUCCESS) rc = bh.update_values(val, val);
    if (rc == BHSPARSE_SUCCESS) rc = bh.get_C(colC, valC);
    return rc == BHSPARSE_SUCCESS ? 0 : 1;
}
'''


def _compile(tmp_path, compiler, args, source, name):
    src = tmp_path / name
    src.write_text(source)
    libdir = os.path.dirname(capi.LIB_PATH)
    r = subprocess.run([compiler, *args, "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                        "-o", str(tmp_path / name.split(".")[0]), "-L", libdir, "-lbhsparse_b200", f"-Wl,-rpath,{libdir}"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_c99_caller_compiles_and_links(tmp_path):
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    if not cc:
        pytest.skip("no C compiler")
    capi.load(build_if_missing=True)
    _compile(tmp_path, cc, ["-std=c99", "-pedantic"], C_CALLER, "caller.c")


def test_cxx_complex_caller_compiles_and_links(tmp_path):
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if not cxx:
        pytest.skip("no C++ compiler")
    capi.load(build_if_missing=True)
    _compile(tmp_path, cxx, ["-std=c++17", "-DBHSPARSE_VALUE_COMPLEX_FLOAT"], CXX_CALLER, "caller.cpp")


# ---- Matrix Market ------------------------------------------------------------------------------------------
ENTRIES = {   # (row, col, re, im), 1-based; the lower triangle for the symmetric kinds
    "general": [(1, 1, 1.5, -2.0), (1, 3, 0.25, 4.0), (2, 2, -1.0, 0.0), (3, 1, 2.0, 2.0), (3, 2, 0.0, -0.5)],
    "symmetric": [(1, 1, 1.5, -2.0), (2, 1, 0.25, 4.0), (3, 2, -1.0, 0.5), (3, 3, 2.0, 1.0)],
    "skew-symmetric": [(2, 1, 0.25, 4.0), (3, 1, -1.0, 0.5), (3, 2, 2.0, -3.0)],
    "hermitian": [(1, 1, 1.5, 0.0), (2, 1, 0.25, 4.0), (3, 2, -1.0, 0.5), (3, 3, 2.0, 0.0)],
}


@pytest.mark.parametrize("symm", list(ENTRIES))
def test_read_complex_mtx_like_scipy(tmp_path, symm):
    sio = pytest.importorskip("scipy.io")
    ent = ENTRIES[symm]
    path = tmp_path / f"{symm}.mtx"
    path.write_text(f"%%MatrixMarket matrix coordinate complex {symm}\n% comment\n3 3 {len(ent)}\n" +
                    "".join(f"{r} {c} {re} {im}\n" for r, c, re, im in ent))
    want = sio.mmread(str(path)).toarray()
    got = mtx.read_mtx(str(path), dtype=np.complex64)
    assert got.val.dtype == np.complex64
    dense = np.zeros((3, 3), np.complex128)
    for i in range(3):
        for p in range(got.rowptr[i], got.rowptr[i + 1]):
            dense[i, got.col[p]] = got.val[p]
        assert np.all(np.diff(got.col[got.rowptr[i]:got.rowptr[i + 1]]) > 0)
    assert np.array_equal(dense, want)


def test_complex_mtx_into_real_dtype_is_refused(tmp_path):
    path = tmp_path / "c.mtx"
    path.write_text("%%MatrixMarket matrix coordinate complex general\n2 2 1\n1 2 1.0 3.0\n")
    with pytest.raises(ValueError, match="complex"):
        mtx.read_mtx(str(path), dtype=np.float64)


# ---- the embedding reference -----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    lib = xr.compile_lib(tmp_path_factory.mktemp("exact_ref"))
    if lib is None:
        pytest.skip("gcc not found")
    return lib


def _fraction_product(A: CSR, B: CSR):
    """{(i, j): (Re, Im, s_re, s_im, products)} by a complex Gustavson over Fractions"""
    out = {}
    for i in range(A.rows):
        for pa in range(A.rowptr[i], A.rowptr[i + 1]):
            k, a = A.col[pa], A.val[pa]
            ar, ai = Fraction(float(a.real)), Fraction(float(a.imag))
            for q in range(B.rowptr[k], B.rowptr[k + 1]):
                b = B.val[q]
                br, bi = Fraction(float(b.real)), Fraction(float(b.imag))
                e = out.setdefault((i, int(B.col[q])), [Fraction(0)] * 4 + [0])
                e[0] += ar * br - ai * bi
                e[1] += ar * bi + ai * br
                e[2] += abs(ar * br) + abs(ai * bi)
                e[3] += abs(ar * bi) + abs(ai * br)
                e[4] += 1
    return out


def _op(X: CSR, o: str) -> CSR:
    """op(X) for o = N, T (transpose) or C (conjugate transpose)"""
    if o == "N":
        return X
    H = cr.conj_transpose(X)
    return H if o == "C" else CSR(H.rows, H.cols, H.rowptr, H.col, np.conj(H.val))


@pytest.mark.parametrize("ops", ["NN", "NC", "CN", "CC", "TC"])
def test_embedding_reference_is_exact(lib, ops):
    rng = np.random.default_rng(5)
    m, k, n = 23, 17, 29

    def stored(rows, cols, o, seed):   # a random complex operand, stored as op(X) needs it
        r, c = (rows, cols) if o == "N" else (cols, rows)
        X = gen.random_csr(r, c, rng.integers(0, 8, r), seed=seed, dtype=np.float32)
        return CSR(X.rows, X.cols, X.rowptr, X.col, cr.tier2(X.nnz, seed + 10))
    opA, opB = _op(stored(m, k, ops[0], 1), ops[0]), _op(stored(k, n, ops[1], 2), ops[1])
    assert (opA.rows, opA.cols, opB.rows, opB.cols) == (m, k, k, n)
    want = _fraction_product(opA, opB)
    re, im = cr.product(lib, opA, opB)
    assert np.array_equal(re["rowptr"], im["rowptr"]) and np.array_equal(re["col"], im["col"])
    rows = xr.row_index(re["rowptr"])
    assert len(want) == re["col"].size
    for t in range(re["col"].size):
        w = want[(int(rows[t]), int(re["col"][t]))]
        for ref, exact, s in ((re, w[0], w[2]), (im, w[1], w[3])):
            assert ref["cls"][t] == xr.FINITE
            assert Fraction(ref["hi"][t]) + Fraction(ref["lo"][t]) == exact
            assert ref["p"][t] == 2 * w[4]
            assert math.isclose(ref["s"][t], float(s), rel_tol=2.0 ** -50)


def test_conjugate_transpose_on_host():
    X = CSR(2, 3, np.array([0, 2, 3], np.int32), np.array([0, 2, 1], np.int32),
            np.array([1 + 2j, 3 - 1j, -4j], np.complex64))
    H = cr.conj_transpose(X)
    assert H.rows == 3 and H.cols == 2
    assert H.rowptr.tolist() == [0, 1, 2, 3] and H.col.tolist() == [0, 1, 0]
    assert H.val.tolist() == [1 - 2j, 4j, 3 + 1j]
