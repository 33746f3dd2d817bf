"""complex128 products without a GPU: the header, the binding and the exports agree on the new type and entry points;
C99 and C++ callers compile and link; the f64 embedding reference of tests/complex128_ref.py gives the complex product
to the reference's own accuracy (checked against complex Fractions), including conjugate-transposed operands; and the host plans of the
direct mode and the diagonal-pattern mode lay out 16-byte values."""
import ctypes
import math
import os
import re
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import complex128_ref as cr
import exact_ref as xr
from benchmark_spgemm_using_csr_b200 import capi, generators as gen
from benchmark_spgemm_using_csr_b200.generators import CSR
from test_complex_api import _compile, _fraction_product, _op
from test_direct_plan import (HEAVY_ROWS, P_MAX, RMAT, RMAT_TOP, SB_B8192, SB_B16384, SB_B32768, SB_G4096, SB_LARGE,
                              heavy, plan, probe, wide)   # noqa: F401 (probe: the planner harness fixture)
from test_pattern_plan import _probe, _stencil27

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "bhsparse_b200.h")
C128_ENTRIES = ("bhb200_init_data_op_c128", "bhb200_update_values_c128", "bhb200_get_C_c128")


def test_header_binding_and_exports_agree():
    h = open(HEADER).read()
    assert re.search(r"^#define BHB200_DTYPE_C128 5$", h, re.M)
    assert not re.search(r"^#define BHB200_\w+ 3$", h, re.M), "dtype 3 stays invalid"
    assert capi.DTYPE_C128 == 5 and capi.VALUE_TYPES[capi.DTYPE_C128] == ("c128", "complex128")
    assert capi.dtype_of(np.dtype(np.complex128)) == capi.DTYPE_C128 and capi.dtype_of("torch.complex128") == capi.DTYPE_C128
    L = capi.load(build_if_missing=True)
    for name in C128_ENTRIES:
        assert name in capi.EXPORTED and re.search(rf"\b{name}\(", h)
        assert getattr(L, name) is not None
    out = subprocess.run(["nm", "-D", "--defined-only", capi.LIB_PATH], capture_output=True, text=True).stdout
    assert all(re.search(rf"\b{name}$", out, re.M) for name in C128_ENTRIES)


C_CALLER = r'''
#include <stddef.h>
#include "bhsparse_b200.h"

int main(void)
{
    bhb200_ctx *ctx = NULL;
    /* A = [[1+2i, 3], [0, -1i]] as interleaved (re, im) doubles; C = A * A^H */
    int32_t rowptr[3] = {0, 2, 3}, col[3] = {0, 1, 1};
    double val[6] = {1.0, 2.0, 3.0, 0.0, 0.0, -1.0};
    int32_t rowptrC[3], colC[4];
    double valC[8];
    int rc;
    if (bhb200_create(&ctx, 0) != BHB200_SUCCESS) return 0;   /* no device: nothing to run */
    rc = bhb200_init_data_op_c128(ctx, BHB200_OP_N, BHB200_OP_C, 2, 2, 2, 3, val, rowptr, col, 3, val, rowptr, col);
    if (rc == BHB200_SUCCESS) rc = bhb200_spgemm(ctx);
    if (rc == BHB200_SUCCESS) rc = bhb200_update_values_c128(ctx, val, val);
    if (rc == BHB200_SUCCESS) rc = bhb200_spgemm_numeric(ctx);
    if (rc == BHB200_SUCCESS) rc = bhb200_get_C_c128(ctx, rowptrC, colC, valC);
    if (rc == BHB200_SUCCESS) rc = bhb200_init_data_device(ctx, BHB200_DTYPE_C128, 0, 0, 0, 0, NULL, rowptr, NULL, 0, NULL,
                                                           rowptr, NULL);
    bhb200_destroy(ctx);
    return rc == BHB200_SUCCESS ? 0 : 1;
}
'''

CXX_CALLER = r'''
#include <type_traits>
#include "bhsparse.h"

static_assert(std::is_same<value_type, std::complex<double>>::value, "BHSPARSE_VALUE_COMPLEX_DOUBLE");

int main()
{
    bool platforms[NUM_PLATFORMS] = {false};
    platforms[BHSPARSE_CUDA] = true;
    bhsparse bh;
    bh.set_verbose(false);
    if (bh.initPlatform(platforms) != BHSPARSE_SUCCESS) return 0;   /* no device: nothing to run */
    index_type rowptr[3] = {0, 2, 3}, col[3] = {0, 1, 1};
    value_type val[3] = {value_type(1.0, 2.0), value_type(3.0, 0.0), value_type(0.0, -1.0)};
    index_type rowptrC[3], colC[4];
    value_type valC[4];
    int rc = bh.initData(2, 2, 2, 3, val, rowptr, col, 3, val, rowptr, col, rowptrC);
    if (rc == BHSPARSE_SUCCESS) rc = bh.spgemm();
    if (rc == BHSPARSE_SUCCESS) rc = bh.update_values(val, val);
    if (rc == BHSPARSE_SUCCESS) rc = bh.get_C(colC, valC);
    return rc == BHSPARSE_SUCCESS ? 0 : 1;
}
'''


def test_c99_caller_compiles_and_links(tmp_path):
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    if not cc:
        pytest.skip("no C compiler")
    capi.load(build_if_missing=True)
    _compile(tmp_path, cc, ["-std=c99", "-pedantic"], C_CALLER, "caller.c")


def test_cxx_complex_double_caller_compiles_and_links(tmp_path):
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if not cxx:
        pytest.skip("no C++ compiler")
    capi.load(build_if_missing=True)
    _compile(tmp_path, cxx, ["-std=c++17", "-DBHSPARSE_VALUE_COMPLEX_DOUBLE"], CXX_CALLER, "caller.cpp")


# ---- the embedding reference in f64 ----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    lib = xr.compile_lib(tmp_path_factory.mktemp("exact_ref"))
    if lib is None:
        pytest.skip("gcc not found")
    return lib


@pytest.mark.parametrize("ops", ["NN", "NC", "CN", "CC", "TC"])
def test_embedding_reference_is_exact_in_f64(lib, ops):
    rng = np.random.default_rng(7)
    m, k, n = 21, 19, 25

    def stored(rows, cols, o, seed):   # a random complex128 operand, stored as op(X) needs it
        r, c = (rows, cols) if o == "N" else (cols, rows)
        X = gen.random_csr(r, c, rng.integers(0, 8, r), seed=seed, dtype=np.float64)
        return CSR(X.rows, X.cols, X.rowptr, X.col, cr.tier2(X.nnz, seed + 10))
    opA, opB = _op(stored(m, k, ops[0], 1), ops[0]), _op(stored(k, n, ops[1], 2), ops[1])
    assert opA.val.dtype == np.complex128 and opB.val.dtype == np.complex128
    want = _fraction_product(opA, opB)
    re_, im = cr.product(lib, opA, opB)
    assert re_["dtype"] == np.float64
    rows = xr.row_index(re_["rowptr"])
    assert len(want) == re_["col"].size
    for t in range(re_["col"].size):
        w = want[(int(rows[t]), int(re_["col"][t]))]
        for ref, exact, s in ((re_, w[0], w[2]), (im, w[1], w[3])):
            assert ref["cls"][t] == xr.FINITE
            # (f64 products are exact in __float128 and summed to about 113 bits: hi + lo holds the sum to 100 bits
            # of s, as test_exact_ref states for f64)
            got = Fraction(float(ref["hi"][t])) + Fraction(float(ref["lo"][t]))
            assert abs(got - exact) <= s * Fraction(1, 2 ** 100) + Fraction(1, 2 ** 1074)
            assert ref["hi"][t] == float(exact)
            assert ref["p"][t] == 2 * w[4]
            assert math.isclose(ref["s"][t], float(s), rel_tol=2.0 ** -50)


def test_complex128_generators_use_the_f64_budgets():
    v = cr.tier2(1000, 3)
    assert v.dtype == np.complex128
    # full f64 significands in both components: not representable in f32
    assert np.any(v.real != v.real.astype(np.float32)) and np.any(v.imag != v.imag.astype(np.float32))
    q = xr.tier1_bits(64, np.float64)
    g = cr.tier1(1000, q, 4)
    assert np.all(np.abs(g.real) <= 2.0 ** q) and np.all(g.real == np.round(g.real)) and np.all(g.imag == np.round(g.imag))
    assert cr.tier3(1000, 5).dtype == np.complex128


# ---- direct-mode plans with 16-byte values ---------------------------------------------------------------------
def heavy16(b, base):
    """a HEAVY bin of complex128 values: k_num_bucket3 takes the rows of at most 4096 products where the bin has any
    (SB_B8192), k_num_bucket_heavy2 the rest"""
    launches = [("heavy", 0, 0, 4096 if b == SB_B8192 else 0, P_MAX, 0)]
    if b == SB_B8192:
        launches.insert(0, ("bucket", 4096, 0, 0, 4096, 0))
    return dict(mode="heavy", cap=0, warp=False, base=base, retry=False, launches=launches)


def test_direct_plan_16_byte_values(probe):
    b8192 = {SB_B8192: (30, 30 * 5000, 0, 0.0)}
    for vs in (8, 16):
        p = plan(probe, {**RMAT, **b8192, **HEAVY_ROWS}, vs=vs)
        if vs == 8:   # (unchanged: SB_B8192 is wide at 8192 and heavy SB_B16384 starts with k_num_bucket3 at 8192)
            assert p["bins"][SB_B8192] == wide(8192, RMAT_TOP)
            assert p["heavy_base"] == RMAT_TOP + 30 * 8192
            assert p["bins"][SB_B16384] == heavy(SB_B16384, p["heavy_base"])
            continue
        # no capacity of 8192 anywhere: SB_B8192 joins the heavy bins, staged at its products
        assert all(d["cap"] < 8192 and all(l[1] <= 4096 for l in d["launches"]) for d in p["bins"].values())
        assert p["bins"][SB_G4096] == wide(4096, 8000 * 32 + 5000 * (512 + 1024 + 2048))
        assert p["heavy_base"] == RMAT_TOP
        assert p["bins"][SB_B8192] == heavy16(SB_B8192, RMAT_TOP)
        for b in (SB_B16384, SB_B32768, SB_LARGE):
            assert p["bins"][b] == heavy16(b, RMAT_TOP)
        assert p["ct_entries"] == RMAT_TOP + 30 * 5000 + 50 * 10000 + 20 * 20000 + 5 * 100000
        assert p["ct_bytes"] == p["ct_entries"] * (4 + 16)
        assert p["uses_bucket"]
    # SB_B8192 after a bin that compresses stays two-pass, with 16-byte values as with 8
    top_tight = {**RMAT, SB_G4096: (5000, 5000 * 2500, 100, 90.0), **b8192, **HEAVY_ROWS}
    for vs in (8, 16):
        p = plan(probe, top_tight, vs=vs)
        assert SB_B8192 not in p["mask"] and p["heavy_base"] == 0
    # BHB200_DEBUG_FORCE_HEAVY sends the bins above SB_B8192 to the heavy kernels, SB_B16384 without k_num_bucket3
    p = plan(probe, top_tight, vs=16, force_heavy=True)
    assert SB_B8192 not in p["mask"]
    assert all(p["bins"][b] == heavy16(b, p["heavy_base"]) for b in (SB_B16384, SB_B32768, SB_LARGE))
    # demotions: dropping the bucket kernels leaves no heavy bin
    p = plan(probe, {**RMAT, **b8192, **HEAVY_ROWS}, vs=16, drops="b")
    assert not {SB_B8192, SB_B16384, SB_B32768, SB_LARGE} & p["mask"]


# ---- diagonal-pattern plans with 16-byte values ----------------------------------------------------------------
def test_pattern_plan_probe_16_byte_values():
    d = _stencil27(128)
    info, pos, offc = _probe(d, d, 16)
    assert info[0] == 1 and info[1] == 125 and info[2] == 4
    ds = sorted(d)
    assert np.array_equal(offc[:125], sorted({a + b for a in ds for b in ds}))
    slot = {}
    for ja, a in enumerate(ds):
        for jb, b in enumerate(ds):
            assert slot.setdefault(a + b, pos[ja, jb]) == pos[ja, jb]
    assert len(set(slot.values())) == 125 and max(slot.values()) < info[3] <= 256
    # lane groups of 8 (8 lanes x 16 bytes per wavefront): 27 A diagonals x 4 groups, and the layout needs no more
    # wavefronts than that
    assert info[5] == 27 * 4 and info[4] == info[5]
    for ja in range(27):
        for j0 in range(0, 27, 8):
            g = pos[ja, j0:j0 + 8] % 8
            assert len(set(g.tolist())) == g.size
    L = capi.load()
    a = np.ascontiguousarray(d, np.int32)
    out = np.zeros(8, np.int32)
    p = lambda x: ctypes.c_void_p(x.ctypes.data)
    for vs in (0, 2, 12, 32):
        assert L.bhb200_pattern_plan_probe(p(a), a.size, p(a), a.size, vs, p(out), None, None) == capi.ERR_INVALID
