"""Structure-only products (BHB200_DTYPE_NONE, include/bhsparse_b200.h): the row pointers and columns of
op(A)*op(B) from operands without values.  Every product is compared bit for bit with two references on the same
operands -- the rowptr/col of the f64 product and of the CPU oracle -- and runs the same path as the f32 product:
same products, nnz(C), symbolic and numeric bins, direct-mode bins and pattern mode.  Covered: the diagonal-pattern
mode (k_pat_emit), every general-path kernel family under the switches that select it, transposed and masked
products, borrowed operands with NULL value pointers, host spill, a context switched between valued and
structure-only operands, empty shapes and the error returns."""
import ctypes

import numpy as np
import pytest

import oracle
from benchmark_spgemm_using_csr_b200 import capi, generators as gen
from benchmark_spgemm_using_csr_b200.bhsparse import bhsparse, spgemm, NUM_PLATFORMS, BHSPARSE_CUDA
from csr_ref import lower_triangle, product, restrict, symmetrize

pytestmark = pytest.mark.gpu

N, T = capi.OP_N, capi.OP_T
SAME_PATH = ["products", "nnzC", "sym_bin_rows", "num_bin_rows", "direct_bin_mask", "pattern_mode"]


def oracle_pattern(A, B, opA=N, opB=N, mask=None):
    m, _, n = capi.op_dims(A, B, opA, opB)
    C = product(A.astype(np.float64), B.astype(np.float64), opA, opB)
    rp, col, _ = restrict(C, m, n, *mask) if mask is not None else C
    return np.asarray(rp, dtype=np.int64), np.asarray(col, dtype=np.int32)


def _device(X, dt):
    """X on the device as borrowed (rowptr, col, val), val None for structure-only"""
    import torch
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return dev(X.rowptr), dev(X.col), None if dt is None else dev(X.val.astype(dt))


def run(A, B, dt, opA=N, opB=N, same=False, mask=None, device=False):
    """dt: np.float32 / np.float64, or None for structure-only operands; returns ((rowptr, col) of C, stats)."""
    dtype = capi.DTYPE_NONE if dt is None else capi.dtype_of(np.dtype(dt))
    with capi.Context() as c:
        if device:
            ta = _device(A, dt)
            c.init_device(ta, ta if B is A else _device(B, dt), *capi.op_dims(A, B, opA, opB), opA, opB, dtype)
        else:
            c.init(A, B, opA, opB, dtype, same)
        if mask is not None:
            c.set_mask(*mask)
        c.spgemm()
        return c.C()[:2], c.stats()


def check_structure(A, B, what, opA=N, opB=N, same=False, mask=None, device=False):
    """The structure-only product against the f64 product's rowptr/col and the oracle's; the same path as f32."""
    got, st = run(A, B, None, opA, opB, same, mask, device)
    f64, _ = run(A, B, np.float64, opA, opB, same, mask, device)
    _, st32 = run(A, B, np.float32, opA, opB, same, mask, device)
    want = oracle_pattern(A, B, opA, opB, mask)
    for ref, name in ((f64, "f64 product"), (want, "oracle")):
        assert np.array_equal(got[0], ref[0]), f"{what}: rowptrC differs from the {name}"
        assert np.array_equal(got[1], ref[1]), f"{what}: colC differs from the {name}"
    for key in SAME_PATH:
        assert st[key] == st32[key], f"{what}: {key} {st[key]} vs f32 {st32[key]}"
    assert st["dtype"] == capi.DTYPE_NONE
    return st


# ---- 1. diagonal-pattern mode: k_pat_emit ----------------------------------------------------------------
@pytest.mark.parametrize("case", ["poisson5pt", "poisson9pt", "poisson7pt", "poisson27pt", "rect_diagonals"])
def test_pattern_mode(case, monkeypatch):
    monkeypatch.delenv("BHB200_PATTERN", raising=False)
    if case == "rect_diagonals":
        A = gen.diagonals(3000, 2500, [-7, -1, 0, 2, 40], keep=0.9)
        B = gen.diagonals(2500, 3200, [-3, 0, 1, 5, 9, 600], keep=0.8, seed=2)
    else:
        A = {"poisson5pt": lambda: gen.poisson5pt(90, 70), "poisson9pt": lambda: gen.poisson9pt(60, 50),
             "poisson7pt": lambda: gen.poisson7pt(20, 18, 16), "poisson27pt": lambda: gen.poisson27pt(24, 20, 18)}[case]()
        B = A
    st = check_structure(A, B, case, same=B is A)
    assert st["pattern_mode"] == 1 and st["pattern_acc_len"] == 0


# ---- 2. general path, kernel by kernel (BHB200_PATTERN=off) ----------------------------------------------
def _identity(n):
    return gen.CSR(n, n, np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32), gen.int_values(n, 5))


GENERAL = {
    # single (p = 1) and ESC (p <= 32) rows
    "single_esc": ({}, lambda: (gen.random_csr(3000, 2000, np.arange(3000) % 6, seed=3),
                                gen.random_csr(2000, 5000, np.arange(2000) % 5, seed=4, value_seed=5))),
    # hash groups, CTA hash and global-bitmap rows with direct mode off
    "hash_cta_global": ({"BHB200_DIRECT": "off", "BHB200_RANGE": "off"},
                        lambda: (gen.random_csr(60, 120000, np.array([40, 300, 900, 3000, 7000, 20000] * 10), seed=9),
                                 _identity(120000))),
    "rmat_direct_off": ({"BHB200_DIRECT": "off"}, lambda: (gen.rmat(13, 16, a=0.57, b=0.19, c=0.19, d=0.05, seed=3),) * 2),
    # shared-memory bitmap (range) kernels, small and large span
    "range_all": ({"BHB200_RANGE": "all"}, lambda: (gen.poisson27pt(128, 128, 6),) * 2),
    "range_small": ({}, lambda: (gen.banded_random(5000, 300, 20, seed=8),) * 2),
    # tight direct bins, and their retry path under a forced capacity
    "direct_tight": ({"BHB200_RANGE": "off"}, lambda: (gen.poisson27pt(24, 24, 24),) * 2),
    "direct_retry_32": ({"BHB200_DEBUG_FORCE_CAP": "32", "BHB200_RANGE": "off"},
                        lambda: (gen.random_csr(6000, 3000, 20 + (np.arange(6000) * 7) % 40, seed=31),
                                 gen.random_csr(3000, 2500, 12, seed=32, value_seed=33))),
    "direct_retry_64": ({"BHB200_DEBUG_FORCE_CAP": "64", "BHB200_RANGE": "off"}, lambda: (gen.poisson27pt(16, 16, 16),) * 2),
    # wide bins: bucket sort (k_num_bucket3) and the wide direct group kernel
    "wide_bucket": ({}, lambda: (gen.random_csr(7 * 4500, 20000, np.array([12, 24, 48, 96, 150, 250, 400])[np.arange(7 * 4500) % 7],
                                                seed=41),
                                 gen.random_csr(20000, 3_000_000, 12, seed=42, value_seed=43))),
    # warp bucket on uniform_rect, and the hash kernels with it switched off
    "warp_bucket": ({}, lambda: (gen.uniform_rect(16384, 4096, 8, seed=1), gen.uniform_rect(4096, 300000, 8, seed=2, value_seed=3))),
    "warp_bucket_off": ({"BHB200_BUCKET_W": "off"},
                        lambda: (gen.uniform_rect(16384, 4096, 8, seed=1), gen.uniform_rect(4096, 300000, 8, seed=2, value_seed=3))),
    # heavy rows: sliced bucket sort, including one column that carries more products than a slice
    "heavy": ({"BHB200_DEBUG_FORCE_HEAVY": "1"},
              lambda: (gen.random_csr(6, 400000, np.array([13000, 60000, 5, 24577, 0, 30000]), seed=21), _identity(400000))),
    "heavy_duplicates": ({"BHB200_DEBUG_FORCE_HEAVY": "1"},
                         lambda: (gen.random_csr(4, 5000, np.array([4000, 1500, 700, 2]), seed=22),
                                  gen.random_csr(5000, 3000, 40, seed=23, value_seed=24))),
    "rmat_skewed": ({}, lambda: (gen.rmat(14, 8, seed=4),) * 2),
}


@pytest.mark.parametrize("case", list(GENERAL))
def test_general_path(case, monkeypatch):
    env, make = GENERAL[case]
    monkeypatch.setenv("BHB200_PATTERN", "off")
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    A, B = make()
    st = check_structure(A, B, case, same=B is A)
    assert st["pattern_mode"] == 0
    if case == "direct_tight":
        assert st["direct_rows"] > 0.9 * A.rows and st["direct_retry_rows"] == 0
    if case.startswith("direct_retry"):
        assert st["direct_retry_rows"] > 0
    if case == "hash_cta_global":
        assert st["num_bin_rows"][12] > 0 and sum(st["num_bin_rows"][3:12]) > 0
    if case.startswith("range"):
        assert sum(st["num_bin_rows"][13:17]) > 0
    if case == "wide_bucket":
        assert all((st["direct_bin_mask"] >> b) & 1 for b in range(4, 10))
    if case in ("warp_bucket", "warp_bucket_off", "heavy"):
        assert st["direct_rows"] > 0


# ---- 3. transposed operands, host and borrowed -------------------------------------------------------------
@pytest.mark.parametrize("ops", [(N, T), (T, N), (T, T)])
@pytest.mark.parametrize("device", [False, True])
def test_transposed(ops, device, monkeypatch):
    monkeypatch.setenv("BHB200_PATTERN", "off")
    m, k, n = 700, 900, 800                       # op(A) m x k, op(B) k x n; the arrays hold A and B as stored
    ra, ca = (k, m) if ops[0] == T else (m, k)
    rb, cb = (n, k) if ops[1] == T else (k, n)
    A = gen.random_csr(ra, ca, (np.arange(ra) * 5) % 60, seed=71)
    B = gen.random_csr(rb, cb, (np.arange(rb) * 3) % 25, seed=72, value_seed=73)
    check_structure(A, B, f"op {ops} device={device}", *ops, device=device)


@pytest.mark.parametrize("ops", [(N, T), (T, N), (T, T)])
def test_same_arrays_uploaded_once(ops):
    A = gen.rmat(11, 8, seed=5)
    st = check_structure(A, A, f"A op {ops} A", *ops, same=True)
    with capi.Context() as c:
        c.init(A, A, *ops, capi.DTYPE_NONE, same=True)
        assert c.lib.bhb200_operands_aliased(c.ctx) == 1
    assert st["transposed_ops"] == (1 if ops[0] == T else 0) | (2 if ops[1] == T else 0)


# ---- 4. masked products ------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["triangle", "rmat_pattern_A", "random_mask_dense_rows"])
def test_masked(case):
    if case == "triangle":                       # (L*L) .* L: every masked bin of a skewed graph, hit flags only
        L = lower_triangle(symmetrize(gen.rmat(12, 16, a=0.57, b=0.19, c=0.19, d=0.05, seed=3)))
        st = check_structure(L, L, case, same=True, mask=(L.rowptr, L.col))
    elif case == "rmat_pattern_A":
        A = gen.rmat(12, 16, seed=6)
        st = check_structure(A, A, case, same=True, mask=(A.rowptr, A.col))
    else:                                        # mask rows beyond the shared-memory tables (global bin)
        A = gen.random_csr(40, 3000, 200, seed=81)
        B = gen.random_csr(3000, 30000, 60, seed=82, value_seed=83)
        M = gen.random_csr(40, 30000, np.array([9000, 20000, 100, 0] * 10), seed=84)
        st = check_structure(A, B, case, mask=(M.rowptr, M.col))
        assert st["mask_bin_rows"][8] > 0
    assert st["masked"] == 1


# ---- 5. borrowed operands: NULL value pointers, and the pattern of valued device arrays ----------------------
@pytest.mark.parametrize("pattern", ["on", "off"])
def test_borrowed_null_values(pattern, monkeypatch):
    monkeypatch.setenv("BHB200_PATTERN", pattern)
    A = gen.poisson27pt(14, 14, 14)
    check_structure(A, A, f"borrowed stencil pattern={pattern}", device=True)
    R = gen.rmat(12, 16, a=0.57, b=0.19, c=0.19, d=0.05, seed=8)
    check_structure(R, R, f"borrowed rmat pattern={pattern}", device=True)
    with capi.Context() as c:   # valued device arrays read as structure: the values are never touched
        tr = _device(R, np.float64)
        c.init_device(tr, tr, R.rows, R.cols, R.cols, dtype=capi.DTYPE_NONE)
        c.spgemm()
        want = oracle_pattern(R, R)
        got = c.C()
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


# ---- 6. host spill ---------------------------------------------------------------------------------------
def test_host_spill(monkeypatch):
    monkeypatch.setenv("BHB200_DEBUG_DEVICE_CAP", "65536")
    A = gen.poisson27pt(16, 16, 16)
    st = check_structure(A, A, "spill stencil", same=True)
    assert st["spill_bytes"] >= 4 * st["nnzC"]
    R = gen.rmat(12, 16, a=0.57, b=0.19, c=0.19, d=0.05)
    st = check_structure(R, R, "spill rmat", same=True)
    assert st["spill_bytes"] > 0


# ---- 7. one context: f64, structure-only, f64 again (pattern plans keyed on the value size) ----------------
@pytest.mark.parametrize("pattern", ["on", "off"])
def test_context_switches_value_type(pattern, monkeypatch):
    monkeypatch.setenv("BHB200_PATTERN", pattern)
    A = gen.poisson27pt(12, 12, 12)
    want = oracle_pattern(A, A)
    with capi.Context() as c:
        for dt in (np.float64, None, np.float64, None, np.float32):
            c.init(A, A, dtype=capi.DTYPE_NONE if dt is None else capi.dtype_of(np.dtype(dt)), same=True)
            c.spgemm()
            got = c.C()
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), f"{dt}"
            st = c.stats()
            assert st["dtype"] == (capi.DTYPE_NONE if dt is None else capi.DTYPE_F32 if dt == np.float32 else capi.DTYPE_F64)
            assert st["pattern_mode"] == (1 if pattern == "on" else 0)
            if dt is not None:   # the values are right after a structure-only product on the same context
                nnz = int(c.lib.bhb200_get_nnzC(c.ctx))
                val = np.empty(nnz, dtype=dt)
                capi.check(c.lib, c.ctx, c.lib.bhb200_get_C_range(c.ctx, 0, nnz, None, ctypes.c_void_p(val.ctypes.data)))
                _, _, wv = oracle.spgemm(A.rows, A.cols, A.cols, A.rowptr, A.col, A.val.astype(dt), A.rowptr, A.col,
                                         A.val.astype(dt))
                assert np.array_equal(val, wv)


# ---- 8. empty shapes -----------------------------------------------------------------------------------------
def test_empty_shapes():
    cases = [
        (gen.CSR(0, 5, np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0)),            # m = 0
         gen.CSR(5, 4, np.zeros(6, np.int32), np.zeros(0, np.int32), np.zeros(0))),
        (gen.CSR(4, 128, np.zeros(5, np.int32), np.zeros(0, np.int32), np.zeros(0)), gen.rmat(7, 4, seed=2)),   # nnzA = 0
        (gen.random_csr(30, 6, 2, seed=3), gen.CSR(6, 0, np.zeros(7, np.int32), np.zeros(0, np.int32), np.zeros(0))),  # n = 0
    ]
    for i, (A, B) in enumerate(cases):
        (rp, col), st = run(A, B, None)
        assert col.size == 0 and np.all(rp == 0) and rp.size == A.rows + 1, f"case {i}"
        assert st["nnzC"] == 0


# ---- 9. errors and the getters -------------------------------------------------------------------------------
def test_error_returns_and_getters():
    A = gen.rmat(10, 8, seed=2)
    c = capi.Context()
    try:
        lib, ctx = c.lib, c.ctx
        rp = np.zeros(A.rows + 1, dtype=np.int32)
        assert lib.bhb200_get_C_structure(ctx, ctypes.c_void_p(rp.ctypes.data), None) == capi.ERR_INVALID   # before spgemm
        assert lib.bhb200_get_C_structure(None, None, None) == capi.ERR_INVALID
        c.init(A, A, dtype=capi.DTYPE_NONE, same=True)
        nnz = c.spgemm()
        buf = np.empty(max(nnz, 1), dtype=np.float64)
        vp = ctypes.c_void_p(buf.ctypes.data)
        for call, what in ((lambda: lib.bhb200_get_C_f64(ctx, None, None, vp), "get_C"),
                           (lambda: lib.bhb200_get_C_f32(ctx, None, None, None), "get_C"),
                           (lambda: lib.bhb200_get_C_range(ctx, 0, nnz, None, vp), "get_C_range"),
                           (lambda: lib.bhb200_update_values_f64(ctx, vp, vp), "update_values"),
                           (lambda: lib.bhb200_update_values_f32(ctx, vp, None), "update_values"),
                           (lambda: lib.bhb200_spgemm_numeric(ctx), "spgemm_numeric")):
            assert call() == capi.ERR_INVALID, what
            assert "structure-only" in c.error() and what in c.error()
        import torch
        dcol = torch.empty(nnz, dtype=torch.int32, device="cuda")
        dval = torch.empty(nnz, dtype=torch.float64, device="cuda")
        assert lib.bhb200_copy_C_to_device(ctx, None, ctypes.c_void_p(dcol.data_ptr()),
                                           ctypes.c_void_p(dval.data_ptr())) == capi.ERR_INVALID
        capi.check(lib, ctx, lib.bhb200_copy_C_to_device(ctx, None, ctypes.c_void_p(dcol.data_ptr()), None))
        want = oracle_pattern(A, A)
        assert np.array_equal(dcol.cpu().numpy(), want[1])
        # the range getter without values, the int64 row pointers, the device view with valC = NULL
        col = np.empty(nnz, dtype=np.int32)
        capi.check(lib, ctx, lib.bhb200_get_C_range(ctx, 0, nnz, ctypes.c_void_p(col.ctypes.data), None))
        rp64 = np.empty(A.rows + 1, dtype=np.int64)
        capi.check(lib, ctx, lib.bhb200_get_rowptrC_i64(ctx, ctypes.c_void_p(rp64.ctypes.data)))
        assert np.array_equal(col, want[1]) and np.array_equal(rp64, want[0])
        ptrs = [ctypes.c_void_p() for _ in range(4)]
        ptrs[3] = ctypes.c_void_p(1)
        capi.check(lib, ctx, lib.bhb200_get_C_device(ctx, *[ctypes.byref(p) for p in ptrs]))
        assert ptrs[2].value and not ptrs[3].value
        # structure of a valued product, and the valued getters again after re-initialising with values
        c.init(A, A, same=True)
        c.spgemm()
        srp, scol = np.empty(A.rows + 1, np.int32), np.empty(nnz, np.int32)
        capi.check(lib, ctx, lib.bhb200_get_C_structure(ctx, ctypes.c_void_p(srp.ctypes.data), ctypes.c_void_p(scol.ctypes.data)))
        assert np.array_equal(srp, want[0]) and np.array_equal(scol, want[1])
        capi.check(lib, ctx, lib.bhb200_get_C_f64(ctx, None, None, vp))
        # null columns with nonzeros, bad dtype
        z = np.zeros(A.rows + 1, dtype=np.int32)
        assert lib.bhb200_init_data_structure(ctx, N, N, A.rows, A.cols, A.cols, A.nnz, ctypes.c_void_p(A.rowptr.ctypes.data),
                                              None, A.nnz, ctypes.c_void_p(A.rowptr.ctypes.data), None) == capi.ERR_INVALID
        assert lib.bhb200_init_data_device(ctx, 3, 1, 1, 1, 0, None, ctypes.c_void_p(z.ctypes.data), None, 0, None,
                                           ctypes.c_void_p(z.ctypes.data), None) == capi.ERR_INVALID
        # valued device operands still need their values
        assert lib.bhb200_init_data_device(ctx, capi.DTYPE_F64, A.rows, A.cols, A.cols, A.nnz, None,
                                           ctypes.c_void_p(dcol.data_ptr()), ctypes.c_void_p(dcol.data_ptr()), A.nnz, None,
                                           ctypes.c_void_p(dcol.data_ptr()), ctypes.c_void_p(dcol.data_ptr())) == capi.ERR_INVALID
    finally:
        c.close()


def test_python_interface():
    A = gen.rmat(11, 8, seed=4)
    B = gen.uniform_rect(A.cols, 3000, 4, seed=5)
    rp, col, val = spgemm(A, B, structure_only=True)
    want = oracle_pattern(A, B)
    assert val is None and np.array_equal(rp, want[0]) and np.array_equal(col, want[1])
    rp2, col2, val2 = spgemm(A, B, transA=True, structure_only=True)
    want = oracle_pattern(A, B, T)
    assert val2 is None and np.array_equal(rp2, want[0]) and np.array_equal(col2, want[1])
    platforms = [False] * NUM_PLATFORMS
    platforms[BHSPARSE_CUDA] = True
    bh = bhsparse()
    try:
        assert bh.initPlatform(platforms) == 0
        rowptrC = np.zeros(A.rows + 1, dtype=np.int32)
        # exactly one of the value arrays missing
        assert bh.initData(A.rows, A.cols, B.cols, A.nnz, A.val, A.rowptr, A.col, B.nnz, None, B.rowptr, B.col,
                           rowptrC) == capi.ERR_INVALID
        assert bh.initData(A.rows, A.cols, B.cols, A.nnz, None, A.rowptr, A.col, B.nnz, B.val, B.rowptr, B.col,
                           rowptrC) == capi.ERR_INVALID
        assert bh.initData(A.rows, A.cols, B.cols, A.nnz, None, A.rowptr, A.col, B.nnz, None, B.rowptr, B.col, rowptrC) == 0
        assert bh.spgemm() == 0
        want = oracle_pattern(A, B)
        assert np.array_equal(rowptrC, want[0])
        colC = np.empty(bh.get_nnzC(), dtype=np.int32)
        assert bh.get_C(colC, None) == 0 and np.array_equal(colC, want[1])
        assert bh.get_C(colC, np.empty(colC.size)) == capi.ERR_INVALID
        c2, v2 = bh.get_C_range(3, 10)
        assert v2 is None and np.array_equal(c2, want[1][3:13])
        assert bh.stats()["dtype"] == capi.DTYPE_NONE
    finally:
        bh.freePlatform()


# ---- 10. workspace --------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["stencil", "rmat", "rect"])
def test_workspace_below_f64(case, monkeypatch):
    if case == "rect":
        A, B = gen.uniform_rect(16384, 4096, 8, seed=1), gen.uniform_rect(4096, 300000, 8, seed=2, value_seed=3)
    else:
        A = gen.poisson27pt(20, 20, 20) if case == "stencil" else gen.rmat(13, 16, seed=5)
        B = A
    _, st = run(A, B, None, same=B is A)
    _, st64 = run(A, B, np.float64, same=B is A)
    assert st["workspace_bytes"] < st64["workspace_bytes"]
    assert st["bytes_compulsory"] < st64["bytes_compulsory"]
