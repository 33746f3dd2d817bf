"""Masked products C = M .* (op(A)*op(B)) (include/bhsparse_b200.h: bhb200_set_mask*,
csrc/stage_masked.cu) against the oracle's unmasked product restricted to the pattern of M:
operand families and mask shapes, every masked kernel bin at its boundaries, cancellation,
triangle counting with host and device-resident L, transposed operands, the mask's lifetime,
error reporting, host-memory staging and empty shapes."""
import ctypes

import numpy as np
import pytest

from benchmark_spgemm_using_csr_b200 import capi, generators as gen
from conftest import assert_csr_equal
from csr_ref import keys, lower_triangle, product, restrict, symmetrize
from ref_cases import _kat

pytestmark = pytest.mark.gpu

N, T = capi.OP_N, capi.OP_T


# ---- references -------------------------------------------------------------------------------------
def unmasked(A, B, opA=N, opB=N):
    m, _, n = capi.op_dims(A, B, opA, opB)
    return product(A, B, opA, opB), m, n


def pattern(rows, cols, rowptr, col):
    return np.asarray(rowptr, dtype=np.int32), np.asarray(col, dtype=np.int32)


def subset(rp, col, keep, seed):
    """Random subset of a pattern: each entry kept with probability `keep`."""
    rng = np.random.Generator(np.random.PCG64(seed))
    sel = rng.random(col.size) < keep
    m = len(rp) - 1
    rows = np.repeat(np.arange(m), np.diff(np.asarray(rp, dtype=np.int64)))
    rowptr = np.zeros(m + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows[sel], minlength=m), out=rowptr[1:])
    return rowptr.astype(np.int32), col[sel].astype(np.int32)


def union(p, q, n):
    m = len(p[0]) - 1
    k = np.union1d(keys(*p, n), keys(*q, n))
    rowptr = np.zeros(m + 1, dtype=np.int64)
    np.cumsum(np.bincount(k // n, minlength=m), out=rowptr[1:])
    return rowptr.astype(np.int32), (k % n).astype(np.int32)


@pytest.fixture
def ctx():
    with capi.Context() as c:
        yield c


def rtol_of(dt, values):
    if values == "int":
        return True, 0.0
    return False, (1e-12 if dt == np.float64 else 1e-5)


def check_masked(c, A, B, rpM, colM, what, opA=N, opB=N, values="int"):
    c.set_mask(rpM, colM)
    c.spgemm()
    C, m, n = unmasked(A, B, opA, opB)
    want = restrict(C, m, n, rpM, colM)
    exact, rtol = rtol_of(A.val.dtype, values)
    assert_csr_equal(c.C(), want, exact_values=exact, rtol=rtol, what=what)
    st = c.stats()
    assert st["masked"] == 1 and st["nnzM"] == colM.size and st["nnzC"] == want[1].size
    return st


# ---- 1. operand families x mask shapes --------------------------------------------------------------
def _cases():
    return [
        ("kat_small", lambda dt, v: _kat(dt)),
        ("poisson5pt", lambda dt, v: (gen.poisson5pt(40, 40, dtype=dt, values=v),) * 2),
        ("poisson27pt", lambda dt, v: (gen.poisson27pt(12, 12, 12, dtype=dt, values=v),) * 2),
        ("rmat10", lambda dt, v: (gen.rmat(10, 8, dtype=dt, values=v),) * 2),
        ("rmat12", lambda dt, v: (gen.rmat(12, 16, dtype=dt, values=v),) * 2),
        ("rmat14", lambda dt, v: (gen.rmat(14, 8, a=0.57, b=0.19, c=0.19, d=0.05, dtype=dt, values=v),) * 2),
        ("uniform_rect", lambda dt, v: (gen.uniform_rect(3000, 2000, 8, seed=1, dtype=dt, values=v),
                                        gen.uniform_rect(2000, 2500, 8, seed=2, value_seed=3, dtype=dt, values=v))),
        ("random_csr", lambda dt, v: (gen.random_csr(500, 3000, np.arange(500) * 7 % 900, seed=3, dtype=dt, values=v),
                                      gen.random_csr(3000, 4000, 6, seed=4, value_seed=5, dtype=dt, values=v))),
        ("banded_random", lambda dt, v: (gen.banded_random(3000, 40, 12, dtype=dt, values=v),) * 2),
    ]


MASKS = ["pattern_A", "keep0", "keep0.1", "keep0.5", "keep1", "outside", "empty_rows", "superset"]


def make_mask(kind, A, C, m, n, seed=5):
    rpC, colC = np.asarray(C[0], dtype=np.int32), C[1]
    if kind == "pattern_A":
        return (A.rowptr, A.col) if A.rows == m and A.cols == n else subset(rpC, colC, 0.3, seed)
    if kind.startswith("keep"):
        return subset(rpC, colC, float(kind[4:]), seed)
    rnd = gen.random_csr(m, n, np.random.Generator(np.random.PCG64(seed)).integers(0, 40, m), seed=seed)
    if kind == "outside":
        return rnd.rowptr, rnd.col
    if kind == "empty_rows":
        rp, col = union((rnd.rowptr, rnd.col), subset(rpC, colC, 0.5, seed), n)
        rows = np.repeat(np.arange(m), np.diff(rp.astype(np.int64)))
        sel = rows % 3 != 0
        rowptr = np.zeros(m + 1, dtype=np.int64)
        np.cumsum(np.bincount(rows[sel], minlength=m), out=rowptr[1:])
        return rowptr.astype(np.int32), col[sel]
    if kind == "superset":
        return union((rnd.rowptr, rnd.col), (rpC, colC), n)
    raise ValueError(kind)


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("name,build", _cases(), ids=[c[0] for c in _cases()])
def test_masked_product(ctx, name, build, dt):
    for values in ("int", "real"):
        A, B = build(dt, values)
        C, m, n = unmasked(A, B)
        ctx.init(A, B, same=A is B)
        for kind in MASKS:
            rpM, colM = make_mask(kind, A, C, m, n)
            check_masked(ctx, A, B, rpM, colM, f"{name}/{values}/{kind}", values=values)
            if kind == "superset":   # a superset of C's pattern is the unmasked product
                exact, rtol = rtol_of(dt, values)
                assert_csr_equal(ctx.C(), C, exact_values=exact, rtol=rtol, what=f"{name}/{values}/superset")


# ---- 2. every masked bin, rows at its boundaries ----------------------------------------------------
# B: rows of length 1, 7, 300 and 4000 (the last two longer than LONG_B = 256: whole-CTA B rows)
_B_LENS = [(0, 1024, 1), (1024, 2048, 7), (2048, 2560, 300), (2560, 2600, 4000)]
_NB = 20000


def _bin_operands(rows, dt):
    """rows = [(p, m)]: row i of A has exactly p products, row i of M has m entries."""
    rng = np.random.Generator(np.random.PCG64(17))
    lens = np.zeros(2600, dtype=np.int64)
    for lo, hi, ln in _B_LENS:
        lens[lo:hi] = ln
    B = gen.random_csr(2600, _NB, lens, seed=18, dtype=dt)
    acols, mcols = [], []
    for p, mm in rows:
        sel = []
        for lo, hi, ln in reversed(_B_LENS):
            q = min(p // ln, hi - lo)
            sel.append(lo + rng.permutation(hi - lo)[:q])
            p -= q * ln
        assert p == 0
        acols.append(np.sort(np.concatenate(sel)))
        mcols.append(np.sort(rng.permutation(_NB)[:mm]))
    arp = np.concatenate([[0], np.cumsum([len(a) for a in acols])]).astype(np.int32)
    A = gen.CSR(len(rows), 2600, arp, np.concatenate(acols).astype(np.int32), gen.int_values(int(arp[-1]), 19, dt))
    mrp = np.concatenate([[0], np.cumsum([len(x) for x in mcols])]).astype(np.int32)
    return A, B, mrp, np.concatenate(mcols).astype(np.int32)


# (products, mask entries) -> masked bin (capi.MASK_BIN_NAMES)
BIN_ROWS = [
    ((0, 5), 0), ((9, 0), 0),
    ((1, 3), 1), ((32, 40), 1), ((32, 9000), 1),
    ((33, 1), 2), ((33, 32), 2), ((2048, 32), 2),
    ((33, 33), 3), ((2048, 128), 3),
    ((33, 129), 4), ((2048, 512), 4),
    ((2049, 1), 5), ((2049, 512), 5), ((100000, 20), 5),
    ((40, 513), 6), ((5000, 2048), 6),
    ((40, 2049), 7), ((9000, 8192), 7),
    ((40, 8193), 8), ((30000, 20000), 8),
]


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_every_masked_bin(ctx, dt):
    A, B, rpM, colM = _bin_operands([r for r, _ in BIN_ROWS], dt)
    ctx.init(A, B)
    st = check_masked(ctx, A, B, rpM, colM, "bins", values="int" if dt == np.float64 else "real")
    want = np.bincount([b for _, b in BIN_ROWS], minlength=capi.NUM_MASK_BINS)
    assert st["mask_bin_rows"] == list(want), st["mask_bin_rows"]


def test_cancellation_keeps_explicit_zero(ctx):
    # row 0: 40 products (warp bin) that sum to 0 in column 0; row 1: 2 products (ESC bin) that do the same
    k = 40
    B = gen.CSR(k, 2, np.arange(0, 2 * k + 1, 2, dtype=np.int32), np.tile([0, 1], k).astype(np.int32),
                np.array([(1.0 if i % 2 == 0 else -1.0) for i in range(k) for _ in (0, 1)]))
    A = gen.CSR(2, k, np.array([0, k, k + 2], np.int32), np.concatenate([np.arange(k), [0, 1]]).astype(np.int32),
                np.ones(k + 2))
    ctx.init(A, B)
    ctx.set_mask(np.array([0, 1, 2], np.int32), np.array([0, 0], np.int32))
    ctx.spgemm()
    rp, col, val = ctx.C()
    assert list(rp) == [0, 1, 2] and list(col) == [0, 0] and list(val) == [0.0, 0.0]


# ---- 3. triangle counting ---------------------------------------------------------------------------
def _lower(scale):
    """L = strictly lower triangle of the symmetrized R-MAT graph with values 1, and its triangle count by scipy."""
    sp = pytest.importorskip("scipy.sparse")
    L = lower_triangle(symmetrize(gen.rmat(scale, 16)))
    L = gen.CSR(L.rows, L.cols, L.rowptr, L.col, np.ones(L.nnz))
    S = sp.csr_matrix((L.val, L.col, L.rowptr), shape=(L.rows, L.cols))
    return L, float((S @ S).multiply(S).sum())


@pytest.mark.parametrize("scale", [12, 13, 14])
def test_triangle_counting(ctx, scale):
    import torch
    X, triangles = _lower(scale)
    n = X.rows
    ctx.init(X, X, same=True)
    ctx.set_mask(X.rowptr, X.col)
    ctx.spgemm()
    assert ctx.C()[2].sum() == triangles
    # device-resident L as A, B and M, no copy
    rp, col, val = (torch.from_numpy(X.rowptr).cuda(), torch.from_numpy(X.col).cuda(), torch.from_numpy(X.val).cuda())
    d = capi.Context()
    try:
        d.init_device((rp, col, val), (rp, col, val), n, n, n)
        d.set_mask_device(rp, col)
        d.spgemm()
        assert d.C()[2].sum() == triangles
        assert d.stats()["masked"] == 1
    finally:
        d.close()


# ---- 4. transposed operands -------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_a_at_masked(ctx, dt):
    import torch
    A = gen.random_csr(800, 1200, np.arange(800) % 60, seed=21, dtype=dt)
    C, m, n = unmasked(A, A, N, T)
    rpM, colM = union(subset(np.asarray(C[0], np.int32), C[1], 0.3, 22), make_mask("outside", A, C, m, n, 23), n)
    ctx.init(A, A, N, T, same=True)
    check_masked(ctx, A, A, rpM, colM, "A*A^T host", N, T)
    dev = tuple(torch.from_numpy(x).cuda() for x in (A.rowptr, A.col, A.val))
    d = capi.Context()
    try:
        d.init_device(dev, dev, 800, 1200, 800, N, T)
        check_masked(d, A, A, rpM, colM, "A*A^T borrowed", N, T)
    finally:
        d.close()


# ---- 5. lifetime ------------------------------------------------------------------------------------
def test_lifecycle(ctx):
    A = gen.rmat(11, 8)
    C, m, n = unmasked(A, A)
    ctx.init(A, A, same=True)
    m1 = subset(np.asarray(C[0], np.int32), C[1], 0.5, 1)
    m2 = make_mask("outside", A, C, m, n, 2)
    check_masked(ctx, A, A, *m1, "mask 1")
    check_masked(ctx, A, A, *m2, "mask 2 replaces mask 1")
    # clear: the unmasked product, with the launches of a fresh context
    ctx.clear_mask()
    assert_csr_equal(ctx.C(), restrict(C, m, n, *m2), what="C readable after clear_mask")
    with pytest.raises(capi.BhsparseError, match="mask") as e:
        ctx.spgemm_numeric()
    assert e.value.code == capi.ERR_INVALID and "mask" in ctx.error()
    ctx.spgemm()
    assert_csr_equal(ctx.C(), C, what="after clear_mask")
    fresh = capi.Context()
    try:
        fresh.init(A, A, same=True)
        fresh.spgemm()
        assert ctx.stats()["kernel_launches"] == fresh.stats()["kernel_launches"]
        assert ctx.stats()["masked"] == 0
    finally:
        fresh.close()
    # init_data clears the mask
    check_masked(ctx, A, A, *m1, "mask again")
    ctx.init(A, A, same=True)
    ctx.spgemm()
    assert_csr_equal(ctx.C(), C, what="init_data cleared the mask")
    # set_mask without a new spgemm: no numeric-only update
    ctx.set_mask(*m1)
    with pytest.raises(capi.BhsparseError, match="mask") as e:
        ctx.spgemm_numeric()
    assert e.value.code == capi.ERR_INVALID and "mask" in ctx.error()
    assert_csr_equal(ctx.C(), C, what="C readable after set_mask")


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_update_values_and_numeric(ctx, dt):
    A, B, rpM, colM = _bin_operands([r for r, _ in BIN_ROWS], dt)
    ctx.init(A, B)
    check_masked(ctx, A, B, rpM, colM, "first values", values="real")
    A2 = gen.CSR(A.rows, A.cols, A.rowptr, A.col, gen.int_values(A.nnz, 31, dt))
    B2 = gen.CSR(B.rows, B.cols, B.rowptr, B.col, gen.int_values(B.nnz, 32, dt))
    ctx.update_values(A2.val, B2.val)
    ctx.spgemm_numeric()
    C, m, n = unmasked(A2, B2)
    exact, rtol = rtol_of(dt, "int" if dt == np.float64 else "real")
    assert_csr_equal(ctx.C(), restrict(C, m, n, rpM, colM), exact_values=exact, rtol=rtol, what="numeric after update")


# ---- 6. errors --------------------------------------------------------------------------------------
def _bad_masks(m, n):
    rp = np.arange(0, 2 * m + 1, 2, dtype=np.int32)
    col = np.tile(np.array([1, 3], np.int32), m)
    unsorted = col.copy()
    unsorted[4:6] = [3, 1]
    dup = col.copy()
    dup[5] = 1
    out = col.copy()
    out[7] = n
    neg = col.copy()
    neg[2] = -1
    bad_rp = rp.copy()
    bad_rp[3] = bad_rp[2] - 1
    short = rp.copy()
    short[-1] -= 1
    return [("unsorted", rp, unsorted, "sorted"), ("duplicate", rp, dup, "duplicate"), ("out of range", rp, out, "outside"),
            ("negative", rp, neg, "outside"), ("rowptr not monotone", bad_rp, col, "row pointers"),
            ("rowptr[m] != nnzM", short, col, "row pointers")]


def test_mask_errors(ctx):
    A = gen.poisson5pt(8, 8)
    with pytest.raises(capi.BhsparseError, match="mask") as e:   # before init_data
        ctx.set_mask(A.rowptr, A.col)
    assert e.value.code == capi.ERR_INVALID and "mask" in ctx.error()
    ctx.init(A, A, same=True)
    for what, rp, col, word in _bad_masks(A.rows, A.cols):
        ctx.set_mask(rp, col)
        with pytest.raises(capi.BhsparseError) as e:
            ctx.spgemm()
        assert e.value.code == capi.ERR_INVALID, what
        assert "mask" in ctx.error() and word in ctx.error(), (what, ctx.error())
    check_masked(ctx, A, A, A.rowptr, A.col, "a good mask after bad ones")


def test_mask_on_dist_context(ctx):
    lib = ctx.lib
    uid = ctypes.create_string_buffer(capi.DIST_ID_BYTES)
    rc = lib.bhb200_dist_unique_id(uid)
    if rc != capi.SUCCESS:
        pytest.skip("NCCL not available")
    capi.check(lib, ctx.ctx, lib.bhb200_dist_init(ctx.ctx, 0, 1, uid))
    import torch
    A = gen.poisson5pt(8, 8)
    dev = [torch.from_numpy(x).cuda() for x in (A.rowptr, A.col, A.val)]
    capi.check(lib, ctx.ctx, lib.bhb200_dist_setup_square(ctx.ctx, 0, capi.DTYPE_F64, A.rows, A.nnz,
                                                          *[ctypes.c_void_p(t.data_ptr()) for t in dev]))
    with pytest.raises(capi.BhsparseError, match="mask") as e:
        ctx.set_mask(A.rowptr, A.col)
    assert e.value.code == capi.ERR_INVALID and "mask" in ctx.error()
    capi.check(lib, ctx.ctx, lib.bhb200_dist_finalize(ctx.ctx))


# ---- 7. staging and C in host memory; empty shapes --------------------------------------------------
def test_device_cap_spills(monkeypatch):
    A = gen.rmat(12, 16)
    C, m, n = unmasked(A, A)
    rpM, colM = union(subset(np.asarray(C[0], np.int32), C[1], 0.5, 3), (A.rowptr, A.col), n)
    want = restrict(C, m, n, rpM, colM)
    monkeypatch.setenv("BHB200_DEBUG_DEVICE_CAP", "4096")
    c = capi.Context()
    try:
        c.init(A, A, same=True)
        st = check_masked(c, A, A, rpM, colM, "spilled")
        assert st["spill_bytes"] > 0
        assert_csr_equal(c.C(), want, what="spilled")
    finally:
        c.close()


def test_empty_shapes(ctx):
    E = gen.CSR(0, 5, np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0))
    B = gen.poisson5pt(5, 1)
    ctx.init(E, B)
    ctx.set_mask(np.zeros(1, np.int32), np.zeros(0, np.int32))
    ctx.spgemm()
    assert ctx.lib.bhb200_get_nnzC(ctx.ctx) == 0
    A = gen.poisson5pt(6, 6)
    ctx.init(A, A, same=True)
    ctx.set_mask(np.zeros(A.rows + 1, np.int32), np.zeros(0, np.int32))
    ctx.spgemm()
    assert ctx.lib.bhb200_get_nnzC(ctx.ctx) == 0
    assert list(ctx.C()[0]) == [0] * (A.rows + 1)
