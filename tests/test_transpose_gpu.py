"""Transposed operands, C = op(A)*op(B) (include/bhsparse_b200.h: bhb200_init_data_op_*,
bhb200_init_data_device_op; csrc/stage_transpose.cu): the device transpose itself bit for bit
against a numpy stable-argsort transpose, NT / TN / TT products against the oracle on operands
transposed on the host, error reporting, aliasing, structure reuse and the device-resident
Galerkin chain P^T*(A*P)."""
import ctypes

import numpy as np
import pytest

import oracle
from benchmark_spgemm_using_csr_b200 import capi, generators as gen
from conftest import assert_csr_equal
from csr_ref import product

pytestmark = pytest.mark.gpu

N, T = capi.OP_N, capi.OP_T


@pytest.fixture(autouse=True, params=["general", "default"])
def _path(request, monkeypatch):
    """Every test runs with the diagonal-pattern mode switched off and with the library's default."""
    if request.param == "general":
        monkeypatch.setenv("BHB200_PATTERN", "off")


# ---- host references -----------------------------------------------------------------------------
def shuffle_rows(X: gen.CSR, seed=7) -> gen.CSR:
    """Same matrix, entries of every stored row in random order."""
    rng = np.random.Generator(np.random.PCG64(seed))
    order = np.arange(X.nnz)
    for i in range(X.rows):
        s, e = int(X.rowptr[i]), int(X.rowptr[i + 1])
        order[s:e] = s + rng.permutation(e - s)
    return gen.CSR(X.rows, X.cols, X.rowptr, X.col[order].copy(), X.val[order].copy())


def assert_same_csr(got: gen.CSR, want: gen.CSR, what):
    assert (got.rows, got.cols) == (want.rows, want.cols), what
    assert np.array_equal(got.rowptr, want.rowptr), f"{what}: rowptr"
    assert np.array_equal(got.col, want.col), f"{what}: col"
    assert got.val.dtype == want.val.dtype and np.array_equal(got.val, want.val), f"{what}: val"


def check_product(c: capi.Context, A, B, opA, opB, what, exact=True):
    c.spgemm()
    want = product(A, B, opA, opB)
    rtol = 0 if exact else (1e-12 if A.val.dtype == np.float64 else 1e-5)
    assert_csr_equal(c.C(), want, exact_values=exact, rtol=rtol, what=what)


# ---- 1. the transpose itself -------------------------------------------------------------------------
def _with_real(X, dt, seed=11):
    return gen.CSR(X.rows, X.cols, X.rowptr, X.col, gen.real_values(X.nnz, seed, dt))


def _transpose_cases():
    big = (1 << 24) + 3
    X = gen.random_csr(2000, big, 9, seed=3)
    X.col[-1] = big - 1                                              # the top column is used
    empty = gen.random_csr(600, 900, np.where(np.arange(600) % 3 == 0, 0, 4), seed=4)   # empty rows; most columns empty
    hub = gen.rmat(14, 16, a=0.57, b=0.19, c=0.19, d=0.05, seed=5)  # R-MAT hub columns
    one = gen.CSR(1 << 20, 64, np.arange((1 << 20) + 1, dtype=np.int32), np.full(1 << 20, 7, dtype=np.int32),
                  np.ones(1 << 20))                                  # one column holds every entry
    return {
        "cols1": gen.random_csr(1000, 1, np.arange(1000) % 2, seed=1),
        "cols200": gen.random_csr(3000, 200, 5, seed=2),
        "cols70000": gen.random_csr(20000, 70000, 8, seed=2),
        "cols2^24+3": X,
        "empty_rows_cols": empty,
        "nnz0": gen.CSR(50, 40, np.zeros(51, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0)),
        "m0": gen.CSR(10, 0, np.zeros(11, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0)),
        "rmat14_hubs": hub,
        "one_column_2^20": one,
        "unsorted_rows": shuffle_rows(gen.random_csr(5000, 3000, 12, seed=6)),
    }


_CASES = _transpose_cases()


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("name", list(_CASES))
def test_transpose_bit_exact(name, dt):
    """op(A) = X^T read back from the device: rowptr, col and val (hence perm) equal the stable host transpose."""
    X = _with_real(_CASES[name], dt)
    empty_b = gen.CSR(X.rows, 1, np.zeros(X.rows + 1, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=dt))
    c = capi.Context()
    try:
        c.init(X, empty_b, T, N)
        c.spgemm()
        (m, k, _), effA, _ = c.operands()
        effA = gen.CSR(m, k, *(t.cpu().numpy() for t in effA))
        assert_same_csr(effA, gen.transpose(X), f"{name} {dt.__name__}")
        st = c.stats()
        assert st["transposed_ops"] == 1 and st["nnzC"] == 0
        c.spgemm()                     # host operands: transposed once, kept
        assert c.stats()["ms_transpose"] == 0.0
    finally:
        c.close()


# ---- 2. products --------------------------------------------------------------------------------------
def _rect_pair(opA, opB, seed):
    m, k, n = 700, 900, 500
    A = gen.random_csr(k if opA == T else m, m if opA == T else k, 9, seed=seed)
    B = gen.random_csr(n if opB == T else k, k if opB == T else n, 7, seed=seed + 1, value_seed=5)
    return A, B


@pytest.mark.parametrize("ops", [(N, T), (T, N), (T, T)], ids=["NT", "TN", "TT"])
def test_products_diagonals(ops):
    """Nonsymmetric diagonal matrix (pattern mode on the effective operands: X^T has the negated offsets)."""
    D = gen.diagonals(3000, 3000, [-7, -1, 0, 2, 5])
    for same in (True, False):
        c = capi.Context()
        try:
            c.init(D, D, *ops, same=same)
            assert c.aliased() == int(same)
            check_product(c, D, D, *ops, f"diagonals {ops} same={same}")
        finally:
            c.close()


@pytest.mark.parametrize("ops", [(N, T), (T, N), (T, T)], ids=["NT", "TN", "TT"])
def test_products_random_rect(ops):
    for seed, dt in ((1, np.float64), (3, np.float32)):
        A, B = _rect_pair(*ops, seed)
        A, B = A.astype(dt), B.astype(dt)
        c = capi.Context()
        try:
            c.init(A, B, *ops)
            check_product(c, A, B, *ops, f"rect {ops} {dt.__name__}")
        finally:
            c.close()
    A, B = _rect_pair(*ops, 9)
    A, B = _with_real(A, np.float64), _with_real(B, np.float64, seed=12)
    c = capi.Context()
    try:
        c.init(A, B, *ops)
        check_product(c, A, B, *ops, f"rect {ops} real", exact=False)
    finally:
        c.close()


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_rmat_a_at(dt):
    A = gen.rmat(14, 16, a=0.57, b=0.19, c=0.19, d=0.05, seed=3, dtype=dt)
    c = capi.Context()
    try:
        c.init(A, A, N, T, same=True)
        assert c.aliased() == 1
        check_product(c, A, A, N, T, f"rmat14 A*A^T {dt.__name__}")
    finally:
        c.close()


def test_uniform_rect_at_a():
    A = gen.uniform_rect(40000, 10000, 8)
    c = capi.Context()
    try:
        c.init(A, A, T, N, same=True)
        assert c.aliased() == 1
        check_product(c, A, A, T, N, "uniform_rect A^T*A")
        assert c.stats()["transposed_ops"] == 1
    finally:
        c.close()


# ---- 3. errors -------------------------------------------------------------------------------------------
def test_out_of_range_column_is_reported():
    A = gen.random_csr(300, 200, 4, seed=2)
    bad = gen.CSR(A.rows, A.cols, A.rowptr, A.col.copy(), A.val)
    bad.col[17] = 200                                      # outside [0, 200)
    B = gen.random_csr(300, 50, 3, seed=3)
    c = capi.Context()
    try:
        c.init(bad, B, T, N)
        with pytest.raises(capi.BhsparseError) as e:
            c.spgemm()
        assert e.value.code == capi.ERR_INVALID and "stored A" in c.error()
        bad.col[17] = -5
        A2 = gen.random_csr(50, 200, 3, seed=4)            # op(B) = bad^T is 200 x 300
        c.init(A2, bad, N, T)
        with pytest.raises(capi.BhsparseError) as e:
            c.spgemm()
        assert e.value.code == capi.ERR_INVALID and "stored B" in c.error()
        c.init(A, B, T, N)                                 # the same context then runs a valid product
        check_product(c, A, B, T, N, "after the error")
    finally:
        c.close()


def test_duplicate_in_transposed_b_is_rejected():
    A = gen.random_csr(100, 80, 4, seed=2)
    B = gen.random_csr(60, 80, 5, seed=3)                  # stored n x k
    dup = gen.CSR(B.rows, B.cols, B.rowptr, B.col.copy(), B.val)
    dup.col[1] = dup.col[0]                                # the same (row, column) twice
    c = capi.Context()
    try:
        c.init(A, dup, N, T)
        with pytest.raises(capi.BhsparseError) as e:
            c.spgemm()
        assert e.value.code == capi.ERR_INVALID
    finally:
        c.close()


def test_unsorted_stored_rows_with_transposed_b():
    A = gen.random_csr(400, 500, 6, seed=2)
    B = shuffle_rows(gen.random_csr(300, 500, 9, seed=3))  # stored n x k, rows in random order
    c = capi.Context()
    try:
        c.init(A, B, N, T)
        check_product(c, A, B, N, T, "unsorted stored rows of B")
    finally:
        c.close()


# ---- 4. aliasing / 5. reuse -------------------------------------------------------------------------
def _vals(nnz, seed, dt):
    return gen.int_values(nnz, seed, dt)


@pytest.mark.parametrize("ops", [(N, T), (T, N), (T, T)], ids=["NT", "TN", "TT"])
def test_aliased_update_values(ops):
    A = gen.random_csr(2000, 2000, 10, seed=8) if ops == (T, T) else gen.random_csr(1500, 2500, 10, seed=8)
    c = capi.Context()
    try:
        c.init(A, A, *ops, same=True)
        assert c.aliased() == 1
        check_product(c, A, A, *ops, f"aliased {ops}")
        v, w = _vals(A.nnz, 21, np.float64), _vals(A.nnz, 22, np.float64)
        for va, vb in ((v, v), (v, w)):
            c.update_values(va, vb)
            c.spgemm_numeric()
            want = product(gen.CSR(A.rows, A.cols, A.rowptr, A.col, va),
                           gen.CSR(A.rows, A.cols, A.rowptr, A.col, vb), *ops)
            assert_csr_equal(c.C(), want, what=f"aliased {ops} update")
        assert c.aliased() == 0                            # split by the second update
    finally:
        c.close()


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("ops", [(N, T), (T, N), (T, T)], ids=["NT", "TN", "TT"])
def test_reuse_transposed_host_operands(ops, dt):
    A, B = _rect_pair(*ops, 4)
    A, B = A.astype(dt), B.astype(dt)
    c = capi.Context()
    try:
        c.init(A, B, *ops)
        c.spgemm()
        for r in range(2):
            va, vb = _vals(A.nnz, 30 + r, dt), _vals(B.nnz, 40 + r, dt)
            c.update_values(va, vb)
            c.spgemm_numeric()
            want = product(gen.CSR(A.rows, A.cols, A.rowptr, A.col, va),
                           gen.CSR(B.rows, B.cols, B.rowptr, B.col, vb), *ops)
            assert_csr_equal(c.C(), want, what=f"reuse {ops} round {r}")
            st = c.stats()
            assert st["num_bin_rows"][17] == 0 and st["ms_symbolic"] < 0.05     # no copy bin, no symbolic pass
    finally:
        c.close()


# ---- 6. the Galerkin chain, device-resident ------------------------------------------------------------
def _aggregation_prolongator(nx):
    """P of 2x2x2 aggregates on an nx^3 grid: row i has one entry, in the column of its aggregate."""
    idx = np.arange(nx ** 3)
    x, y, z = idx % nx, (idx // nx) % nx, idx // (nx * nx)
    na = nx // 2
    agg = (x // 2) + na * ((y // 2) + na * (z // 2))
    return gen.CSR(nx ** 3, na ** 3, np.arange(nx ** 3 + 1, dtype=np.int32), agg.astype(np.int32), _vals(nx ** 3, 51, np.float64))


def test_galerkin_chain_device_resident():
    import torch
    nx = 24
    A = gen.poisson27pt(nx, nx, nx)
    P = _aggregation_prolongator(nx)
    nf, nc = P.rows, P.cols
    dev = torch.device("cuda")
    tA = [torch.from_numpy(x).to(dev) for x in (A.rowptr, A.col, A.val)]
    tP = [torch.from_numpy(x).to(dev) for x in (P.rowptr, P.col, P.val)]
    stream = torch.cuda.Stream()
    torch.cuda.synchronize()
    c1, c2 = capi.Context(), capi.Context()
    try:
        for c in (c1, c2):
            c.set_stream(stream.cuda_stream)
        c1.init_device(tA, tP, nf, nf, nc)
        nnzAP = c1.spgemm()
        rp32, rp64, colC, valC = (ctypes.c_void_p() for _ in range(4))
        capi.check(c1.lib, c1.ctx, c1.lib.bhb200_get_C_device(c1.ctx, ctypes.byref(rp32), ctypes.byref(rp64), ctypes.byref(colC),
                                                              ctypes.byref(valC)))
        dp = lambda q: ctypes.c_void_p(q.value)
        rc = c2.lib.bhb200_init_data_device_op(c2.ctx, capi.DTYPE_F64, T, N, nc, nf, nc, P.nnz, ctypes.c_void_p(tP[2].data_ptr()),
                                               ctypes.c_void_p(tP[0].data_ptr()), ctypes.c_void_p(tP[1].data_ptr()),
                                               nnzAP, dp(valC), dp(rp32), dp(colC))
        capi.check(c2.lib, c2.ctx, rc)
        c2.m = nc
        c2.spgemm()

        def want(Av, Pv):
            a = gen.CSR(nf, nf, A.rowptr, A.col, Av)
            p = gen.CSR(nf, nc, P.rowptr, P.col, Pv)
            ap = oracle.spgemm(nf, nf, nc, a.rowptr, a.col, a.val, p.rowptr, p.col, p.val)
            pt = gen.transpose(p)
            return ap, oracle.spgemm(nc, nf, nc, pt.rowptr, pt.col, pt.val, *ap)

        ap, rap = want(A.val, P.val)
        assert_csr_equal(c1.C(), ap, what="A*P")
        assert_csr_equal(c2.C(), rap, what="P^T*(A*P)")
        # new values of A and P, written in place on the device; numeric-only refresh of both products
        Av2, Pv2 = _vals(A.nnz, 61, np.float64), _vals(P.nnz, 62, np.float64)
        with torch.cuda.stream(stream):
            tA[2].copy_(torch.from_numpy(Av2).to(dev, non_blocking=False))
            tP[2].copy_(torch.from_numpy(Pv2).to(dev, non_blocking=False))
        c1.spgemm_numeric()
        c2.spgemm_numeric()
        ap2, rap2 = want(Av2, Pv2)
        assert_csr_equal(c1.C(), ap2, what="A*P refreshed")
        assert_csr_equal(c2.C(), rap2, what="P^T*(A*P) refreshed")
        assert c2.stats()["ms_transpose"] >= 0.0
    finally:
        c2.close()
        c1.close()


# ---- 7. N,N is unchanged ----------------------------------------------------------------------------------
def test_nn_op_matches_plain_init():
    A = gen.rmat(12, 8, seed=2)
    B = gen.random_csr(A.cols, 3000, 6, seed=3)
    results = []
    for use_op in (False, True):
        c = capi.Context()
        try:
            if use_op:
                c.init(A, B, N, N)
            else:
                p = lambda a: ctypes.c_void_p(a.ctypes.data)
                capi.check(c.lib, c.ctx, c.lib.bhb200_init_data_f64(c.ctx, A.rows, A.cols, B.cols, A.nnz, p(A.val), p(A.rowptr),
                                                                    p(A.col), B.nnz, p(B.val), p(B.rowptr), p(B.col)))
                c.m = A.rows
            c.spgemm()
            st = c.stats()
            results.append((c.C(), st["kernel_launches"], st["transposed_ops"], st["ms_transpose"]))
        finally:
            c.close()
    (c0, l0, t0, _), (c1, l1, t1, ms1) = results
    assert all(np.array_equal(x, y) for x, y in zip(c0, c1))
    assert l0 == l1 and t0 == t1 == 0 and ms1 == 0.0
