"""The quad-precision reference (tests/exact_ref.c), the error bound and the value generators that
tests/test_values_gpu.py checks the library with -- no GPU needed.  The reference is checked against exact
rational arithmetic (fractions.Fraction) on small operands with signs, forced cancellation, explicit zeros,
+-inf, NaN, inf * 0 and subnormal products."""
import math
from fractions import Fraction

import numpy as np
import pytest

import exact_ref as xr
from benchmark_spgemm_using_csr_b200 import generators as gen
from benchmark_spgemm_using_csr_b200.generators import CSR


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    lib = xr.compile_lib(tmp_path_factory.mktemp("exact_ref"))
    if lib is None:
        pytest.skip("gcc not found")
    return lib


def _dense_fraction(A: CSR, B: CSR):
    """{(i, j): (exact sum or None, sum of |products|, p, class)} from Fractions; the class from the products
    rounded to the value type."""
    dt = A.val.dtype.type
    out = {}
    for i in range(A.rows):
        for pa in range(A.rowptr[i], A.rowptr[i + 1]):
            k, a = A.col[pa], A.val[pa]
            for q in range(B.rowptr[k], B.rowptr[k + 1]):
                j, b = B.col[q], dt(B.val[q])
                with np.errstate(all="ignore"):
                    vt = float(dt(a) * b)
                e = out.setdefault((i, int(j)), [Fraction(0), Fraction(0), 0, set()])
                if math.isfinite(a) and math.isfinite(b):
                    prod = Fraction(float(a)) * Fraction(float(b))
                    e[0] += prod
                    e[1] += abs(prod)
                e[2] += 1
                if not math.isfinite(vt):
                    e[3].add("nan" if math.isnan(vt) else "+inf" if vt > 0 else "-inf")
    res = {}
    for key, (c, s, p, seen) in out.items():
        cls = (xr.NAN if "nan" in seen or {"+inf", "-inf"} <= seen else xr.PINF if "+inf" in seen
               else xr.NINF if "-inf" in seen else xr.FINITE)
        res[key] = (c, s, p, cls)
    return res


def _special_operands(dt, seed):
    """Small operands with signed values, cancelling pairs, explicit zeros, +-inf, NaN and subnormal products."""
    rng = np.random.default_rng(seed)
    m, k, n = 30, 24, 28
    A = gen.random_csr(m, k, rng.integers(0, 10, m), seed=seed, dtype=dt)
    B = gen.random_csr(k, n, rng.integers(0, 9, k), seed=seed + 1, dtype=dt)
    tiny = 2.0 ** -70 if dt == np.float32 else 2.0 ** -530
    va = xr.tier2(A.nnz, seed + 2, dt).astype(np.float64)
    vb = xr.tier2(B.nnz, seed + 3, dt).astype(np.float64)
    # the specials, in fixed slots: A gets +inf, NaN, zeros and tiny values; B gets -inf, zeros and tiny values
    va[3], va[5], va[7], va[11:20] = np.inf, np.nan, 0.0, va[11:20] * tiny
    vb[2], vb[4], vb[9:16] = -np.inf, 0.0, vb[9:16] * tiny
    vb[20] = np.inf
    A = CSR(m, k, A.rowptr, A.col, va.astype(dt))
    B = CSR(k, n, B.rowptr, B.col, vb.astype(dt))
    return A, B


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_reference_matches_fractions(lib, dt, seed):
    for A, B in (_special_operands(dt, seed), xr.paired(*_special_operands(dt, seed + 10)[:2], seed=seed)):
        ref = xr.product(lib, A, B)
        want = _dense_fraction(A, B)
        rows = xr.row_index(ref["rowptr"])
        keys = list(zip(rows.tolist(), ref["col"].tolist()))
        assert sorted(want) == keys, "structure differs from the exact product"
        for t, key in enumerate(keys):
            c, s, p, cls = want[key]
            assert ref["p"][t] == p and ref["cls"][t] == cls, (key, ref["p"][t], p, ref["cls"][t], cls)
            if cls != xr.FINITE:
                continue
            # products of two f32 / f64 values are exact in __float128, and a few of them are summed to about 113
            # bits; hi + lo holds that sum to 106 bits, or to the smallest f64 subnormal 2^-1074 below 2^-969
            got = Fraction(float(ref["hi"][t])) + Fraction(float(ref["lo"][t]))
            assert abs(got - c) <= s * Fraction(1, 2 ** 100) + Fraction(1, 2 ** 1074), key
            assert ref["hi"][t] == float(c) and abs(Fraction(float(ref["s"][t])) - s) <= s * Fraction(1, 2 ** 53) + Fraction(1, 2 ** 1074)
    # the cases above do what they are meant to
    ref = xr.product(lib, *_special_operands(dt, seed))
    for cls in (xr.NAN, xr.FINITE):
        assert (ref["cls"] == cls).any()
    assert ((ref["cls"] == xr.PINF) | (ref["cls"] == xr.NINF)).any()


def test_inf_times_stored_zero_is_nan(lib):
    """One entry of two products: inf * 0 and 1 * 1."""
    A = CSR(1, 2, np.array([0, 2], np.int32), np.array([0, 1], np.int32), np.array([np.inf, 1.0]))
    B = CSR(2, 1, np.array([0, 1, 2], np.int32), np.array([0, 0], np.int32), np.array([0.0, 1.0]))
    ref = xr.product(lib, A, B)
    assert ref["cls"].tolist() == [xr.NAN] and ref["p"].tolist() == [2]
    B = CSR(2, 1, B.rowptr, B.col, np.array([-2.0, 1.0]))
    assert xr.product(lib, A, B)["cls"].tolist() == [xr.NINF]
    A = CSR(1, 2, A.rowptr, A.col, np.array([np.inf, np.inf]))
    assert xr.product(lib, A, B)["cls"].tolist() == [xr.NAN]              # -inf + inf


def test_f32_class_uses_f32_products(lib):
    """2^70 * 2^70 is finite in f64 but +inf in f32: the class follows what an f32 kernel multiplies."""
    A = CSR(1, 1, np.array([0, 1], np.int32), np.array([0], np.int32), np.array([2.0 ** 70]))
    for dt, cls in ((np.float64, xr.FINITE), (np.float32, xr.PINF)):
        ref = xr.product(lib, A.astype(dt), A.astype(dt))
        assert ref["cls"].tolist() == [cls]
        assert ref["hi"][0] == 2.0 ** 140 or cls != xr.FINITE


def test_subnormal_products_are_exact(lib):
    """Products far below the smallest subnormal of the value type stay exact in the reference."""
    for dt, e in ((np.float64, -530), (np.float32, -70)):
        v = np.array([3.0 * 2.0 ** e, -2.0 ** e], dtype=dt)
        A = CSR(1, 2, np.array([0, 2], np.int32), np.array([0, 1], np.int32), v)
        B = CSR(2, 1, np.array([0, 1, 2], np.int32), np.array([0, 0], np.int32), v[::-1].copy())
        ref = xr.product(lib, A, B)
        # 3*2^e * -2^e + -2^e * 3*2^e = -6 * 2^(2e), far below the f32 / f64 normal range
        assert Fraction(float(ref["hi"][0])) + Fraction(float(ref["lo"][0])) == -6 * Fraction(2) ** (2 * e)
        assert ref["s"][0] == 6 * 2.0 ** (2 * e) and ref["cls"][0] == xr.FINITE


def test_bound_hand_cases():
    u64, u32 = 2.0 ** -53, 2.0 ** -24
    # one product: u/(1-u) * s + 2 lam
    assert xr.bound(1, 1.0, np.float64) == u64 / (1 - u64) + 2 * 2.0 ** -1022
    # s = 0 leaves the underflow term alone: 2 * p * lam
    assert xr.bound(5, 0.0, np.float64) == 10 * 2.0 ** -1022
    assert xr.bound(5, 0.0, np.float32) == 10 * 2.0 ** -126
    # 2^20 f32 products: gamma = 2^-4 / (1 - 2^-4) = 1/15
    assert xr.bound(2 ** 20, 3.0, np.float32) == pytest.approx(3.0 / 15 + 2 ** 21 * 2.0 ** -126, rel=1e-15)
    # 1000 f64 products of magnitude sum 2: gamma(1000) * 2 ~ 2.2e-13
    assert xr.bound(1000, 2.0, np.float64) == pytest.approx(2000 * u64 / (1 - 1000 * u64), rel=1e-15)
    assert np.array_equal(xr.bound(np.array([1, 2]), np.array([4.0, 4.0]), np.float32),
                          [4 * u32 / (1 - u32) + 2 * 2.0 ** -126, 8 * u32 / (1 - 2 * u32) + 4 * 2.0 ** -126])


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_tier1_bit_budget(lib, dt):
    t = xr.FORMAT[dt][0]
    for p_max in (1, 2, 3, 27, 64, 65, 729, 4096, 30000, 2 ** 20):
        q = xr.tier1_bits(p_max, dt)
        assert q >= 1 and p_max * 2 ** (2 * q) <= 2 ** (t - 1), (p_max, q)
    # f64 products above 2^24 at the largest p_max the GPU cases reach: rounding through f32 shows
    assert 2 * xr.tier1_bits(30000, np.float64) > 24
    # on a real case: the reference's p_max gives q, and every entry is then exact in the value type
    A = gen.random_csr(300, 200, np.arange(300) % 60, seed=4, dtype=dt)
    B = gen.random_csr(200, 50, 30, seed=5, dtype=dt)
    p_max = int(xr.product(lib, A, B)["p"].max())
    q = xr.tier1_bits(p_max, dt)
    A = CSR(A.rows, A.cols, A.rowptr, A.col, np.full(A.nnz, -(2 ** q), dt))
    B = CSR(B.rows, B.cols, B.rowptr, B.col, np.full(B.nnz, 2 ** q, dt))
    ref = xr.product(lib, A, B)
    assert np.array_equal(ref["hi"], -ref["p"] * 2.0 ** (2 * q)) and not ref["lo"].any()
    assert np.array_equal(ref["hi"].astype(dt).astype(np.float64), ref["hi"])
    assert -ref["hi"].min() <= 2.0 ** (t - 1)
    v = xr.tier1(10000, q, 3, dt)
    assert 2 ** (q - 1) < np.abs(v).max() <= 2 ** q and (v < 0).any() and (v == 0).any() and np.array_equal(v, np.round(v))


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_generators(lib, dt):
    t = xr.FORMAT[dt][0]
    v = xr.tier2(20000, 1, dt).astype(np.float64)
    m, e = np.frexp(np.abs(v))
    assert (e >= -3).all() and (e <= 5).all() and (v < 0).any() and (v > 0).any()
    assert ((m * 2.0 ** t) % 2 == 1).mean() > 0.4          # the last significand bit is set about half the time
    v = xr.tier3(20000, 2, dt).astype(np.float64)
    assert np.isnan(v).any() and (v == np.inf).any() and (v == -np.inf).any() and (v == 0).any()
    assert (np.abs(v[np.isfinite(v) & (v != 0)]) < 2.0 ** -60).any()
    # the cancelling operands: same pattern as A*B, and |c| far below s on most entries
    A = gen.random_csr(200, 150, 12, seed=6, dtype=dt, values="real")
    B = gen.random_csr(150, 300, 9, seed=7, dtype=dt, values="real")
    A = CSR(A.rows, A.cols, A.rowptr, A.col, xr.tier2(A.nnz, 8, dt))
    B = CSR(B.rows, B.cols, B.rowptr, B.col, xr.tier2(B.nnz, 9, dt))
    ref, ref2 = xr.product(lib, A, B), xr.product(lib, *xr.paired(A, B, seed=10))
    assert np.array_equal(ref["rowptr"], ref2["rowptr"]) and np.array_equal(ref["col"], ref2["col"])
    assert np.array_equal(ref2["p"], 2 * ref["p"])
    assert np.median(np.abs(ref2["hi"]) / ref2["s"]) < 2.0 ** -8
