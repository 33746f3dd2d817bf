"""Parity of the CUDA path (through the C-ABI / the bhsparse class mirror) against
the CPU oracle on the same seeded inputs.  rowptrC and colC bit-exact; values
bit-exact for the integer-valued inputs the reference driver uses (main.cu:82,93),
<= 1e-12 relative (double) / 1e-5 (float) for real-valued inputs -- the tolerances
BASELINE.json's north_star states (the reference itself only checks 10 %,
ref_spgemm.h:110)."""
import os

import numpy as np
import pytest

import oracle
from benchmark_spgemm_using_csr_b200 import (BHSPARSE_CUDA, BHSPARSE_SUCCESS, NUM_PLATFORMS, bhsparse, capi,
                                             generators as gen, spgemm)
from benchmark_spgemm_using_csr_b200.generators import CSR
from conftest import assert_csr_equal

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["general", "default"])
def _path(request, monkeypatch):
    """Every test of this module runs twice: with the diagonal-pattern mode switched off (the
    general hash / ESC / range / bitmap kernels these tests were written for) and with the
    library's default (structured operands then take csrc/stage_pattern.cuh)."""
    if request.param == "general":
        monkeypatch.setenv("BHB200_PATTERN", "off")

RTOL = {np.float64: 1e-12, np.float32: 1e-5}


def _oracle(A, B):
    return oracle.spgemm(A.rows, A.cols, B.cols, A.rowptr, A.col, A.val, B.rowptr, B.col, B.val)


def _check(A, B, what, exact=True):
    got = spgemm(A, B, return_stats=True, return_row_products=True)
    st = got[3]
    want = _oracle(A, B)
    dt = A.val.dtype.type
    assert_csr_equal(got[:3], want, exact_values=exact, rtol=RTOL[dt], what=what)
    prod, total = oracle.row_products(A.rows, A.rowptr, A.col, B.rowptr)
    assert st["products"] == total and st["nnzC"] == want[0][-1]
    # compute_nnzCt (bhsparse_cuda.h:210-237): the per-row upper bounds, row by row
    assert np.array_equal(got[4].astype(np.int64), prod), f"{what}: per-row product counts differ"
    return st


# ---- the reference's own cases ------------------------------------------------
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_kat_small_reference_call_sequence(golden, dt):
    """test_small_spgemm (main.cu:149-246), call by call (main.cu:203-229)."""
    g = golden("kat_small")
    m, k, n = int(g["m"]), int(g["k"]), int(g["n"])
    platforms = [False] * NUM_PLATFORMS
    platforms[BHSPARSE_CUDA] = True
    csrRowPtrC = np.zeros(m + 1, dtype=np.int32)
    bh = bhsparse()
    assert bh.initPlatform(platforms) == BHSPARSE_SUCCESS
    assert bh.initData(m, k, n, 6, g["valA"].astype(dt), g["rowptrA"], g["colA"],
                       7, g["valB"].astype(dt), g["rowptrB"], g["colB"], csrRowPtrC) == BHSPARSE_SUCCESS
    assert bh.spgemm() == BHSPARSE_SUCCESS
    nnzC = bh.get_nnzC()
    assert nnzC == 6
    csrColIndC = np.empty(nnzC, dtype=np.int32)
    csrValC = np.empty(nnzC, dtype=dt)
    assert bh.get_C(csrColIndC, csrValC) == BHSPARSE_SUCCESS
    assert np.array_equal(bh.get_row_products(), g["products"])
    assert bh.free_mem() == BHSPARSE_SUCCESS
    assert bh.freePlatform() == BHSPARSE_SUCCESS
    assert_csr_equal((csrRowPtrC, csrColIndC, csrValC), (g["rowptrC"], g["colC"], g["valC"].astype(dt)), what="kat")


def test_cage4_squared(golden):
    g = golden("cage4_sq")
    m = int(g["m"])
    A = CSR(m, m, g["rowptrA"], g["colA"], g["valA"])
    got = spgemm(A, A)
    assert_csr_equal(got, (g["rowptrC"], g["colC"], g["valC"]), exact_values=False, rtol=1e-12, what="cage4")


@pytest.mark.parametrize("name,args,P,nnzC", [
    ("poisson5pt", (256, 256), 1629192, 846852),         # -spgemm 1
    ("poisson9pt", (256, 256), 5262436, 1623076),        # -spgemm 2
    ("poisson7pt", (51, 51, 51), 6298245, 3207645),      # -spgemm 3
    ("poisson27pt", (51, 51, 51), 90518849, 15438249),   # -spgemm 4
])
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_stock_workloads(name, args, P, nnzC, dt):
    A = getattr(gen, name)(*args, dtype=dt)
    st = _check(A, A, f"{name}{args} {dt.__name__}")
    assert st["products"] == P and st["nnzC"] == nnzC


# ---- every bin boundary ----------------------------------------------------------
def _identity(n, dt):
    return CSR(n, n, np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32), gen.int_values(n, 5, dt))


P_EDGES = [0, 1, 2, 3, 31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128, 129, 191, 192, 193, 255, 256, 257, 383, 384, 385,
           511, 512, 513, 767, 768, 769, 1023, 1024, 1025, 1535, 1536, 1537, 2047, 2048, 2049, 3071, 3072, 3073,
           4095, 4096, 4097, 6143, 6144, 6145, 8191, 8192, 8193, 12287, 12288, 12289, 24575, 24576, 24577, 40000]


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_bin_boundaries_no_duplicates(dt):
    """B = scaled identity: nnz(C_i) = products(i) = nnz(A_i), so one matrix walks
    both the symbolic (by upper bound) and numeric (by nnz(C_i)) bin edges."""
    n = 300000          # wider than the largest shared-memory bitmap, so the long rows stay on the hash path
    sizes = np.array(P_EDGES * 2, dtype=np.int64)
    A = gen.random_csr(sizes.size, n, sizes, seed=7, dtype=dt)
    st = _check(A, _identity(n, dt), f"bin edges identity {dt.__name__}")
    assert st["sym_bin_rows"][12] > 0 and st["num_bin_rows"][12] > 0      # the large bins ran


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("brow,ncols", [(5, 3000), (27, 2000), (64, 30000)])
def test_bin_boundaries_with_duplicates(dt, brow, ncols):
    """B rows of `brow` entries over few columns: heavy duplicate merging,
    nnz(C_i) well below the upper bound, so symbolic and numeric bins differ."""
    k = 4000
    sizes = np.array([0, 1, 2, 3, 6, 7, 12, 13, 19, 20, 38, 39, 60, 77, 120, 150, 240, 300, 480, 600, 900, 1200, 2000,
                      3000, 3999] * 2, dtype=np.int64)
    A = gen.random_csr(sizes.size, k, sizes, seed=11, dtype=dt)
    B = gen.random_csr(k, ncols, brow, seed=12, value_seed=13, dtype=dt)
    _check(A, B, f"dup edges brow={brow} {dt.__name__}")


def test_short_b_rows_select_narrow_groups():
    """average referenced B row <= 10 -> 8-lane groups (config 4's shape, scaled down)."""
    A = gen.uniform_rect(20000, 3000, per_row=8, seed=1, dtype=np.float32)
    B = gen.uniform_rect(3000, 20000, per_row=8, seed=2, value_seed=3, dtype=np.float32)
    st = _check(A, B, "uniform rect 8/row f32")
    assert st["products"] == 20000 * 64
    A2 = gen.random_csr(3000, 2500, (np.arange(3000) * 13) % 400, seed=5, dtype=np.float64)
    B2 = gen.random_csr(2500, 6000, (np.arange(2500) * 7) % 9, seed=6, value_seed=8, dtype=np.float64)
    _check(A2, B2, "short B rows, long A rows f64")


def test_many_empty_b_rows_in_a_small_row():
    """A row with > 32 entries whose products still fit one warp (ESC chunk loop)."""
    k, n = 500, 400
    lens = np.zeros(k, dtype=np.int64)
    lens[::40] = 2
    B = gen.random_csr(k, n, lens, seed=3)
    A = gen.random_csr(64, k, 300, seed=4)
    _check(A, B, "sparse B rows")


# ---- narrow column span: the shared-memory bitmap ("range") kernels ------------------
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_range_kernels_large_span(dt, monkeypatch):
    """27-point rows on a 128x128 plane span 66 053 columns -> RANGE_L bins (config 2's rows).
    These bins are off by default (measured slower than the hash kernels at that span,
    DESIGN.md); BHB200_RANGE=all switches them on."""
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("asserts on the general path's kernels; the pattern mode has its own tests")
    monkeypatch.setenv("BHB200_RANGE", "all")
    A = gen.poisson27pt(128, 128, 6, dtype=dt)
    st = _check(A, A, f"27pt 128x128x6 {dt.__name__}")
    assert st["sym_bin_rows"][14] > 0 and st["num_bin_rows"][15] > 0      # SB_RANGE_L / NB_RANGE_L128


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_range_kernels_irregular_band(dt, monkeypatch):
    """Irregular banded operands: B rows longer than a warp (tail loop), nnz(C_i) on both
    sides of the 128 / 512 accumulator limits, rows that leave the range path for the hash
    kernels after a range symbolic pass."""
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("asserts on the general path's kernels; the pattern mode has its own tests")
    monkeypatch.setenv("BHB200_RANGE", "all")
    for n, hb, k, what in ((3000, 300, 40, "span<12K c~500"), (6000, 3000, 70, "span~12K c>512"),
                           (20000, 9000, 9, "large span c<=128"), (20000, 9000, 12, "large span c<=512"),
                           (20000, 9000, 45, "large span c>512")):
        A = gen.banded_random(n, hb, k, seed=21, dtype=dt)
        B = gen.banded_random(n, hb, k + 3, seed=22, value_seed=23, dtype=dt)
        _check(A, B, f"banded {what} {dt.__name__}")


def test_range_kernels_pool_overflow_fallback(monkeypatch):
    """Word-list pool too small: the numeric range kernel must mark those rows itself."""
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("asserts on the general path's kernels; the pattern mode has its own tests")
    monkeypatch.setenv("BHB200_RANGE", "all")
    monkeypatch.setenv("BHB200_DEBUG_WORDLIST_CAP", "1000")
    A = gen.poisson27pt(40, 40, 8)
    _check(A, A, "27pt, pool of 1000 entries")
    B = gen.banded_random(4000, 2500, 30, seed=5)
    _check(B, B, "banded, pool of 1000 entries")
    monkeypatch.setenv("BHB200_DEBUG_WORDLIST_CAP", "0")
    _check(A, A, "27pt, no pool")


# ---- direct (single-pass) mode: sampled capacity, staging buffer, overflow retry --------------
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_direct_mode_speculation_holds(dt, monkeypatch):
    """27-point rows: 729 products -> at most 125 outputs; the sampled bound holds for every
    row, no symbolic pass runs for them and nothing is retried."""
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("asserts on the general path's kernels; the pattern mode has its own tests")
    monkeypatch.setenv("BHB200_RANGE", "off")      # (narrow-span rows would take the bitmap kernels instead)
    A = gen.poisson27pt(40, 40, 40, dtype=dt)
    st = _check(A, A, f"27pt 40^3 direct {dt.__name__}")
    assert st["direct_rows"] > 0.9 * A.rows and st["direct_retry_rows"] == 0
    assert st["num_bin_rows"][17] == st["direct_rows"]          # all of them came back through the Ct -> C copy


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("cap", ["32", "64", "128"])
def test_direct_mode_overflow_is_retried(dt, cap, monkeypatch):
    """Force a speculated capacity that is too small for most rows: every row that does not
    fit must be detected and redone by the two-pass path, bit for bit."""
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("asserts on the general path's kernels; the pattern mode has its own tests")
    monkeypatch.setenv("BHB200_DEBUG_FORCE_CAP", cap)
    monkeypatch.setenv("BHB200_RANGE", "off")
    A = gen.poisson27pt(24, 24, 24, dtype=dt)
    st = _check(A, A, f"27pt forced cap {cap} {dt.__name__}")
    assert st["direct_rows"] > 0
    if int(cap) < 125:
        assert st["direct_retry_rows"] > 0
    # irregular rows: outputs per row from a handful to several hundred inside one symbolic bin
    R = gen.random_csr(6000, 3000, 20 + (np.arange(6000) * 7) % 40, seed=31, dtype=dt)
    S = gen.random_csr(3000, 2500, 12, seed=32, value_seed=33, dtype=dt)
    st = _check(R, S, f"random forced cap {cap} {dt.__name__}")
    assert st["direct_retry_rows"] > 0


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_direct_mode_wide_bins(dt, monkeypatch):
    """Rows that barely compress (wide random column space): the sampled mean nnz(C_i) is close
    to the product bound, so the bins up to 6144 products run single-pass with the capacity the
    bound dictates (group kernel for 256, CTA kernels for 512..8192) and skip the symbolic pass."""
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("asserts on the general path's kernels; the pattern mode has its own tests")
    per_row = np.array([12, 24, 48, 96, 150, 250, 400])[np.arange(7 * 4500) % 7]
    A = gen.random_csr(7 * 4500, 20000, per_row, seed=41, dtype=dt)
    B = gen.random_csr(20000, 3_000_000, 12, seed=42, value_seed=43, dtype=dt)
    st = _check(A, B, f"wide direct {dt.__name__}")
    mask = st["direct_bin_mask"]
    assert all((mask >> b) & 1 for b in range(4, 10)), bin(mask)      # SB_G256 .. SB_B8192
    assert st["direct_retry_rows"] == 0 and st["direct_rows"] >= 6 * 4500
    assert st["num_bin_rows"][17] == st["direct_rows"]
    monkeypatch.setenv("BHB200_DIRECT", "tight")
    st = _check(A, B, f"wide direct disabled {dt.__name__}")
    assert all(not ((st["direct_bin_mask"] >> b) & 1) for b in range(4, 10))


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_wide_rows_bucket_sort_edges(dt):
    """k_num_bucket3 (csrc/stage_bucket.cuh) beyond uniform rows: (a) rows of A with more entries than one
    staging chunk and B rows longer than the whole-CTA threshold (512), (b) a hub column present in every B
    row -- hundreds of equal columns in ONE bucket of every output row (the warp-cooperative ranking and the
    run-summing emit)."""
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("general path only")
    rows = 5 * 4200
    # (a) many short B rows per A row + a few very long B rows referenced by every fifth A row
    k, n = 30000, 2_500_000
    b_len = np.full(k, 3)
    b_len[:40] = np.array([600, 900, 1500, 2500])[np.arange(40) % 4]
    B = gen.random_csr(k, n, b_len, seed=52, value_seed=53, dtype=dt)
    per_row = np.array([150, 300, 700, 40, 1100])[np.arange(rows) % 5]
    A = gen.random_csr(rows, k - 40, per_row, seed=51, dtype=dt)
    # shift A's columns past the long rows, then give every fifth row one of them (rows stay sorted: 0..39 < 40)
    colA = A.col + 40
    first = A.rowptr[:-1][::5]
    colA[first] = np.arange(first.size) % 40
    A = CSR(rows, k, A.rowptr, colA.astype(np.int32), A.val)
    st = _check(A, B, f"bucket chunks + long B rows {dt.__name__}")
    assert st["direct_rows"] >= 4 * 4200
    # (b) hub column: every B row holds column 7 and eleven random ones
    k = 20000
    rng = np.random.default_rng(6)
    others = 8 + np.sort(rng.choice((n - 8) // 11, size=(k, 11)), axis=1) * 11 + np.arange(11)
    cols = np.concatenate([np.full((k, 1), 7), others], axis=1)
    B = CSR(k, n, (np.arange(k + 1) * 12).astype(np.int32), cols.reshape(-1).astype(np.int32), gen.int_values(12 * k, 9, dt))
    per_row = np.array([50, 90, 180, 330, 600])[np.arange(rows) % 5]
    A = gen.random_csr(rows, k, per_row, seed=54, dtype=dt)
    st = _check(A, B, f"bucket hub column {dt.__name__}")
    assert st["direct_rows"] >= 4 * 4200


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_small_rows_warp_bucket_sort(dt, monkeypatch):
    """k_num_bucket3w (csrc/stage_bucket.cuh): bins of at most 96 / 192 products whose rows barely compress --
    BASELINE config 4 in small (8 x 8 products per row, 8 lanes per B row), longer B rows (32 lanes per B row),
    a tight bin with a few rows beyond the speculated capacity (retry queue), and the hash kernels as a cross-check."""
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("general path only")
    A = gen.uniform_rect(16384, 4096, 8, seed=1, dtype=dt)
    B = gen.uniform_rect(4096, 300000, 8, seed=2, value_seed=3, dtype=dt)
    st0 = _check(A, B, f"warp bucket 8x8 {dt.__name__}")
    assert st0["direct_rows"] == 16384 and st0["direct_retry_rows"] == 0
    # B rows of 20 entries: 4 x 20 = 80 products (SB_G128) and 8 x 20 = 160 (SB_G256), 32 lanes per B row
    per_row = np.array([4, 8])[np.arange(2 * 5000) % 2]
    A2 = gen.random_csr(2 * 5000, 6000, per_row, seed=61, dtype=dt)
    B2 = gen.random_csr(6000, 2_000_000, 20, seed=62, value_seed=63, dtype=dt)
    st = _check(A2, B2, f"warp bucket 20-entry B rows {dt.__name__}")
    assert st["direct_rows"] == 2 * 5000
    # tight bin: most rows 8 x 8 = 64 outputs, one row in 300 has 11 x 8 = 88 (same bin, beyond a capacity of 64
    # unless the sample happened to see one)
    per_row = np.where(np.arange(12000) % 300 == 7, 11, 8)
    A3 = gen.random_csr(12000, 4096, per_row, seed=64, dtype=dt)
    st = _check(A3, B, f"warp bucket tight overflow {dt.__name__}")
    assert st["direct_rows"] == 12000
    monkeypatch.setenv("BHB200_BUCKET_W", "off")
    st = _check(A, B, f"hash kernels 8x8 {dt.__name__}")
    assert st["direct_rows"] == 16384
    # the hash kernels need no column CDF: k_colcount, k_cdf_hist and k_cdf_scan are not launched
    assert st["kernel_launches"] == st0["kernel_launches"] - 3


def test_direct_mode_off_matches(monkeypatch):
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("asserts on the general path's kernels; the pattern mode has its own tests")
    monkeypatch.setenv("BHB200_DIRECT", "off")
    monkeypatch.setenv("BHB200_RANGE", "off")
    A = gen.poisson27pt(30, 30, 30)
    st = _check(A, A, "27pt direct off")
    assert st["direct_rows"] == 0


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_rmat_skewed(dt):
    """Graph500-style skew: long rows -> block-hash and global-bitmap bins."""
    A = gen.rmat(13, 16, a=0.57, b=0.19, c=0.19, d=0.05, seed=3, dtype=dt)
    st = _check(A, A, f"rmat13 g500 {dt.__name__}")
    assert sum(st["num_bin_rows"][9:13]) > 0
    A = gen.rmat(14, 8, seed=4, dtype=dt)
    _check(A, A, f"rmat14 mild {dt.__name__}")


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_real_values_within_tolerance(dt):
    A = gen.poisson27pt(20, 20, 20, dtype=dt, values="real")
    _check(A, A, "27pt real", exact=False)
    A = gen.rmat(12, 16, a=0.57, b=0.19, c=0.19, d=0.05, seed=9, dtype=dt, values="real")
    _check(A, A, "rmat real", exact=False)


def test_explicit_zero_is_kept():
    A = CSR(1, 2, np.array([0, 2], np.int32), np.array([0, 1], np.int32), np.array([1.0, -1.0]))
    B = CSR(2, 1, np.array([0, 1, 2], np.int32), np.array([0, 0], np.int32), np.array([1.0, 1.0]))
    rp, c, v = spgemm(A, B)
    assert rp.tolist() == [0, 1] and c.tolist() == [0] and v.tolist() == [0.0]


def test_empty_cases():
    A = gen.random_csr(7, 5, [0, 2, 0, 1, 0, 0, 3], seed=1)
    B = gen.random_csr(5, 9, 0, seed=2)
    rp, c, v = spgemm(A, B)
    assert rp.tolist() == [0] * 8 and c.size == 0
    Z = gen.random_csr(6, 5, 0, seed=1)
    B = gen.random_csr(5, 9, 3, seed=2)
    rp, c, v = spgemm(Z, B)
    assert rp.tolist() == [0] * 7 and c.size == 0
    E = CSR(0, 5, np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0))
    rp, c, v = spgemm(E, B)
    assert rp.tolist() == [0] and c.size == 0


def test_wide_column_space():
    """n > 2^26 switches the small-row kernel to 64-bit sort keys."""
    n = (1 << 27) + 11
    k = 64
    rng = np.random.default_rng(5)
    cols = np.sort(rng.integers(0, n - 3, size=(k, 3)), axis=1) + np.arange(3)[None, :]   # strictly ascending
    cols[0] = [0, (1 << 27) - 1, n - 1]
    cols = cols.astype(np.int32)
    B = CSR(k, n, (np.arange(k + 1) * 3).astype(np.int32), cols.reshape(-1), gen.int_values(3 * k, 1))
    A = gen.random_csr(200, k, (np.arange(200) % 11), seed=2)
    _check(A, B, "wide columns")
    # mid-size rows over the same wide column space: direct mode without the packed (column, index) sort
    A2 = gen.random_csr(5000, k, 12 + (np.arange(5000) % 20), seed=6)
    st = _check(A2, B, "wide columns, hash bins")
    assert st["direct_rows"] > 0


def test_repeated_calls_and_reinit():
    """spgemm() twice on one initData (undefined in the reference, counters are
    never reset: bhsparse.h:379-380) and re-initialisation on one context."""
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("asserts on the general path's kernels; the pattern mode has its own tests")
    platforms = [False] * NUM_PLATFORMS
    platforms[BHSPARSE_CUDA] = True
    bh = bhsparse()
    assert bh.initPlatform(platforms) == 0
    for dt, A in ((np.float64, gen.poisson9pt(64, 64)), (np.float32, gen.rmat(10, 8, dtype=np.float32))):
        rowptrC = np.zeros(A.rows + 1, np.int32)
        assert bh.initData(A.rows, A.cols, A.cols, A.nnz, A.val, A.rowptr, A.col,
                           A.nnz, A.val, A.rowptr, A.col, rowptrC) == 0
        want = _oracle(A, A)
        for _ in range(3):
            assert bh.warmup() == 0
            assert bh.spgemm() == 0
            colC = np.empty(bh.get_nnzC(), np.int32)
            valC = np.empty(bh.get_nnzC(), dt)
            assert bh.get_C(colC, valC) == 0
            assert_csr_equal((rowptrC, colC, valC), want, what="repeat")
            assert np.array_equal(bh.get_rowptrC_i64(), want[0])
    assert bh.free_mem() == 0 and bh.freePlatform() == 0


def test_error_paths():
    bh = bhsparse()
    assert bh.spgemm() != 0                              # before initPlatform
    assert bh.initPlatform([False] * NUM_PLATFORMS) != 0   # no CUDA platform selected
    platforms = [False] * NUM_PLATFORMS
    platforms[BHSPARSE_CUDA] = True
    assert bh.initPlatform(platforms) == 0
    assert bh.spgemm() == capi.ERR_INVALID                # before initData
    assert bh.get_nnzC() == -1
    A = gen.poisson5pt(8, 8)
    bad = A.rowptr.copy()
    bad[-1] += 1
    assert bh.initData(A.rows, A.cols, A.cols, A.nnz, A.val, bad, A.col, A.nnz, A.val, A.rowptr, A.col,
                       np.zeros(A.rows + 1, np.int32)) == capi.ERR_INVALID
    assert "rowptrA" in bh.last_error()
    assert bh.freePlatform() == 0


def test_operand_preconditions_are_checked():
    """Rows of B must be sorted, duplicate-free and inside [0, n); columns of A inside [0, k)
    (include/bhsparse_b200.h).  The reference silently assumes it (bhsparse_cuda.h:1730,1762);
    here a violation is an error code, never corrupted memory or lost contributions."""
    platforms = [False] * NUM_PLATFORMS
    platforms[BHSPARSE_CUDA] = True
    A = gen.random_csr(300, 200, 9, seed=3)
    B = gen.random_csr(200, 400, 12, seed=4, value_seed=5)

    def run(A, B):
        bh = bhsparse()
        assert bh.initPlatform(platforms) == 0
        err = bh.initData(A.rows, A.cols, B.cols, A.nnz, A.val, A.rowptr, A.col, B.nnz, B.val, B.rowptr, B.col,
                          np.zeros(A.rows + 1, np.int32))
        if err == 0:
            err = bh.spgemm()
        msg = bh.last_error()
        bh.freePlatform()
        return err, msg

    assert run(A, B)[0] == 0
    c = B.col.copy()
    s = B.rowptr[57]
    c[s], c[s + 1] = c[s + 1], c[s]                       # one unsorted pair
    err, msg = run(A, CSR(B.rows, B.cols, B.rowptr, c, B.val))
    assert err == capi.ERR_INVALID and "sorted" in msg
    c = B.col.copy()
    c[B.rowptr[120] + 3] = c[B.rowptr[120] + 2]           # a duplicate column
    assert run(A, CSR(B.rows, B.cols, B.rowptr, c, B.val))[0] == capi.ERR_INVALID
    c = B.col.copy()
    c[B.rowptr[199 + 1] - 1] = B.cols                     # column == n
    assert run(A, CSR(B.rows, B.cols, B.rowptr, c, B.val))[0] == capi.ERR_INVALID
    ca = A.col.copy()
    ca[A.rowptr[10]] = -1                                 # column of A outside [0, k)
    err, msg = run(CSR(A.rows, A.cols, A.rowptr, ca, A.val), B)
    assert err == capi.ERR_INVALID and "A" in msg


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_host_memory_spill(dt, monkeypatch):
    """SURVEY.md 8f-4 (the reference's OpenCL `-opencl-hcmp` mode, bhsparse_opencl.cpp:219-227,
    832-863): when the device cannot hold C or the staging buffer they live in pinned, device-mapped
    host memory.  Forced here by a debug cap on the size of a single device buffer."""
    monkeypatch.setenv("BHB200_DEBUG_DEVICE_CAP", "65536")
    A = gen.poisson27pt(16, 16, 16, dtype=dt)              # pattern mode or direct mode + staging
    rp, col, val, st = spgemm(A, A, return_stats=True)
    assert st["spill_bytes"] >= (4 + A.val.itemsize) * st["nnzC"]
    assert_csr_equal((rp, col, val), _oracle(A, A), what="spill stencil")
    R = gen.rmat(12, 16, a=0.57, b=0.19, c=0.19, d=0.05, dtype=dt)     # hash / CTA / global-bitmap bins
    rp, col, val, st = spgemm(R, R, return_stats=True)
    assert st["spill_bytes"] > 0
    assert_csr_equal((rp, col, val), _oracle(R, R), what="spill rmat")
    # rows beyond the on-chip tables: global bitmap-rank kernel, red.global.add into the spilled C
    L = gen.random_csr(6, 120000, np.array([40000, 3, 9000, 0, 20000, 17]), seed=9, dtype=dt)
    rp, col, val, st = spgemm(L, _identity(120000, dt), return_stats=True)
    assert st["spill_bytes"] > 0 and st["num_bin_rows"][12] > 0
    assert_csr_equal((rp, col, val), _oracle(L, _identity(120000, dt)), what="spill large rows")


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_heavy_rows_sliced_bucket_sort(dt, monkeypatch):
    """Rows with more products than the on-chip tables hold (k_num_bucket_heavy): forced here, since small
    matrices never pass the sampling that selects it.  Cases: rows that do not compress at all, rows with
    heavy duplication, a row just over the smallest heavy bin, and the pathological one -- tens of thousands
    of products in ONE column, which no slicing of the column axis can split (reduced column by column)."""
    if os.environ.get("BHB200_PATTERN") != "off":
        pytest.skip("general path only")
    monkeypatch.setenv("BHB200_DEBUG_FORCE_HEAVY", "1")
    n = 400000
    # (a) no compression: B = identity, rows of A with 13000 .. 60000 distinct columns
    A = gen.random_csr(6, n, np.array([13000, 60000, 5, 24577, 0, 30000]), seed=21, dtype=dt)
    st = _check(A, _identity(n, dt), f"heavy identity {dt.__name__}")
    assert st["direct_rows"] >= 4
    # (b) duplicates: B rows of 40 entries over 3000 columns -> every output column hit ~50 times
    k = 5000
    A = gen.random_csr(4, k, np.array([4000, 1500, 700, 2]), seed=22, dtype=dt)
    B = gen.random_csr(k, 3000, 40, seed=23, value_seed=24, dtype=dt)
    _check(A, B, f"heavy duplicates {dt.__name__}")
    # (c) one column carries 30000 products: every B row holds column 7 (+ three random ones)
    k = 30000
    rng = np.random.default_rng(5)
    others = 8 + np.sort(rng.integers(0, (n - 8) // 3, size=(k, 3)), axis=1) * 3 + np.arange(3)     # three distinct columns > 7
    cols = np.concatenate([np.full((k, 1), 7), others], axis=1)
    B = CSR(k, n, (np.arange(k + 1) * 4).astype(np.int32), cols.reshape(-1).astype(np.int32), gen.int_values(4 * k, 9, dt))
    A = gen.random_csr(3, k, np.array([k, 20000, 9]), seed=25, dtype=dt)
    _check(A, B, f"heavy single column {dt.__name__}")
