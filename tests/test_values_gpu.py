"""Values of every numeric kernel family against the quad-precision reference (tests/exact_ref.c) under the
library's value contract (DESIGN.md §2, include/bhsparse_b200.h):
  - finite inputs: |c_hat - c| <= gamma(p)*s + 2*p*lam for every entry (exact_ref.bound);
  - integers inside the bit budget of exact_ref.tier1_bits: equal values (the sign of a zero is not compared);
  - non-finite entries: NaN / +inf / -inf exactly as the products in the value type dictate.

Each row of CASES builds operands whose product one kernel family computes, sets the switches that send it
there, and proves from the statistics that the family ran, so that a later change of a heuristic cannot move the
case to another kernel unnoticed.  Every row runs in f64 and f32:
  1. tier 1, exact signed integers (products above 2^24 in f64, so rounding through f32 shows);
  2. tier 2, signed full-significand values, then update_values with fresh tier-2 values and spgemm_numeric on
     the same context;
  3. tier 2 on the cancelling operands of exact_ref.paired (|c| far below s), where the family keeps them;
  4. tier 3, tier-2 values with +-inf, NaN, stored zeros and subnormal products.
The structure of C is compared bit for bit with the reference's in every run, and the statistics proof holds after
spgemm_numeric too: there the rows of direct-mode cases are re-binned into the two-pass numeric bins, which the
proof of those cases checks instead.

Most cases hold about 2M products or fewer.  The direct-mode cases are larger because the direct mode samples only
symbolic bins of at least 4096 rows, so each bin they need takes 4096 rows or more: bucket3_wide (six bins, about
19M products), bucket3_chunks_long_b (about 29M) and bucket3_hub_column (about 11M)."""
from dataclasses import dataclass, field
from typing import Callable

import numpy as np
import pytest

import exact_ref as xr
from benchmark_spgemm_using_csr_b200 import capi, generators as gen
from benchmark_spgemm_using_csr_b200.generators import CSR
from csr_ref import keys, stored
from test_mask_gpu import BIN_ROWS, _bin_operands

pytestmark = pytest.mark.gpu

N, T = capi.OP_N, capi.OP_T


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    lib = xr.compile_lib(tmp_path_factory.mktemp("exact_ref"))
    assert lib is not None, "gcc is needed to build the quad-precision reference"
    return lib


# ---- comparison ------------------------------------------------------------------------------------------
CLASS_NAMES = {xr.FINITE: "finite", xr.NAN: "NaN", xr.PINF: "+inf", xr.NINF: "-inf"}


def restrict(ref, n, rpM, colM):
    """The exact product restricted to the pattern of M (what a masked product computes)."""
    rows = xr.row_index(ref["rowptr"])
    keep = np.isin(rows * n + ref["col"].astype(np.int64), keys(rpM, colM, n))
    out = {k: v[keep] for k, v in ref.items() if isinstance(v, np.ndarray) and k != "rowptr"}
    rowptr = np.zeros(ref["rowptr"].size, dtype=np.int64)
    np.cumsum(np.bincount(rows[keep], minlength=rowptr.size - 1), out=rowptr[1:])
    return dict(out, rowptr=rowptr, dtype=ref["dtype"])


def check_values(got, ref, what, exact=False):
    """got = (rowptr, col, val) from the library; ref from exact_ref.product.  Structure bit for bit; values equal
    (exact) or within the bound; non-finite classes exactly.  A failure names the row, column, p, s, bound and
    error of the first few offending entries."""
    rp, col, val = got
    assert np.array_equal(np.asarray(rp, dtype=np.int64), ref["rowptr"]), (
        f"{what}: rowptrC differs from the exact product, first at row "
        f"{int(np.flatnonzero(np.asarray(rp, dtype=np.int64) != ref['rowptr'])[0]) - 1}")
    if not np.array_equal(col, ref["col"]):
        t = int(np.flatnonzero(col != ref["col"])[0])
        raise AssertionError(f"{what}: colC differs at row {int(xr.row_index(ref['rowptr'])[t])} entry {t}: "
                             f"{col[t]} vs {ref['col'][t]}")
    dt = ref["dtype"]
    v = val.astype(np.float64)
    cls, hi, lo, s, p = ref["cls"], ref["hi"], ref["lo"], ref["s"], ref["p"]
    fin = cls == xr.FINITE
    bad = ((cls == xr.NAN) & ~np.isnan(v)) | ((cls == xr.PINF) & (v != np.inf)) | ((cls == xr.NINF) & (v != -np.inf))
    bad |= fin & ~np.isfinite(v)
    with np.errstate(invalid="ignore"):
        err = np.abs((v - hi) - lo)
    bnd = xr.bound(p, s, dt)
    if exact:
        assert not lo[fin].any(), f"{what}: tier-1 values outside the exact regime"
        bad |= fin & (v != hi)
    else:
        # 2^-20 of slack covers the reference's own rounding (sums to 113 bits, s rounded to f64)
        bad |= fin & ~(err <= bnd * (1 + 2.0 ** -20))
    if bad.any():
        rows = xr.row_index(ref["rowptr"])
        idx = np.flatnonzero(bad)
        lines = [f"row {rows[t]} col {col[t]}: p={p[t]} s={s[t]:.6g} bound={bnd[t]:.6g} err={err[t]:.6g} "
                 f"got={val[t]!r} want={'%.17g' % (hi[t] + lo[t]) if fin[t] else CLASS_NAMES[int(cls[t])]}"
                 for t in idx[:6]]
        raise AssertionError(f"{what}: {idx.size} of {val.size} entries break the value contract "
                             f"({'equal values' if exact else 'bound'}):\n  " + "\n  ".join(lines))


# ---- the case table ----------------------------------------------------------------------------------------
@dataclass
class Case:
    name: str
    build: Callable                       # dt -> (op(A), op(B)) as CSR: the effective operands
    proof: Callable                       # stats -> bool: the family ran
    env: dict = field(default_factory=dict)
    ops: tuple = (N, N)
    cancel: bool = True                   # the cancelling operands stay in the family
    mask: Callable = None                 # (op(A), op(B)) -> (rowptrM, colM)
    direct: bool = False                  # direct-mode rows: spgemm_numeric re-bins them (REBINNED)
    twin_of: dict = None                  # switches of a configuration that launches 3 kernels more than this one


GENERAL = {"BHB200_PATTERN": "off"}
NB = lambda st, lo, hi: all(st["num_bin_rows"][b] > 0 for b in range(lo, hi + 1))


def REBINNED(st):
    """spgemm_numeric after a direct-mode product: every row in a two-pass numeric bin, none in the copy bin."""
    return st["direct_rows"] == 0 and st["num_bin_rows"][17] == 0 and sum(st["num_bin_rows"][:17]) == st["m"]


def _vstack(X: CSR, Y: CSR) -> CSR:
    return CSR(X.rows + Y.rows, max(X.cols, Y.cols), np.concatenate([X.rowptr, X.rowptr[-1] + Y.rowptr[1:]]).astype(np.int32),
               np.concatenate([X.col, Y.col]).astype(np.int32), np.concatenate([X.val, Y.val]))


def _single_esc(dt):
    """5-point rows (25 products: ESC) and rows of exactly one product (the single-product kernel)."""
    P = gen.poisson5pt(100, 100, dtype=dt)
    k = P.cols + 1000
    brp = np.concatenate([P.rowptr, P.rowptr[-1] + 1 + np.arange(1000)]).astype(np.int32)
    bcol = np.concatenate([P.col, (np.arange(1000) * 7) % P.cols]).astype(np.int32)
    B = CSR(k, P.cols, brp, bcol, np.ones(bcol.size, dt))
    arp = np.concatenate([P.rowptr, P.rowptr[-1] + 1 + np.arange(2000)]).astype(np.int32)
    acol = np.concatenate([P.col, P.cols + np.arange(2000) % 1000]).astype(np.int32)
    return CSR(P.rows + 2000, k, arp, acol, np.ones(acol.size, dt)), B


def _hash_two_pass(dt):
    """Rows of 50 .. 1500 products that barely compress (numeric bins 4 .. 9: the group hash kernels and the first
    CTA hash bin), and 500 rows of 50 products that compress to at most 30 columns (bin 3)."""
    per_row = np.array([5, 10, 20, 40, 80, 150])[np.arange(3000) % 6]
    A = gen.random_csr(3000, 5000, per_row, seed=71, dtype=dt)
    cols = np.sort(5000 + (np.arange(500)[:, None] * 7 + np.arange(5) * 100) % 500, axis=1)
    A = _vstack(A, CSR(500, 5500, (np.arange(501) * 5).astype(np.int32), cols.reshape(-1).astype(np.int32), np.ones(2500, dt)))
    B = _vstack(gen.random_csr(5000, 200000, 10, seed=72, dtype=dt), gen.random_csr(500, 30, 10, seed=73, dtype=dt))
    return A, B


def _irregular(dt):
    return (gen.random_csr(4000, 3000, 20 + (np.arange(4000) * 7) % 40, seed=31, dtype=dt),
            gen.random_csr(3000, 2500, 12, seed=32, dtype=dt))


def _wide(dt):
    """Rows that barely compress: 4100 in each of SB_G256 .. SB_G4096 (each sampled: direct wide mode) and a few
    in SB_B8192, which follows the bin below it."""
    per_row = np.repeat([12, 24, 48, 96, 180, 350], [4100] * 5 + [400])
    return (gen.random_csr(per_row.size, 20000, per_row, seed=41, dtype=dt),
            gen.random_csr(20000, 3_000_000, 12, seed=42, dtype=dt))


def _bucket_chunks(dt):
    """k_num_bucket3: A rows with more entries than one staging chunk, and B rows longer than the whole-CTA
    threshold (512) referenced by every fifth A row."""
    rows, k, n = 5 * 4200, 30000, 2_500_000
    b_len = np.full(k, 3)
    b_len[:40] = np.array([600, 900, 1500, 2500])[np.arange(40) % 4]
    B = gen.random_csr(k, n, b_len, seed=52, dtype=dt)
    A = gen.random_csr(rows, k - 40, np.array([150, 300, 700, 40, 1100])[np.arange(rows) % 5], seed=51, dtype=dt)
    colA = A.col + 40
    first = A.rowptr[:-1][::5]
    colA[first] = np.arange(first.size) % 40
    return CSR(rows, k, A.rowptr, colA.astype(np.int32), A.val), B


def _hub_rows(k, n, others, seed):
    """k rows of B holding column 7 and `others` distinct random columns above it."""
    rng = np.random.default_rng(seed)
    oth = 8 + np.sort(rng.choice((n - 8) // others, size=(k, others)), axis=1) * others + np.arange(others)
    cols = np.concatenate([np.full((k, 1), 7), oth], axis=1)
    return CSR(k, n, (np.arange(k + 1) * (others + 1)).astype(np.int32), cols.reshape(-1).astype(np.int32),
               np.ones(k * (others + 1)))


def _bucket_hub(dt):
    """k_num_bucket3: a hub column present in every B row, hundreds of equal columns in one bucket."""
    B = _hub_rows(20000, 2_500_000, 7, seed=6).astype(dt)
    per_row = np.repeat([50, 90, 180], 4200)
    return gen.random_csr(per_row.size, 20000, per_row, seed=54, dtype=dt), B


def _cta_hash(dt):
    """Compressing rows of about 3400 and 5800 outputs: the CTA hash kernels."""
    per_row = np.array([200, 400])[np.arange(300) % 2]
    return gen.random_csr(300, 3000, per_row, seed=81, dtype=dt), gen.random_csr(3000, 12000, 20, seed=82, dtype=dt)


def _global_bitmap(dt):
    """Rows of 80 000 products over 20 000 columns (about 4 per column): the global bitmap kernel."""
    return gen.random_csr(16, 3000, 2000, seed=83, dtype=dt), gen.random_csr(3000, 20000, 40, seed=84, dtype=dt)


def _heavy_duplicates(dt):
    """Rows of 28 000 .. 160 000 products on 3000 columns spread over 400 000: every output column hit about 50
    times."""
    B = gen.random_csr(5000, 3000, 40, seed=23, dtype=dt)
    return (gen.random_csr(4, 5000, np.array([4000, 1500, 700, 2]), seed=22, dtype=dt),
            CSR(B.rows, 400000, B.rowptr, (B.col * 133).astype(np.int32), B.val))


def _identity(n, dt):
    return CSR(n, n, np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32), np.ones(n, dt))


def _rect(dt):
    return (gen.random_csr(3000, 2000, 8 + np.arange(3000) % 33, seed=91, dtype=dt),
            gen.random_csr(2000, 2500, 6 + np.arange(2000) % 5, seed=92, dtype=dt))


def _mask_bins(dt):
    A, B, rpM, colM = _bin_operands([r for r, _ in BIN_ROWS], dt)
    return A, B


def _mask_of_bins(A, B):
    return _bin_operands([r for r, _ in BIN_ROWS], A.val.dtype)[2:]


MASK_BINS = list(np.bincount([b for _, b in BIN_ROWS], minlength=capi.NUM_MASK_BINS))


def _uniform_8x8(dt):
    return (gen.uniform_rect(16384, 4096, 8, seed=1, dtype=dt), gen.uniform_rect(4096, 300000, 8, seed=2, dtype=dt))


CASES = [
    Case("pattern_27pt", lambda dt: (gen.poisson27pt(12, 12, 12, dtype=dt),) * 2, lambda st: st["pattern_mode"] == 1,
         cancel=False),
    Case("pattern_7pt", lambda dt: (gen.poisson7pt(30, 30, 30, dtype=dt),) * 2, lambda st: st["pattern_mode"] == 1,
         cancel=False),
    Case("single_esc", _single_esc, lambda st: NB(st, 1, 2), GENERAL, cancel=False),
    Case("hash_two_pass", _hash_two_pass, lambda st: NB(st, 3, 9) and st["direct_rows"] == 0,
         dict(GENERAL, BHB200_DIRECT="off", BHB200_RANGE="off")),
    Case("direct_cap32_retry", _irregular, lambda st: st["direct_retry_rows"] > 0,
         dict(GENERAL, BHB200_DEBUG_FORCE_CAP="32", BHB200_RANGE="off"), direct=True),
    Case("direct_cap64_retry", _irregular, lambda st: st["direct_retry_rows"] > 0,
         dict(GENERAL, BHB200_DEBUG_FORCE_CAP="64", BHB200_RANGE="off"), direct=True),
    Case("bucket3_wide", _wide, lambda st: all((st["direct_bin_mask"] >> b) & 1 for b in range(4, 10)), GENERAL,
         cancel=False, direct=True),
    Case("bucket3w", _uniform_8x8, lambda st: st["direct_rows"] == 16384, GENERAL, cancel=False, direct=True),
    # the hash kernels need no column CDF: k_colcount, k_cdf_hist and k_cdf_scan are not launched
    Case("hash_twin_of_bucket3w", _uniform_8x8, lambda st: st["direct_rows"] == 16384,
         dict(GENERAL, BHB200_BUCKET_W="off"), cancel=False, direct=True, twin_of=GENERAL),
    Case("bucket3_chunks_long_b", _bucket_chunks, lambda st: st["direct_rows"] >= 4 * 4200, GENERAL, cancel=False,
         direct=True),
    Case("bucket3_hub_column", _bucket_hub, lambda st: st["direct_rows"] >= 2 * 4200, GENERAL, cancel=False,
         direct=True),
    # numeric bin 9 (the first CTA hash bin) is reached by hash_two_pass
    Case("cta_hash", _cta_hash, lambda st: NB(st, 10, 11), dict(GENERAL, BHB200_DIRECT="off", BHB200_RANGE="off")),
    Case("global_bitmap", _global_bitmap, lambda st: NB(st, 12, 12), dict(GENERAL, BHB200_RANGE="off")),
    Case("range_vec_pool1000", lambda dt: (gen.poisson27pt(24, 24, 8, dtype=dt),) * 2, lambda st: NB(st, 13, 13),
         dict(GENERAL, BHB200_RANGE="all", BHB200_DEBUG_WORDLIST_CAP="1000")),
    Case("range_no_pool", lambda dt: (gen.banded_random(4000, 300, 12, seed=5, dtype=dt),
                                      gen.banded_random(4000, 300, 15, seed=6, dtype=dt)),
         lambda st: NB(st, 14, 14), dict(GENERAL, BHB200_RANGE="all", BHB200_DEBUG_WORDLIST_CAP="0")),
    # column spans above 12 224: the large-span range kernels, vectorised for rows of at most 128 outputs
    Case("range_large_vec", lambda dt: (gen.banded_random(20000, 9000, 9, seed=21, dtype=dt),
                                        gen.banded_random(20000, 9000, 12, seed=22, dtype=dt)),
         lambda st: NB(st, 15, 15), dict(GENERAL, BHB200_RANGE="all")),
    Case("range_large", lambda dt: (gen.banded_random(20000, 9000, 12, seed=21, dtype=dt),
                                    gen.banded_random(20000, 9000, 15, seed=22, dtype=dt)),
         lambda st: NB(st, 16, 16), dict(GENERAL, BHB200_RANGE="all")),
    Case("heavy_identity", lambda dt: (gen.random_csr(6, 400000, np.array([13000, 60000, 5, 24577, 0, 30000]), seed=21,
                                                      dtype=dt), _identity(400000, dt)),
         lambda st: st["direct_rows"] >= 4, dict(GENERAL, BHB200_DEBUG_FORCE_HEAVY="1"), direct=True),
    Case("heavy_duplicates", _heavy_duplicates, lambda st: st["direct_rows"] >= 2,
         dict(GENERAL, BHB200_DEBUG_FORCE_HEAVY="1", BHB200_RANGE="off"), direct=True),
    Case("heavy_single_column", lambda dt: (gen.random_csr(3, 30000, np.array([30000, 20000, 9]), seed=25, dtype=dt),
                                            _hub_rows(30000, 400000, 3, seed=5).astype(dt)),
         lambda st: st["direct_rows"] >= 2, dict(GENERAL, BHB200_DEBUG_FORCE_HEAVY="1"), direct=True),
    Case("masked_bins", _mask_bins, lambda st: st["mask_bin_rows"] == MASK_BINS, cancel=False, mask=_mask_of_bins),
    Case("transpose_NT", _rect, lambda st: st["transposed_ops"] == 2, ops=(N, T)),
    Case("transpose_TN", _rect, lambda st: st["transposed_ops"] == 1, ops=(T, N)),
    Case("transpose_TT", _rect, lambda st: st["transposed_ops"] == 3, ops=(T, T)),
    Case("spill_rmat", lambda dt: (gen.rmat(11, 16, a=0.57, b=0.19, c=0.19, d=0.05, seed=3, dtype=dt),) * 2,
         lambda st: st["spill_bytes"] > 0, dict(BHB200_DEBUG_DEVICE_CAP="65536")),
    Case("spill_global_bitmap", _global_bitmap, lambda st: st["spill_bytes"] > 0 and NB(st, 12, 12),
         dict(GENERAL, BHB200_RANGE="off", BHB200_DEBUG_DEVICE_CAP="65536")),
]


def with_values(X: CSR, v) -> CSR:
    return CSR(X.rows, X.cols, X.rowptr, X.col, np.asarray(v).astype(X.val.dtype))


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_values(lib, case, dt, monkeypatch):
    for k, v in case.env.items():
        monkeypatch.setenv(k, v)
    A, B = case.build(dt)
    A, B = A.astype(dt), B.astype(dt)
    mask = case.mask(A, B) if case.mask else None
    opA, opB = case.ops

    def reference(A, B):
        ref = xr.product(lib, A, B)
        return restrict(ref, B.cols, *mask) if mask is not None else ref

    A2, B2 = with_values(A, xr.tier2(A.nnz, 1, dt)), with_values(B, xr.tier2(B.nnz, 2, dt))
    twin_launches = None
    if case.twin_of is not None:
        # the launches of the configuration this case is the twin of, on a context of its own
        for k in case.env:
            monkeypatch.delenv(k)
        for k, v in case.twin_of.items():
            monkeypatch.setenv(k, v)
        with capi.Context() as other:
            other.init(stored(A2, opA), stored(B2, opB), opA, opB)
            other.spgemm()
            twin_launches = other.stats()["kernel_launches"] - 3
        for k in case.twin_of:
            monkeypatch.delenv(k)
        for k, v in case.env.items():
            monkeypatch.setenv(k, v)

    def prove(st, what, reuse=False):
        ok = (REBINNED(st) if reuse and case.direct else case.proof(st)) and (
            reuse or twin_launches is None or st["kernel_launches"] == twin_launches)
        assert ok, f"{case.name} {what}: the statistics do not show the family ran: " + str(
            {k: st[k] for k in ("num_bin_rows", "direct_rows", "direct_retry_rows", "direct_bin_mask", "pattern_mode",
                                "spill_bytes", "transposed_ops", "mask_bin_rows", "kernel_launches")})

    with capi.Context() as ctx:
        def run(A, B, what, exact=False, ref=None):
            """A, B: the effective operands with values; a fresh init_data and spgemm."""
            ctx.init(stored(A, opA), stored(B, opB), opA, opB)
            if mask is not None:
                ctx.set_mask(*mask)
            ctx.spgemm()
            got = ctx.C()
            prove(ctx.stats(), what)
            check_values(got, reference(A, B) if ref is None else ref, f"{case.name} {np.dtype(dt).name} {what}", exact)

        # tier 2's reference first: its p_max sets tier 1's bit budget
        ref2 = reference(A2, B2)
        q = xr.tier1_bits(int(ref2["p"].max(initial=1)), dt)
        run(with_values(A, xr.tier1(A.nnz, q, 3, dt)), with_values(B, xr.tier1(B.nnz, q, 4, dt)), f"tier 1 (q={q})",
            exact=True)
        run(A2, B2, "tier 2", ref=ref2)
        # fresh values on the same context: update_values (values as stored) and spgemm_numeric
        A3, B3 = with_values(A, xr.tier2(A.nnz, 5, dt)), with_values(B, xr.tier2(B.nnz, 6, dt))
        ctx.update_values(stored(A3, opA).val, stored(B3, opB).val)
        ctx.spgemm_numeric()
        got = ctx.C()
        prove(ctx.stats(), "spgemm_numeric", reuse=True)
        check_values(got, reference(A3, B3), f"{case.name} {np.dtype(dt).name} tier 2 after update_values")
        if case.cancel:
            run(*xr.paired(A2, B2, seed=7), "tier 2 cancelling")
        run(with_values(A, xr.tier3(A.nnz, 8, dt)), with_values(B, xr.tier3(B.nnz, 9, dt)), "tier 3")


# ---- masks and non-finite values ---------------------------------------------------------------------------
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_nonfinite_outside_mask_stays_outside(lib, dt):
    """inf and NaN only in B entries none of whose products lands inside the mask: every masked bin gives a
    finite C within the bound of the restricted exact product."""
    A, B, rpM, colM = _bin_operands([r for r, _ in BIN_ROWS], dt)
    A, B = with_values(A, xr.tier2(A.nnz, 11, dt)), with_values(B, xr.tier2(B.nnz, 12, dt))
    # every product (i, k, j) with the index of its B entry
    a_rows = xr.row_index(A.rowptr)
    lens = np.diff(B.rowptr.astype(np.int64))[A.col]
    prod_rows = np.repeat(a_rows, lens)
    b_idx = np.repeat(B.rowptr[A.col].astype(np.int64), lens) + (
        np.arange(lens.sum()) - np.repeat(np.cumsum(lens) - lens, lens))
    inside = np.isin(prod_rows * B.cols + B.col[b_idx], keys(rpM, colM, B.cols))
    free = np.setdiff1d(np.arange(B.nnz), b_idx[inside])
    assert free.size > 1000
    v = B.val.astype(np.float64)
    pick = np.random.default_rng(13).permutation(free)[:free.size // 3]
    v[pick[0::3]], v[pick[1::3]], v[pick[2::3]] = np.inf, -np.inf, np.nan
    B = with_values(B, v)
    with capi.Context() as ctx:
        ctx.init(A, B)
        ctx.set_mask(rpM, colM)
        ctx.spgemm()
        got = ctx.C()
        assert ctx.stats()["mask_bin_rows"] == MASK_BINS
        ref = restrict(xr.product(lib, A, B), B.cols, rpM, colM)
        assert (ref["cls"] == xr.FINITE).all()
        assert np.isfinite(got[2]).all(), "a non-finite product outside the mask reached C"
        check_values(got, ref, f"mask, non-finite outside {np.dtype(dt).name}")


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_masked_cancelling_within_bound(lib, dt):
    """Cancelling operands under random masks over C's pattern: masked C within the bound of the restricted
    exact product."""
    A, B = _cta_hash(dt)
    A, B = xr.paired(with_values(A, xr.tier2(A.nnz, 21, dt)), with_values(B, xr.tier2(B.nnz, 22, dt)), seed=23)
    ref = xr.product(lib, A, B)
    rng = np.random.default_rng(24)
    with capi.Context() as ctx:
        ctx.init(A, B)
        for keep in (0.05, 0.5):
            sel = rng.random(ref["col"].size) < keep
            rows = xr.row_index(ref["rowptr"])
            rpM = np.zeros(A.rows + 1, np.int64)
            np.cumsum(np.bincount(rows[sel], minlength=A.rows), out=rpM[1:])
            colM = ref["col"][sel]
            ctx.set_mask(rpM, colM)
            ctx.spgemm()
            assert ctx.stats()["masked"] == 1
            check_values(ctx.C(), restrict(ref, B.cols, rpM, colM), f"mask keep {keep} cancelling {np.dtype(dt).name}")
