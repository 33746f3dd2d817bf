"""complex128 products on the device against the embedding reference in f64 (tests/complex128_ref.py): every
kernel family of test_values_gpu's case table in every value tier, the path against f64 with the documented
re-routing of 16-byte values, conjugate transposes, the interfaces and the multi-GPU set-up.

Values are checked per component under the value contract (include/bhsparse_b200.h): each component of C_ij is a
real sum of 2p products of f64 values, so test_values_gpu.check_values applies to the real and the imaginary part
with the reference's p = 2p and s of those 2p products.

The on-chip tables sized for 8-byte values do not all hold 16-byte ones (DESIGN.md 4.13).  Rows that take another
kernel than in f64 are proven to run where the library says they do:
  - numeric bin 11 (the 16384-slot CTA hash table) runs in the global-bitmap kernel: counted in bin 12;
  - masked bin 7 (the 16384-slot CTA table) runs in the kernel of masked bin 8: counted there;
  - the direct-mode bin SB_B8192 that follows a wide neighbour is staged as HEAVY (at its products, not at 8192
    entries per row), and HEAVY bins hand k_num_bucket3 rows of at most 4096 products."""
import ctypes
import os
import socket

import numpy as np
import pytest

import complex128_ref as cr
import exact_ref as xr
from benchmark_spgemm_using_csr_b200 import capi, generators as gen
from benchmark_spgemm_using_csr_b200.bhsparse import spgemm
from benchmark_spgemm_using_csr_b200.generators import CSR
from csr_ref import stored
from test_values_gpu import CASES, MASK_BINS, NB, REBINNED, check_values, restrict

pytestmark = pytest.mark.gpu

N, T, C = capi.OP_N, capi.OP_T, capi.OP_C
F64, C128 = np.float64, np.complex128


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    lib = xr.compile_lib(tmp_path_factory.mktemp("exact_ref"))
    assert lib is not None, "gcc is needed to build the quad-precision reference"
    return lib


def cplx(X: CSR, v) -> CSR:
    return CSR(X.rows, X.cols, X.rowptr, X.col, np.asarray(v, C128))


def check_c(got, refs, what, exact=False):
    rp, col, val = got
    assert val.dtype == C128
    check_values((rp, col, val.real), refs[0], what + " (Re)", exact)
    check_values((rp, col, val.imag), refs[1], what + " (Im)", exact)


def product(lib, A, B):
    return cr.product(lib, A, B)


# ---- the routes of 16-byte values --------------------------------------------------------------------------
def routed_num_bins(rows):
    """numeric bin rows as a complex128 product reports them: bin 11's rows in bin 12"""
    rows = list(rows)
    rows[12] += rows[11]
    rows[11] = 0
    return rows


def routed_mask_bins(rows):
    """masked bin rows as a complex128 product reports them: bin 7's rows in bin 8"""
    rows = list(rows)
    rows[8] += rows[7]
    rows[7] = 0
    return rows


def _wide_heavy(st):
    """bins SB_G256 .. SB_B8192 in direct mode, and SB_B8192 staged at its products (HEAVY), not at 8192 per row"""
    wide_entries = sum(st["sym_bin_rows"][b] * (128 << (b - 3)) for b in range(4, 10))
    return (all((st["direct_bin_mask"] >> b) & 1 for b in range(4, 10)) and
            0 < st["direct_ct_bytes"] < wide_entries * (4 + 16))


PROOF_C128 = {
    "cta_hash": lambda st: NB(st, 10, 10) and st["num_bin_rows"][11] == 0 and NB(st, 12, 12),
    "bucket3_wide": _wide_heavy,
    "masked_bins": lambda st: st["mask_bin_rows"] == routed_mask_bins(MASK_BINS),
}


# ---- every kernel family, every tier -------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_values_c128(lib, case, monkeypatch):
    for k, v in case.env.items():
        monkeypatch.setenv(k, v)
    A, B = case.build(F64)
    A, B = A.astype(F64), B.astype(F64)
    mask = case.mask(A, B) if case.mask else None
    opA, opB = case.ops
    proof = PROOF_C128.get(case.name, case.proof)

    def reference(A, B):
        refs = product(lib, A, B)
        return [restrict(r, B.cols, *mask) for r in refs] if mask is not None else refs

    A2, B2 = cplx(A, cr.tier2(A.nnz, 1)), cplx(B, cr.tier2(B.nnz, 2))
    twin_launches = None
    if case.twin_of is not None:
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
        assert st["dtype"] == capi.DTYPE_C128
        ok = (REBINNED(st) if reuse and case.direct else proof(st)) and (
            reuse or twin_launches is None or st["kernel_launches"] == twin_launches)
        assert ok, f"{case.name} {what}: the statistics do not show the family ran: " + str(
            {k: st[k] for k in ("num_bin_rows", "direct_rows", "direct_retry_rows", "direct_bin_mask", "direct_ct_bytes",
                                "pattern_mode", "spill_bytes", "transposed_ops", "mask_bin_rows", "kernel_launches")})

    with capi.Context() as ctx:
        def run(A, B, what, exact=False, ref=None):
            ctx.init(stored(A, opA), stored(B, opB), opA, opB)
            if mask is not None:
                ctx.set_mask(*mask)
            ctx.spgemm()
            got = ctx.C()
            prove(ctx.stats(), what)
            check_c(got, reference(A, B) if ref is None else ref, f"{case.name} c128 {what}", exact)

        ref2 = reference(A2, B2)
        q = xr.tier1_bits(int(ref2[0]["p"].max(initial=1)), F64)   # (p of the reference is 2p: Gaussian integers)
        run(cplx(A, cr.tier1(A.nnz, q, 3)), cplx(B, cr.tier1(B.nnz, q, 4)), f"tier 1 (q={q})", exact=True)
        run(A2, B2, "tier 2", ref=ref2)
        A3, B3 = cplx(A, cr.tier2(A.nnz, 5)), cplx(B, cr.tier2(B.nnz, 6))
        ctx.update_values(stored(A3, opA).val, stored(B3, opB).val)
        ctx.spgemm_numeric()
        got = ctx.C()
        prove(ctx.stats(), "spgemm_numeric", reuse=True)
        check_c(got, reference(A3, B3), f"{case.name} c128 tier 2 after update_values")
        if case.cancel:
            run(*cr.paired(A2, B2, seed=7), "tier 2 cancelling")
        run(cplx(A, cr.tier3(A.nnz, 8)), cplx(B, cr.tier3(B.nnz, 9)), "tier 3")


EQUAL = ("sym_bin_rows", "direct_rows", "direct_retry_rows", "pattern_mode", "nnzC", "transposed_ops")


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_path_against_f64(case, monkeypatch):
    """The same operands in f64 and complex128 take the same path but for the documented routes of 16-byte values:
    numeric bin 11 and masked bin 7 are counted where they ran, and the direct-mode bins SB_B8192 and SB_B16384
    run other launches (so kernel_launches is compared only where none of those rows exist)."""
    for k, v in case.env.items():
        monkeypatch.setenv(k, v)
    A, B = case.build(F64)
    A, B = A.astype(F64), B.astype(F64)
    mask = case.mask(A, B) if case.mask else None
    opA, opB = case.ops
    stats = {}
    real = lambda X, seed: CSR(X.rows, X.cols, X.rowptr, X.col, xr.tier2(X.nnz, seed, F64))
    for name, a, b in (("f64", real(A, 1), real(B, 2)),
                       ("c128", cplx(A, cr.tier2(A.nnz, 1)), cplx(B, cr.tier2(B.nnz, 2)))):
        with capi.Context() as ctx:
            ctx.init(stored(a, opA), stored(b, opB), opA, opB)
            if mask is not None:
                ctx.set_mask(*mask)
            ctx.spgemm()
            stats[name] = ctx.stats()
    f, c = stats["f64"], stats["c128"]
    diff = {k: (f[k], c[k]) for k in EQUAL if f[k] != c[k]}
    if routed_num_bins(f["num_bin_rows"]) != c["num_bin_rows"]:
        diff["num_bin_rows"] = (f["num_bin_rows"], c["num_bin_rows"])
    if routed_mask_bins(f["mask_bin_rows"]) != c["mask_bin_rows"]:
        diff["mask_bin_rows"] = (f["mask_bin_rows"], c["mask_bin_rows"])
    if f["direct_bin_mask"] != c["direct_bin_mask"]:
        diff["direct_bin_mask"] = (f["direct_bin_mask"], c["direct_bin_mask"])
    rerouted = (f["num_bin_rows"][11] > 0 or f["mask_bin_rows"][7] > 0 or (f["direct_bin_mask"] >> 9) & 3)
    if not rerouted and f["kernel_launches"] != c["kernel_launches"]:
        diff["kernel_launches"] = (f["kernel_launches"], c["kernel_launches"])
    assert not diff, f"{case.name}: complex128 took another path than f64 and its routes allow: {diff}"


# ---- conjugate transposes -------------------------------------------------------------------------------------
def _rect_ops():
    """op(A) 700 x 500, op(B) 500 x 900, with complex values"""
    A = gen.random_csr(700, 500, 5 + np.arange(700) % 17, seed=61, dtype=F64)
    B = gen.random_csr(500, 900, 4 + np.arange(500) % 9, seed=62, dtype=F64)
    return cplx(A, cr.tier2(A.nnz, 63)), cplx(B, cr.tier2(B.nnz, 64))


@pytest.mark.parametrize("ops", [(N, C), (C, N), (C, C), (T, C)], ids=["NC", "CN", "CC", "TC"])
def test_conjugate_transpose(lib, ops):
    A, B = _rect_ops()
    with capi.Context() as ctx:
        ctx.init(stored(A, ops[0]), stored(B, ops[1]), *ops)
        ctx.spgemm()
        assert ctx.stats()["transposed_ops"] == (ops[0] != N) | 2 * (ops[1] != N)
        check_c(ctx.C(), product(lib, A, B), f"ops {ops}")
        A3, B3 = cplx(A, cr.tier2(A.nnz, 65)), cplx(B, cr.tier2(B.nnz, 66))
        ctx.update_values(stored(A3, ops[0]).val, stored(B3, ops[1]).val)
        ctx.spgemm_numeric()
        check_c(ctx.C(), product(lib, A3, B3), f"ops {ops} after update_values")


def test_aliased_a_times_a_h(lib):
    """A*A^H from the same host arrays: one upload, one transposition"""
    X = gen.random_csr(600, 450, 3 + np.arange(600) % 11, seed=67, dtype=F64)
    X = cplx(X, cr.tier2(X.nnz, 68))
    with capi.Context() as ctx:
        ctx.init(X, X, N, C, same=True)
        assert ctx.aliased() == 1
        ctx.spgemm()
        check_c(ctx.C(), product(lib, X, cr.conj_transpose(X)), "aliased A*A^H")
        assert ctx.stats()["transposed_ops"] == 2
        X2 = cplx(X, cr.tier2(X.nnz, 69))
        ctx.update_values(X2.val, X2.val)
        ctx.spgemm_numeric()
        check_c(ctx.C(), product(lib, X2, cr.conj_transpose(X2)), "aliased A*A^H after update_values")


# ---- borrowed torch.complex128 operands and the interfaces ----------------------------------------------------
def _torch_operands(X: CSR, dev):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (X.rowptr, X.col, X.val))


def _bits(v):
    return np.ascontiguousarray(v).view(np.uint64)


def test_borrowed_device_operands_and_getters(lib):
    import torch
    dev = torch.device("cuda", 0)
    A, B = _rect_ops()
    Bs = stored(B, C)
    tA, tB = _torch_operands(A, dev), _torch_operands(Bs, dev)
    assert tA[2].dtype == torch.complex128
    ctx = capi.Context()
    L = ctx.lib
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    try:
        ctx.init_device(tA, tB, A.rows, A.cols, B.cols, N, C)
        ctx.spgemm()
        check_c(ctx.C(), product(lib, A, B), "borrowed N,C")
        st = ctx.stats()
        assert st["dtype"] == capi.DTYPE_C128 and st["transposed_ops"] == 2
        # rewritten in place, then spgemm_numeric: the conjugation survives the re-gather
        A3, B3 = cplx(A, cr.tier2(A.nnz, 71)), cplx(B, cr.tier2(B.nnz, 72))
        tA[2].copy_(torch.from_numpy(A3.val).to(dev))
        tB[2].copy_(torch.from_numpy(stored(B3, C).val).to(dev))
        torch.cuda.synchronize(dev)
        ctx.spgemm_numeric()
        rp, col, val = ctx.C()
        check_c((rp, col, val), product(lib, A3, B3), "borrowed N,C after spgemm_numeric")
        nnz = col.size
        # get_C_c128, get_C_range of a slice, get_C_device, copy_C_to_device: bit for bit the same values
        rp32, col2, val2 = np.empty(A.rows + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz, C128)
        capi.check(L, ctx.ctx, L.bhb200_get_C_c128(ctx.ctx, *(ctypes.c_void_p(a.ctypes.data) for a in (rp32, col2, val2))))
        assert np.array_equal(rp32, rp) and np.array_equal(col2, col) and np.array_equal(_bits(val2), _bits(val))
        c3, v3 = np.empty(100, np.int32), np.empty(100, C128)
        capi.check(L, ctx.ctx, L.bhb200_get_C_range(ctx.ctx, nnz - 100, 100, ctypes.c_void_p(c3.ctypes.data),
                                                    ctypes.c_void_p(v3.ctypes.data)))
        assert np.array_equal(c3, col[-100:]) and np.array_equal(_bits(v3), _bits(val[-100:]))
        dvp = ctypes.c_void_p()
        capi.check(L, ctx.ctx, L.bhb200_get_C_device(ctx.ctx, None, None, None, ctypes.byref(dvp)))
        assert dvp.value and dvp.value % 16 == 0
        dview = capi.device_view(dvp.value, 2 * nnz, "float64", dev)
        assert np.array_equal(dview.cpu().numpy().view(np.uint64), _bits(val))
        drp = torch.empty(A.rows + 1, dtype=torch.int64, device=dev)
        dcol = torch.empty(nnz, dtype=torch.int32, device=dev)
        dval = torch.empty(nnz, dtype=torch.complex128, device=dev)
        capi.check(L, ctx.ctx, L.bhb200_copy_C_to_device(ctx.ctx, p(drp), p(dcol), p(dval)))
        assert np.array_equal(drp.cpu().numpy(), rp) and np.array_equal(dcol.cpu().numpy(), col)
        assert np.array_equal(_bits(dval.cpu().numpy()), _bits(val))
        # the structure of the same borrowed arrays, without values
        ctx.init_device((*tA[:2], None), (*tB[:2], None), A.rows, A.cols, B.cols, N, T, capi.DTYPE_NONE)
        ctx.spgemm()
        srp, scol = np.empty(A.rows + 1, np.int32), np.empty(nnz, np.int32)
        capi.check(L, ctx.ctx, L.bhb200_get_C_structure(ctx.ctx, ctypes.c_void_p(srp.ctypes.data),
                                                        ctypes.c_void_p(scol.ctypes.data)))
        assert np.array_equal(srp, rp) and np.array_equal(scol, col)
    finally:
        ctx.close()


def test_misaligned_borrowed_values_are_refused():
    import torch
    dev = torch.device("cuda", 0)
    X = cplx(gen.random_csr(100, 100, 5, seed=3, dtype=F64), cr.tier2(500, 4))
    rp, col, val = _torch_operands(X, dev)
    buf = torch.zeros(2 * X.nnz + 2, dtype=torch.float64, device=dev)   # values at an offset of 8 bytes
    ctx = capi.Context()
    L = ctx.lib
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    try:
        for a, b in ((ctypes.c_void_p(buf.data_ptr() + 8), p(val)), (p(val), ctypes.c_void_p(buf.data_ptr() + 8))):
            rc = L.bhb200_init_data_device(ctx.ctx, capi.DTYPE_C128, 100, 100, 100, X.nnz, a, p(rp), p(col), X.nnz, b,
                                           p(rp), p(col))
            assert rc == capi.ERR_INVALID, "init accepted a complex128 value pointer that is not 16-byte aligned"
            assert "aligned" in L.bhb200_last_error(ctx.ctx).decode()
        # the same pointer is fine for complex64 (8-byte aligned)
        assert L.bhb200_init_data_device(ctx.ctx, capi.DTYPE_C64, 100, 100, 100, X.nnz, ctypes.c_void_p(buf.data_ptr() + 8),
                                         p(rp), p(col), X.nnz, ctypes.c_void_p(buf.data_ptr() + 8), p(rp), p(col)) == 0
    finally:
        ctx.close()


def test_cross_type_refusals():
    L = capi.load()
    X = gen.random_csr(80, 80, 4, seed=5, dtype=F64)
    Xc = cplx(X, cr.tier2(X.nnz, 6))
    out = [np.empty(81, np.int32), np.empty(10000, np.int32), np.empty(20000, C128)]
    po = [ctypes.c_void_p(a.ctypes.data) for a in out]
    ctx = capi.Context()
    try:
        ctx.init(Xc, Xc, same=True)
        ctx.spgemm()
        for fn in (L.bhb200_get_C_f64, L.bhb200_get_C_f32, L.bhb200_get_C_c64):
            assert fn(ctx.ctx, *po) == capi.ERR_INVALID
        for fn in (L.bhb200_update_values_f64, L.bhb200_update_values_f32, L.bhb200_update_values_c64):
            assert fn(ctx.ctx, po[2], po[2]) == capi.ERR_INVALID
        for other in (X, CSR(X.rows, X.cols, X.rowptr, X.col, Xc.val.astype(np.complex64))):
            o = capi.Context()
            try:
                o.init(other, other, same=True)
                o.spgemm()
                assert L.bhb200_get_C_c128(o.ctx, *po) == capi.ERR_INVALID
                assert L.bhb200_update_values_c128(o.ctx, po[2], po[2]) == capi.ERR_INVALID
            finally:
                o.close()
    finally:
        ctx.close()


def test_bhsparse_spgemm_complex128(lib):
    Ar, Br = gen.random_csr(300, 200, 6, seed=7, dtype=F64), gen.random_csr(200, 250, 5, seed=9, dtype=F64)
    A, B = cplx(Ar, cr.tier2(Ar.nnz, 8)), cplx(Br, cr.tier2(Br.nnz, 10))
    check_c(spgemm(A, B), product(lib, A, B), "bhsparse.spgemm")
    check_c(spgemm(A, stored(B, C), transB="C"), product(lib, A, B), "bhsparse.spgemm transB=C")
    B64 = CSR(B.rows, B.cols, B.rowptr, B.col, B.val.astype(np.complex64))
    A64 = CSR(A.rows, A.cols, A.rowptr, A.col, A.val.astype(np.complex64))
    for a, b in ((A, B64), (A64, B), (A, Br)):
        with pytest.raises(capi.BhsparseError, match="mixed value types"):
            spgemm(a, b)


# ---- multi-GPU ---------------------------------------------------------------------------------------------
def _square():
    X = gen.rmat(11, 8, seed=12, dtype=F64)
    return cplx(X, cr.tier2(X.nnz, 13))


def _dist_run(rank, world, out_dir):
    import torch
    from benchmark_spgemm_using_csr_b200.dist import CudaEngine, NcclRowBlockSpGEMM
    dev = torch.device("cuda", rank)
    eng = CudaEngine(rank)
    rb = NcclRowBlockSpGEMM(eng, dev)
    X = _square()
    rb.setup_square_from_device_root(_torch_operands(X, dev) if rank == 0 else None, X.rows)
    rb.spgemm()
    r0, r1, off, total = rb.layout()
    res = eng.result()
    np.savez(os.path.join(out_dir, f"c128_r{rank}.npz"), r0=r0, r1=r1, grp=rb.global_rowptr().cpu().numpy(),
             col=res.col.cpu().numpy(), val=res.val.cpu().numpy())
    eng.close()


def _dist_check(lib, out_dir, world):
    X = _square()
    re, im = product(lib, X, X)
    rp = re["rowptr"]
    cols, vals = [], []
    for r in range(world):
        g = np.load(os.path.join(out_dir, f"c128_r{r}.npz"))
        assert np.array_equal(g["grp"], rp[int(g["r0"]):int(g["r1"]) + 1])
        assert g["val"].dtype == C128
        cols.append(g["col"])
        vals.append(g["val"])
    check_c((rp, np.concatenate(cols), np.concatenate(vals)), (re, im), f"dist_setup_square c128, {world} rank(s)")


def test_dist_setup_square_single_rank(lib, tmp_path):
    _dist_run(0, 1, str(tmp_path))
    _dist_check(lib, str(tmp_path), 1)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _dist_worker(rank, world, port, out_dir):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)     # only carries the 128-byte NCCL id
    try:
        _dist_run(rank, world, out_dir)
    finally:
        dist.destroy_process_group()


def test_dist_setup_square_two_ranks(lib, tmp_path):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mp.spawn(_dist_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    _dist_check(lib, str(tmp_path), 2)
