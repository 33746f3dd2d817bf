"""complex64 products on the device against the embedding reference (tests/complex_ref.py): every kernel family of
test_values_gpu's case table in every value tier, the same path as f64, conjugate transposes, the interfaces and the
multi-GPU set-up.

Values are checked per component under the value contract (include/bhsparse_b200.h): each component of C_ij is a
real sum of 2p products of f32 values, so test_values_gpu.check_values applies to the real and the imaginary part
with the reference's p = 2p and s of those 2p products."""
import ctypes
import os
import socket

import numpy as np
import pytest

import complex_ref as cr
import exact_ref as xr
from benchmark_spgemm_using_csr_b200 import capi, generators as gen
from benchmark_spgemm_using_csr_b200.bhsparse import spgemm
from benchmark_spgemm_using_csr_b200.generators import CSR
from csr_ref import stored
from test_values_gpu import CASES, REBINNED, check_values, restrict

pytestmark = pytest.mark.gpu

N, T, C = capi.OP_N, capi.OP_T, capi.OP_C
F32 = np.float32


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    lib = xr.compile_lib(tmp_path_factory.mktemp("exact_ref"))
    assert lib is not None, "gcc is needed to build the quad-precision reference"
    return lib


def cplx(X: CSR, v) -> CSR:
    return CSR(X.rows, X.cols, X.rowptr, X.col, np.asarray(v, np.complex64))


def check_c(got, refs, what, exact=False):
    rp, col, val = got
    assert val.dtype == np.complex64
    check_values((rp, col, val.real), refs[0], what + " (Re)", exact)
    check_values((rp, col, val.imag), refs[1], what + " (Im)", exact)


# ---- every kernel family, every tier -------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_values_c64(lib, case, monkeypatch):
    for k, v in case.env.items():
        monkeypatch.setenv(k, v)
    A, B = case.build(F32)
    A, B = A.astype(F32), B.astype(F32)
    mask = case.mask(A, B) if case.mask else None
    opA, opB = case.ops

    def reference(A, B):
        refs = cr.product(lib, A, B)
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
        assert st["dtype"] == capi.DTYPE_C64
        ok = (REBINNED(st) if reuse and case.direct else case.proof(st)) and (
            reuse or twin_launches is None or st["kernel_launches"] == twin_launches)
        assert ok, f"{case.name} {what}: the statistics do not show the family ran: " + str(
            {k: st[k] for k in ("num_bin_rows", "direct_rows", "direct_retry_rows", "direct_bin_mask", "pattern_mode",
                                "spill_bytes", "transposed_ops", "mask_bin_rows", "kernel_launches")})

    with capi.Context() as ctx:
        def run(A, B, what, exact=False, ref=None):
            ctx.init(stored(A, opA), stored(B, opB), opA, opB)
            if mask is not None:
                ctx.set_mask(*mask)
            ctx.spgemm()
            got = ctx.C()
            prove(ctx.stats(), what)
            check_c(got, reference(A, B) if ref is None else ref, f"{case.name} c64 {what}", exact)

        ref2 = reference(A2, B2)
        q = xr.tier1_bits(int(ref2[0]["p"].max(initial=1)), F32)   # (p of the reference is 2p: Gaussian integers)
        run(cplx(A, cr.tier1(A.nnz, q, 3)), cplx(B, cr.tier1(B.nnz, q, 4)), f"tier 1 (q={q})", exact=True)
        run(A2, B2, "tier 2", ref=ref2)
        A3, B3 = cplx(A, cr.tier2(A.nnz, 5)), cplx(B, cr.tier2(B.nnz, 6))
        ctx.update_values(stored(A3, opA).val, stored(B3, opB).val)
        ctx.spgemm_numeric()
        got = ctx.C()
        prove(ctx.stats(), "spgemm_numeric", reuse=True)
        check_c(got, reference(A3, B3), f"{case.name} c64 tier 2 after update_values")
        if case.cancel:
            run(*cr.paired(A2, B2, seed=7), "tier 2 cancelling")
        run(cplx(A, cr.tier3(A.nnz, 8)), cplx(B, cr.tier3(B.nnz, 9)), "tier 3")


SAME_PATH = ("sym_bin_rows", "num_bin_rows", "direct_bin_mask", "direct_rows", "direct_retry_rows", "pattern_mode",
             "mask_bin_rows", "nnzC", "kernel_launches")


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_same_path_as_f64(case, monkeypatch):
    """A complex64 value has the size of a double: the product of the same operands takes the same bins, plans,
    modes and kernels."""
    for k, v in case.env.items():
        monkeypatch.setenv(k, v)
    A, B = case.build(np.float64)
    A, B = A.astype(np.float64), B.astype(np.float64)
    mask = case.mask(A, B) if case.mask else None
    opA, opB = case.ops
    stats = {}
    real = lambda X, seed: CSR(X.rows, X.cols, X.rowptr, X.col, xr.tier2(X.nnz, seed, np.float64))
    for name, a, b in (("f64", real(A, 1), real(B, 2)), ("c64", cplx(A, cr.tier2(A.nnz, 1)), cplx(B, cr.tier2(B.nnz, 2)))):
        with capi.Context() as ctx:
            ctx.init(stored(a, opA), stored(b, opB), opA, opB)
            if mask is not None:
                ctx.set_mask(*mask)
            ctx.spgemm()
            stats[name] = ctx.stats()
    diff = {k: (stats["f64"][k], stats["c64"][k]) for k in SAME_PATH if stats["f64"][k] != stats["c64"][k]}
    assert not diff, f"{case.name}: complex64 took another path than f64: {diff}"


# ---- conjugate transposes -------------------------------------------------------------------------------------
def _rect_ops(opA, opB):
    """op(A) 700 x 500, op(B) 500 x 900, with complex values"""
    A = gen.random_csr(700, 500, 5 + np.arange(700) % 17, seed=61, dtype=F32)
    B = gen.random_csr(500, 900, 4 + np.arange(500) % 9, seed=62, dtype=F32)
    return cplx(A, cr.tier2(A.nnz, 63)), cplx(B, cr.tier2(B.nnz, 64))


@pytest.mark.parametrize("ops", [(N, C), (C, N), (C, C), (T, C)], ids=["NC", "CN", "CC", "TC"])
def test_conjugate_transpose(lib, ops):
    A, B = _rect_ops(*ops)
    with capi.Context() as ctx:
        ctx.init(stored(A, ops[0]), stored(B, ops[1]), *ops)
        ctx.spgemm()
        assert ctx.stats()["transposed_ops"] == (ops[0] != N) | 2 * (ops[1] != N)
        check_c(ctx.C(), cr.product(lib, A, B), f"ops {ops}")
        # new values as stored: conjugated again into the transposed copies
        A3, B3 = cplx(A, cr.tier2(A.nnz, 65)), cplx(B, cr.tier2(B.nnz, 66))
        ctx.update_values(stored(A3, ops[0]).val, stored(B3, ops[1]).val)
        ctx.spgemm_numeric()
        check_c(ctx.C(), cr.product(lib, A3, B3), f"ops {ops} after update_values")


@pytest.mark.parametrize("ops", [(N, C), (C, C)], ids=["A_AH", "AH_AH"])
def test_aliased_host_arrays(lib, ops):
    """A*A^H and A^H*A^H from the same host arrays: one upload, one transposed copy when both ops are equal"""
    X = gen.random_csr(600, 600 if ops == (C, C) else 450, 3 + np.arange(600) % 11, seed=67, dtype=F32)
    X = cplx(X, cr.tier2(X.nnz, 68))
    with capi.Context() as ctx:
        ctx.init(X, X, *ops, same=True)
        assert ctx.lib.bhb200_operands_aliased(ctx.ctx) == 1
        eff = [X if o == N else cr.conj_transpose(X) for o in ops]
        ctx.spgemm()
        check_c(ctx.C(), cr.product(lib, *eff), f"aliased {ops}")
        assert ctx.stats()["transposed_ops"] == (ops[0] != N) | 2
        X2 = cplx(X, cr.tier2(X.nnz, 69))
        ctx.update_values(X2.val, X2.val)
        ctx.spgemm_numeric()
        eff = [X2 if o == N else cr.conj_transpose(X2) for o in ops]
        check_c(ctx.C(), cr.product(lib, *eff), f"aliased {ops} after update_values")


def test_real_operands_refuse_op_c():
    c = capi.Context()
    lib, ctx = c.lib, c.ctx
    try:
        X = gen.random_csr(50, 50, 4, seed=1)
        p = [ctypes.c_void_p(np.ascontiguousarray(a).ctypes.data) for a in (X.val, X.rowptr, X.col)]
        for op in ((N, C), (C, N)):
            assert lib.bhb200_init_data_op_f64(ctx, *op, 50, 50, 50, X.nnz, *p, X.nnz, *p) == capi.ERR_INVALID
            assert lib.bhb200_init_data_op_f32(ctx, *op, 50, 50, 50, X.nnz, *p, X.nnz, *p) == capi.ERR_INVALID
            assert lib.bhb200_init_data_structure(ctx, *op, 50, 50, 50, X.nnz, *p[1:], X.nnz, *p[1:]) == capi.ERR_INVALID
            assert lib.bhb200_init_data_device_op(ctx, capi.DTYPE_F64, *op, 50, 50, 50, 0, None, p[1], None, 0, None, p[1],
                                                  None) == capi.ERR_INVALID
    finally:
        c.close()


# ---- borrowed torch.complex64 operands and the interfaces -----------------------------------------------------
def _torch_operands(X: CSR, dev):
    import torch
    return tuple(torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (X.rowptr, X.col, X.val))


def test_borrowed_device_operands(lib):
    import torch
    dev = torch.device("cuda", 0)
    A, B = _rect_ops(N, C)
    Bs = stored(B, C)
    tA, tB = _torch_operands(A, dev), _torch_operands(Bs, dev)
    ctx = capi.Context()
    L = ctx.lib
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    try:
        ctx.init_device(tA, tB, A.rows, A.cols, B.cols, N, C)
        ctx.spgemm()
        got = ctx.C()
        check_c(got, cr.product(lib, A, B), "borrowed N,C")
        st = ctx.stats()
        assert st["dtype"] == capi.DTYPE_C64 and st["transposed_ops"] == 2
        # rewritten in place, then spgemm_numeric: the conjugation survives the re-gather
        A3, B3 = cplx(A, cr.tier2(A.nnz, 71)), cplx(B, cr.tier2(B.nnz, 72))
        tA[2].copy_(torch.from_numpy(A3.val).to(dev))
        tB[2].copy_(torch.from_numpy(stored(B3, C).val).to(dev))
        torch.cuda.synchronize(dev)
        ctx.spgemm_numeric()
        rp, col, val = ctx.C()
        check_c((rp, col, val), cr.product(lib, A3, B3), "borrowed N,C after spgemm_numeric")
        nnz = col.size
        # get_C_c64, get_C_range of a slice, get_C_device, copy_C_to_device
        rp32, col2, val2 = np.empty(A.rows + 1, np.int32), np.empty(nnz, np.int32), np.empty(nnz, np.complex64)
        capi.check(L, ctx.ctx, L.bhb200_get_C_c64(ctx.ctx, *(ctypes.c_void_p(a.ctypes.data) for a in (rp32, col2, val2))))
        assert np.array_equal(rp32, rp) and np.array_equal(col2, col) and np.array_equal(val2.view(np.uint64), val.view(np.uint64))
        c3, v3 = np.empty(100, np.int32), np.empty(100, np.complex64)
        capi.check(L, ctx.ctx, L.bhb200_get_C_range(ctx.ctx, nnz - 100, 100, ctypes.c_void_p(c3.ctypes.data), ctypes.c_void_p(v3.ctypes.data)))
        assert np.array_equal(c3, col[-100:]) and np.array_equal(v3.view(np.uint64), val[-100:].view(np.uint64))
        dvp = ctypes.c_void_p()
        capi.check(L, ctx.ctx, L.bhb200_get_C_device(ctx.ctx, None, None, None, ctypes.byref(dvp)))
        assert dvp.value and dvp.value % 8 == 0
        drp = torch.empty(A.rows + 1, dtype=torch.int64, device=dev)
        dcol = torch.empty(nnz, dtype=torch.int32, device=dev)
        dval = torch.empty(nnz, dtype=torch.complex64, device=dev)
        capi.check(L, ctx.ctx, L.bhb200_copy_C_to_device(ctx.ctx, p(drp), p(dcol), p(dval)))
        assert np.array_equal(drp.cpu().numpy(), rp) and np.array_equal(dcol.cpu().numpy(), col)
        assert np.array_equal(dval.cpu().numpy().view(np.uint64), val.view(np.uint64))
        # the structure of the same borrowed arrays, without values
        ctx.init_device((*tA[:2], None), (*tB[:2], None), A.rows, A.cols, B.cols, N, T, capi.DTYPE_NONE)
        ctx.spgemm()
        srp, scol = np.empty(A.rows + 1, np.int32), np.empty(nnz, np.int32)
        capi.check(L, ctx.ctx, L.bhb200_get_C_structure(ctx.ctx, ctypes.c_void_p(srp.ctypes.data), ctypes.c_void_p(scol.ctypes.data)))
        assert np.array_equal(srp, rp) and np.array_equal(scol, col)
    finally:
        ctx.close()


def test_misaligned_borrowed_values_are_refused():
    import torch
    dev = torch.device("cuda", 0)
    X = cplx(gen.random_csr(100, 100, 5, seed=3, dtype=F32), cr.tier2(500, 4))
    rp, col, val = _torch_operands(X, dev)
    buf = torch.zeros(2 * X.nnz + 2, dtype=torch.float32, device=dev)   # values at an offset of 4 bytes
    ctx = capi.Context()
    L = ctx.lib
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    try:
        rc = L.bhb200_init_data_device(ctx.ctx, capi.DTYPE_C64, 100, 100, 100, X.nnz, ctypes.c_void_p(buf.data_ptr() + 4),
                                       p(rp), p(col), X.nnz, p(val), p(rp), p(col))
        assert rc == capi.ERR_INVALID, "init accepted a complex64 value pointer that is not 8-byte aligned"
        assert "aligned" in L.bhb200_last_error(ctx.ctx).decode()
    finally:
        ctx.close()


def test_cross_type_refusals():
    L = capi.load()
    X = gen.random_csr(80, 80, 4, seed=5, dtype=F32)
    Xc = cplx(X, cr.tier2(X.nnz, 6))
    out = [np.empty(81, np.int32), np.empty(10000, np.int32), np.empty(20000, np.float64)]
    po = [ctypes.c_void_p(a.ctypes.data) for a in out]
    ctx = capi.Context()
    try:
        ctx.init(Xc, Xc, same=True)
        ctx.spgemm()
        for fn in (L.bhb200_get_C_f64, L.bhb200_get_C_f32):
            assert fn(ctx.ctx, *po) == capi.ERR_INVALID
        for fn in (L.bhb200_update_values_f64, L.bhb200_update_values_f32):
            assert fn(ctx.ctx, po[2], po[2]) == capi.ERR_INVALID
        real = capi.Context()
        try:
            real.init(X, X, same=True)
            real.spgemm()
            assert L.bhb200_get_C_c64(real.ctx, *po) == capi.ERR_INVALID
            assert L.bhb200_update_values_c64(real.ctx, po[2], po[2]) == capi.ERR_INVALID
        finally:
            real.close()
    finally:
        ctx.close()


def test_bhsparse_spgemm_complex(lib):
    Ar, Br = gen.random_csr(300, 200, 6, seed=7, dtype=F32), gen.random_csr(200, 250, 5, seed=9, dtype=F32)
    A, B = cplx(Ar, cr.tier2(Ar.nnz, 8)), cplx(Br, cr.tier2(Br.nnz, 10))
    check_c(spgemm(A, B), cr.product(lib, A, B), "bhsparse.spgemm")
    check_c(spgemm(A, stored(B, C), transB="C"), cr.product(lib, A, B), "bhsparse.spgemm transB=C")
    A128 = CSR(A.rows, A.cols, A.rowptr, A.col, A.val.astype(np.complex128))
    with pytest.raises(capi.BhsparseError, match="complex64"):
        spgemm(A128, B)


# ---- multi-GPU ---------------------------------------------------------------------------------------------
def _square():
    X = gen.rmat(11, 8, seed=12, dtype=F32)
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
    np.savez(os.path.join(out_dir, f"c64_r{rank}.npz"), r0=r0, r1=r1, grp=rb.global_rowptr().cpu().numpy(),
             col=res.col.cpu().numpy(), val=res.val.cpu().numpy())
    eng.close()


def _dist_check(lib, out_dir, world):
    X = _square()
    re, im = cr.product(lib, X, X)
    rp = re["rowptr"]
    cols, vals = [], []
    for r in range(world):
        g = np.load(os.path.join(out_dir, f"c64_r{r}.npz"))
        assert np.array_equal(g["grp"], rp[int(g["r0"]):int(g["r1"]) + 1])
        assert g["val"].dtype == np.complex64
        cols.append(g["col"])
        vals.append(g["val"])
    check_c((rp, np.concatenate(cols), np.concatenate(vals)), (re, im), f"dist_setup_square c64, {world} rank(s)")


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
