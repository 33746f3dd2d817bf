"""1-D row-block SpGEMM across the GPUs of one node (one process per GPU).

The reference is single-GPU (device 0 hard-wired, bhsparse_cuda.h:100-101); this
is the multi-GPU scheme BASELINE.json's north_star asks for (SURVEY.md 8e):

  * rows of A are split into contiguous blocks whose boundaries sit on the prefix
    sum of the per-row intermediate-product counts (NOT equal row counts: R-MAT
    rows range from 0 to >10^5 products);
  * B is broadcast once from the root with NCCL (three arrays: rowptr, col, val);
  * every rank runs the single-GPU pipeline on its block (device-resident operands,
    C-ABI bhb200_init_data_device / bhb200_spgemm);
  * the per-rank nnz(C) are all-gathered (one int64 per rank) and exclusive-scanned
    into each rank's global offset, so C is assembled without a host round trip:
    global rowptrC of block r = local rowptrC + offset[r]; C stays row-sharded.

There is no data-path collective inside the SpGEMM itself: C's row block depends
only on A's row block and B.  torch.distributed is plumbing (NCCL on GPUs; gloo
with CPU tensors in the host-logic tests, where the compute engine is injected).
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np
import torch
import torch.distributed as dist

from . import capi
from .generators import CSR


def _torch_dtype(name) -> torch.dtype:
    """torch dtype of a supported value type (capi.dtype_of raises for others)"""
    return getattr(torch, capi.VALUE_TYPES[capi.dtype_of(name)][1])


def row_products_host(A: CSR, B_rowptr: np.ndarray) -> np.ndarray:
    """Per-row intermediate products on the host (partitioning only; the device
    pipeline recomputes them in k_row_products)."""
    lenB = np.diff(B_rowptr.astype(np.int64))
    per_entry = lenB[A.col]
    csum = np.zeros(A.nnz + 1, dtype=np.int64)
    np.cumsum(per_entry, out=csum[1:])
    return csum[A.rowptr[1:].astype(np.int64)] - csum[A.rowptr[:-1].astype(np.int64)]


COST_HEAVY_ROW = 12288


def row_cost(row_products: np.ndarray) -> np.ndarray:
    """Cost of a row for the partition (csrc/dist_nccl.cu::k_row_cost is the same function): its
    intermediate products, times 11/8 beyond 12288 products -- rows that leave the on-chip tables (sliced
    through global memory by k_num_bucket_heavy2) cost about that much more per product, and R-MAT's hub rows all
    sit in the first block (R-MAT 24 / 8 blocks, measured per block: 24.4 products/ns in block 0, 26.1 in block 3;
    the factor was 2.5 for the first heavy-row kernel; 1.25 left block 0 the slowest by 3 % at 8 GPUs)."""
    p = row_products.astype(np.int64)
    return np.minimum(np.where(p > COST_HEAVY_ROW, (p * 11) // 8, p), np.int64(0x7FFFFFFF))


def partition_rows_by_products(row_products: np.ndarray, world: int) -> np.ndarray:
    """Boundaries b[0..world] with b[0]=0, b[world]=m such that every block holds
    about the same number of intermediate products (a row is never split)."""
    m = int(row_products.size)
    prefix = np.zeros(m + 1, dtype=np.int64)
    np.cumsum(row_products, out=prefix[1:])
    total = int(prefix[-1])
    bounds = np.zeros(world + 1, dtype=np.int64)
    bounds[world] = m
    for r in range(1, world):
        target = (total * r) // world
        bounds[r] = int(np.searchsorted(prefix, target, side="left"))
    bounds = np.maximum.accumulate(np.minimum(bounds, m))
    return bounds


@dataclass
class LocalResult:
    nnzC: int
    rowptr64: object      # torch int64 [rows+1] (device) or numpy
    col: object
    val: object


class CudaEngine(capi.Context):
    """Runs one row block through the C-ABI with device-resident operands."""

    def __init__(self, device: int):
        super().__init__(device)
        # The library must run on a stream that is ordered after the producers of its operands
        # (torch kernels, NCCL receives) -- not on the context's private non-blocking stream.
        # Default: torch's current stream; the legacy default stream has handle 0, which
        # bhb200_set_stream reads as "own stream", so a dedicated torch stream is used then and
        # set_operands()/spgemm() make it wait for the current stream.
        cur = torch.cuda.current_stream(device)
        self._own = None
        if cur.cuda_stream == 0:
            self._own = torch.cuda.Stream(device=device)
            self.use_stream(self._own.cuda_stream)
        else:
            self.use_stream(cur.cuda_stream)

    def use_stream(self, cuda_stream_ptr: int):
        self.set_stream(cuda_stream_ptr)
        if self._own is not None and cuda_stream_ptr != self._own.cuda_stream:
            self._own = None

    def _order_after_producers(self):
        if self._own is not None:
            self._own.wait_stream(torch.cuda.current_stream(self.device))

    @property
    def vdtype(self):
        """torch dtype of the values of C"""
        return getattr(torch, capi.VALUE_TYPES[self.dtype][1])

    def set_operands(self, m, k, n, A, B):
        """A, B = (rowptr, col, val) torch CUDA tensors (int32, int32, f32/f64/complex64/complex128)."""
        self._order_after_producers()
        self.init_device(A, B, m, k, n)

    def spgemm(self) -> int:
        self._order_after_producers()
        return super().spgemm()

    def result(self) -> LocalResult:
        """Copies of the device-resident result as torch tensors (capi.Context.C_device)."""
        rowptr, col, val = self.C_device()
        return LocalResult(int(col.numel()), rowptr, col, val)


class RowBlockSpGEMM:
    """C = A*B with A row-partitioned over the ranks of `group` (see module doc)."""

    def __init__(self, engine, device: torch.device, group=None):
        self.engine = engine
        self.device = device
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.bounds = None
        self.meta = None
        self.A = None
        self.B = None
        self.timings = {}

    # -- setup: partition, broadcast B, hand out the row blocks of A ---------------
    def setup_from_root(self, A: CSR | None, B: CSR | None, root: int = 0, a_equals_b: bool = False):
        """A, B are host CSR on `root` (None elsewhere).  With a_equals_b the row
        blocks of A are sliced out of the broadcast copy of B instead of being sent."""
        dev = self.device
        if self.rank == root:
            prods = row_products_host(A, B.rowptr)
            bounds = partition_rows_by_products(row_cost(prods), self.world)
            meta = dict(m=A.rows, k=A.cols, n=B.cols, nnzA=A.nnz, nnzB=B.nnz, dtype=str(A.val.dtype),
                        bounds=bounds.tolist(), nnz_bounds=[int(A.rowptr[b]) for b in bounds],
                        products=int(prods.sum()))
        else:
            meta = None
        if self.world > 1:
            box = [meta]
            dist.broadcast_object_list(box, src=root, group=self.group)
            meta = box[0]
        self.meta = meta
        self.bounds = np.asarray(meta["bounds"], dtype=np.int64)
        vt = _torch_dtype(meta["dtype"])

        # B: three broadcasts (rowptr first: it is all k_row_products needs)
        def bcast(host_arr, numel, tdtype):
            if self.rank == root:
                t = torch.from_numpy(np.ascontiguousarray(host_arr)).to(dev, non_blocking=False)
            else:
                t = torch.empty(numel, dtype=tdtype, device=dev)
            if self.world > 1:
                dist.broadcast(t, src=root, group=self.group)
            return t

        t0 = _now(dev)
        Brp = bcast(B.rowptr if B is not None else None, meta["k"] + 1, torch.int32)
        Bc = bcast(B.col if B is not None else None, meta["nnzB"], torch.int32)
        Bv = bcast(B.val if B is not None else None, meta["nnzB"], vt)
        self.timings["broadcast_B_s"] = _now(dev) - t0
        self.B = (Brp, Bc, Bv)

        r0, r1 = int(self.bounds[self.rank]), int(self.bounds[self.rank + 1])
        e0, e1 = meta["nnz_bounds"][self.rank], meta["nnz_bounds"][self.rank + 1]
        if a_equals_b and self.world == 1:
            self.A = self.B                    # one rank: A IS B (same arrays: the library sees C = B*B)
        elif a_equals_b:
            Arp = (Brp[r0:r1 + 1] - Brp[r0]).contiguous()
            self.A = (Arp, Bc[e0:e1], Bv[e0:e1])
        else:
            self.A = self._scatter_A(A, root, vt)
        self.engine.set_operands(r1 - r0, meta["k"], meta["n"], self.A, self.B)
        return self

    def setup_square_from_device_root(self, B_dev, n: int, root: int = 0):
        """C = B*B with B = (rowptr int32, col int32, val) torch tensors ALREADY ON `root`'s device
        (None elsewhere), n x n.  Partition on the per-row products (computed on the device),
        B broadcast with NCCL -- rowptr first --, every rank slices its row block of A out of its
        copy of B.  Nothing passes through host memory except the few partition boundaries."""
        dev = self.device
        if self.rank == root:
            Brp, Bc, Bv = B_dev
            lenB = (Brp[1:] - Brp[:-1]).to(torch.int64)
            csum = torch.zeros(Bc.numel() + 1, dtype=torch.int64, device=dev)
            torch.cumsum(lenB[Bc.to(torch.int64)], 0, out=csum[1:])
            rp64 = Brp.to(torch.int64)
            prods = csum[rp64[1:]] - csum[rp64[:-1]]
            prefix = torch.zeros(n + 1, dtype=torch.int64, device=dev)
            torch.cumsum(prods, 0, out=prefix[1:])
            total = int(prefix[-1].item())
            cost = torch.where(prods > COST_HEAVY_ROW, (prods * 11) // 8, prods).clamp(max=0x7FFFFFFF)      # row_cost()
            cprefix = torch.zeros(n + 1, dtype=torch.int64, device=dev)
            torch.cumsum(cost, 0, out=cprefix[1:])
            ctotal = int(cprefix[-1].item())
            targets = torch.tensor([(ctotal * r) // self.world for r in range(1, self.world)], dtype=torch.int64, device=dev)
            inner = torch.searchsorted(cprefix, targets, right=False).clamp(max=n).cpu().numpy() if self.world > 1 else []
            bounds = np.maximum.accumulate(np.concatenate([[0], np.asarray(inner, dtype=np.int64), [n]]).astype(np.int64))
            nnz_bounds = [int(x) for x in Brp[torch.from_numpy(bounds).to(dev)].cpu().numpy()]
            block_products = [int((prefix[int(bounds[r + 1])] - prefix[int(bounds[r])]).item()) for r in range(self.world)]
            meta = dict(m=n, k=n, n=n, nnzA=int(Bc.numel()), nnzB=int(Bc.numel()), dtype=str(Bv.dtype).replace("torch.", ""),
                        bounds=bounds.tolist(), nnz_bounds=nnz_bounds, products=total, block_products=block_products,
                        max_row_products=int(prods.max().item()))
            del lenB, csum, rp64, prods, prefix, cost, cprefix
        else:
            meta = None
        if self.world > 1:
            box = [meta]
            dist.broadcast_object_list(box, src=root, group=self.group)
            meta = box[0]
        self.meta = meta
        self.bounds = np.asarray(meta["bounds"], dtype=np.int64)
        vt = _torch_dtype(meta["dtype"])

        def bcast(t, numel, tdtype):
            if self.rank != root:
                t = torch.empty(numel, dtype=tdtype, device=dev)
            if self.world > 1:
                dist.broadcast(t, src=root, group=self.group)
            return t

        t0 = _now(dev)
        Brp = bcast(B_dev[0] if self.rank == root else None, n + 1, torch.int32)
        Bc = bcast(B_dev[1] if self.rank == root else None, meta["nnzB"], torch.int32)
        Bv = bcast(B_dev[2] if self.rank == root else None, meta["nnzB"], vt)
        self.timings["broadcast_B_s"] = _now(dev) - t0
        self.B = (Brp, Bc, Bv)
        r0, r1 = int(self.bounds[self.rank]), int(self.bounds[self.rank + 1])
        e0, e1 = meta["nnz_bounds"][self.rank], meta["nnz_bounds"][self.rank + 1]
        if self.world == 1:
            self.A = self.B                    # one rank: A IS B (same arrays: the library sees C = B*B)
        else:
            Arp = (Brp[r0:r1 + 1] - Brp[r0]).contiguous()
            self.A = (Arp, Bc[e0:e1], Bv[e0:e1])
        self.engine.set_operands(r1 - r0, n, n, self.A, self.B)
        return self

    def _scatter_A(self, A, root, vt):
        dev = self.device
        nb = self.meta["nnz_bounds"]
        mine = None
        if self.rank == root:
            for r in range(self.world):
                r0, r1 = int(self.bounds[r]), int(self.bounds[r + 1])
                blk = (torch.from_numpy((A.rowptr[r0:r1 + 1] - A.rowptr[r0]).astype(np.int32)),
                       torch.from_numpy(np.ascontiguousarray(A.col[nb[r]:nb[r + 1]])),
                       torch.from_numpy(np.ascontiguousarray(A.val[nb[r]:nb[r + 1]])))
                blk = tuple(t.to(dev) for t in blk)
                if r == root:
                    mine = blk
                else:
                    for t in blk:
                        dist.send(t, dst=r, group=self.group)
        else:
            r0, r1 = int(self.bounds[self.rank]), int(self.bounds[self.rank + 1])
            cnt = nb[self.rank + 1] - nb[self.rank]
            mine = (torch.empty(r1 - r0 + 1, dtype=torch.int32, device=dev),
                    torch.empty(cnt, dtype=torch.int32, device=dev), torch.empty(cnt, dtype=vt, device=dev))
            for t in mine:
                dist.recv(t, src=root, group=self.group)
        return mine

    # -- the step: local pipeline + one int64 all-gather ------------------------------
    def spgemm(self):
        """Returns (nnzC_local, global_offset, nnzC_total)."""
        nnz_local = self.engine.spgemm()
        if self.world > 1:
            mine = torch.tensor([nnz_local], dtype=torch.int64, device=self.device)
            parts = [torch.empty(1, dtype=torch.int64, device=self.device) for _ in range(self.world)]
            dist.all_gather(parts, mine, group=self.group)
            counts = torch.cat(parts).cpu().numpy()
        else:
            counts = np.array([nnz_local], dtype=np.int64)
        offs = np.zeros(self.world + 1, dtype=np.int64)
        np.cumsum(counts, out=offs[1:])
        self.counts = counts
        return nnz_local, int(offs[self.rank]), int(offs[-1])

    # -- optional assembly: the full C on every rank (tests / small problems) ----------
    def gather_full(self, offset: int, total: int):
        """All-gather the row-sharded C into (rowptr int64[m+1], col, val) on every
        rank.  Each rank contributes its block at its final offset; no host staging
        of the payload."""
        res = self.engine.result()
        rowptr = _dev(res.rowptr64, self.device, torch.int64)
        col = _dev(res.col, self.device, torch.int32)
        val = _dev(res.val, self.device, None)
        if self.world == 1:
            return rowptr.cpu().numpy(), col.cpu().numpy(), val.cpu().numpy()
        m = self.meta["m"]
        g_rowptr = torch.zeros(m + 1, dtype=torch.int64, device=self.device)
        g_col = torch.zeros(total, dtype=torch.int32, device=self.device)
        g_val = torch.zeros(total, dtype=val.dtype, device=self.device)
        r0, r1 = int(self.bounds[self.rank]), int(self.bounds[self.rank + 1])
        g_rowptr[r0 + 1:r1 + 1] = rowptr[1:] + offset
        g_col[offset:offset + res.nnzC] = col
        g_val[offset:offset + res.nnzC] = val
        # disjoint supports -> a sum all-reduce assembles the arrays in place
        for t in (g_rowptr, g_col, g_val):
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return g_rowptr.cpu().numpy(), g_col.cpu().numpy(), g_val.cpu().numpy()


def _dev(x, device, dtype):
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x))
    x = x.to(device)
    return x if dtype is None else x.to(dtype)


def _now(device) -> float:
    import time
    if device.type == "cuda":
        torch.cuda.synchronize(device)
    return time.perf_counter()


class NcclRowBlockSpGEMM:
    """C = B*B across the ranks THROUGH THE C-ABI (bhb200_dist_*, csrc/dist_nccl.cu): partition,
    NCCL broadcast of B, per-step all-gather of nnz(C) and the global row pointers all happen inside
    the library; torch.distributed only carries the 128-byte NCCL id to the ranks.  Same interface
    as RowBlockSpGEMM where bench.py and the tests need it."""

    def __init__(self, engine: CudaEngine, device: torch.device, group=None):
        self.engine, self.device, self.group = engine, device, group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.meta, self.timings, self._keep = None, {}, None
        lib, ctx = engine.lib, engine.ctx
        uid = ctypes.create_string_buffer(capi.DIST_ID_BYTES)
        if self.rank == 0:
            capi.check(lib, ctx, lib.bhb200_dist_unique_id(uid))
        if self.world > 1:
            box = [uid.raw]
            dist.broadcast_object_list(box, src=0, group=group)
            uid = ctypes.create_string_buffer(box[0], capi.DIST_ID_BYTES)
        capi.check(lib, ctx, lib.bhb200_dist_init(ctx, self.rank, self.world, uid))

    def setup_square_from_device_root(self, B_dev, n: int = 0, root: int = 0):
        lib, ctx = self.engine.lib, self.engine.ctx
        self.engine._order_after_producers()
        info = [None]
        if self.rank == root:
            Brp, Bc, Bv = B_dev
            self._keep = B_dev
            info = [(int(Bc.numel()), str(Bv.dtype).replace("torch.", ""), int(Brp.numel()) - 1)]
        if self.world > 1:
            dist.broadcast_object_list(info, src=root, group=self.group)
        nnz, dname, n = info[0]              # (n is taken from the root's arrays)
        dtype = capi.dtype_of(dname)
        p = (lambda t: ctypes.c_void_p(t.data_ptr())) if self.rank == root else (lambda t: None)
        capi.check(lib, ctx, lib.bhb200_dist_setup_square(
            ctx, root, dtype, n, nnz, p(B_dev[0] if B_dev else None), p(B_dev[1] if B_dev else None),
            p(B_dev[2] if B_dev else None)))
        ms = ctypes.c_float(0)
        capi.check(lib, ctx, lib.bhb200_dist_broadcast_ms(ctx, ctypes.byref(ms)))
        self.timings["broadcast_B_s"] = ms.value * 1e-3
        r0, r1, ptot = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
        capi.check(lib, ctx, lib.bhb200_dist_get_layout(ctx, ctypes.byref(r0), ctypes.byref(r1), None, None, ctypes.byref(ptot)))
        bp = (ctypes.c_int64 * self.world)()
        capi.check(lib, ctx, lib.bhb200_dist_get_block_products(ctx, bp))
        self.rows = (int(r0.value), int(r1.value))
        self.engine.m, self.engine.dtype = self.rows[1] - self.rows[0], dtype
        self.meta = dict(m=n, k=n, n=n, nnzA=nnz, nnzB=nnz, dtype=dname, products=int(ptot.value),
                         block_products=[int(x) for x in bp])
        return self

    def spgemm(self):
        """Returns (nnzC_local, None, None): offsets and totals stay on the device; layout() reads them."""
        lib, ctx = self.engine.lib, self.engine.ctx
        self.engine._order_after_producers()
        capi.check(lib, ctx, lib.bhb200_dist_spgemm(ctx))
        return int(lib.bhb200_get_nnzC(ctx)), None, None

    @property
    def A(self):
        """This rank's row block of A as the library holds it (views of device memory)."""
        return self.engine.operands()[1]

    @property
    def B(self):
        return self.engine.operands()[2]

    def layout(self):
        """(row_begin, row_end, nnz_offset, nnz_total) of this rank -- copies nranks int64 from the device."""
        lib, ctx = self.engine.lib, self.engine.ctx
        v = [ctypes.c_int64() for _ in range(4)]
        capi.check(lib, ctx, lib.bhb200_dist_get_layout(ctx, *(ctypes.byref(x) for x in v), None))
        return tuple(int(x.value) for x in v)

    def global_rowptr(self) -> torch.Tensor:
        """Device tensor (copy) of this block's GLOBAL row pointers."""
        lib, ctx = self.engine.lib, self.engine.ctx
        ptr = ctypes.c_void_p()
        capi.check(lib, ctx, lib.bhb200_dist_get_global_rowptr_device(ctx, ctypes.byref(ptr)))
        capi.check(lib, ctx, lib.bhb200_synchronize(ctx))
        return capi.device_view(ptr.value, self.engine.m + 1, "int64", self.device).clone()


_DevicePtr = capi.DevicePtr   # the name code written against earlier versions of this module imports
