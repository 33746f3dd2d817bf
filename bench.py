#!/usr/bin/env python
"""bench.py -- SpGEMM GFLOPS (2 x intermediate products / time) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload poisson27|poisson5|rmat|rmat_c5|rect] [--dtype f64|f32]
                    [--dump-outputs DIR]

A "step" is one full C = A*B: all four stages of bhsparse::spgemm
(SpGEMM_cuda/bhsparse.h:297-339) -- upper bound + binning, symbolic, row-pointer
scan + allocation, numeric -- from device-resident A, B to device-resident C,
the span the reference times (bhsparse.h:268-289).  Device buffers are grow-only
and cached by the context, so after the warm-up no cudaMalloc / memset sits in
the step (the reference's own timing includes them, bhsparse_cuda.h:285-301).

Headline (the JSON line's top level): BASELINE.json configs[1], Poisson 27-point
128^3, C = A^2, double.  At N>1 (weak scaling) the same stencil on a
128 x 128 x (128*N) grid.  A is split into N row blocks on the prefix sum of the
per-row products, B is broadcast with NCCL, every rank runs the single-GPU
pipeline on its block, one int64 all-gather of nnz(C) gives the offsets.

"rmat" sub-record (default run only): R-MAT scale 21 + log2(N), edge factor 16,
(.45,.15,.15,.25) -- scale 24 at N = 8 is BASELINE config 5 -- generated on rank
0's GPU (counter-based generator, identical in numpy), partitioned on the
product prefix sums, B broadcast over NCCL (timed, reported), per-rank times
min/max (= the load imbalance) reported.

Every run ends with an UNTIMED parity gate against the CPU oracle ("parity" in
the line): each rank checks its own row block entry for entry.

`--impl reference`: the reference has no CPU SpGEMM (ref_spgemm.h calls CUSP on
the device), so this arm times the CPU oracle (oracle/, a row-wise Gustavson
restatement, OpenMP over all host cores) on the same workload -- kind "port".
Where oracle/_ref (the reference's own CUDA code compiled for sm_100a) is
present its GPU time on the headline workload is reported beside it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "spgemm_gflops_2x_products_per_s"
UNIT = "GFLOPS"
VALUES = "integers 1..9 (fixed seed)"
RMAT_PARAMS = (0.45, 0.15, 0.15, 0.25)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def rmat_c5_scale(n_gpus: int) -> int:
    return 21 + int(np.log2(n_gpus))


def workload_desc(name: str, n_gpus: int) -> str:
    if name == "poisson27":
        return f"Poisson27pt 3D 128x128x{128 * n_gpus} C=A^2"
    if name == "poisson27thin":
        return f"Poisson27pt 3D 48x48x{1024 * n_gpus} C=A^2"
    if name == "poisson5":
        return f"Poisson5pt 2D 1024x{1024 * n_gpus} C=A^2"
    if name == "rmat":
        return f"R-MAT scale-{20 + int(np.log2(n_gpus))} ef16 (.45,.15,.15,.25) C=A^2"
    if name == "rmat_c5":
        return f"R-MAT scale-{rmat_c5_scale(n_gpus)} ef16 (.45,.15,.15,.25) counter-based generator C=A^2"
    if name == "rect":
        return f"uniform rect A({4194304 * n_gpus}x1M,8/row)*B(1Mx4M,8/row)"
    raise ValueError(name)


def make_workload(name: str, n_gpus: int, dtype):
    """Returns (A, B, a_equals_b) as host CSR (root only)."""
    from benchmark_spgemm_using_csr_b200 import generators as gen
    if name == "poisson27":
        A = gen.poisson27pt(128, 128, 128 * n_gpus, dtype=dtype)
        return A, A, True
    if name == "poisson27thin":          # same stencil, narrow column span (48 x 48 planes)
        A = gen.poisson27pt(48, 48, 1024 * n_gpus, dtype=dtype)
        return A, A, True
    if name == "poisson5":
        A = gen.poisson5pt(1024, 1024 * n_gpus, dtype=dtype)
        return A, A, True
    if name == "rmat":
        A = gen.rmat(20 + int(np.log2(n_gpus)), 16, dtype=dtype)
        return A, A, True
    if name == "rmat_c5":
        A = rmat_c5_host(n_gpus, dtype)
        return A, A, True
    if name == "rect":
        A = gen.uniform_rect(4194304 * n_gpus, 1048576, per_row=8, seed=1, dtype=dtype)
        B = gen.uniform_rect(1048576, 4194304, per_row=8, seed=2, value_seed=3, dtype=dtype)
        return A, B, False
    raise ValueError(name)


def rmat_c5_device(n_gpus: int, dtype, device):
    """Config-5 style R-MAT on a torch device: (rowptr, col, val) tensors."""
    import torch
    from benchmark_spgemm_using_csr_b200 import generators as gen
    a, b, c, d = RMAT_PARAMS
    td = torch.float64 if dtype == np.float64 else torch.float32
    return gen.rmat_counter_torch(rmat_c5_scale(n_gpus), 16, a, b, c, d, dtype=td, device=device)


def rmat_c5_host(n_gpus: int, dtype):
    """The same matrix on the host: through the GPU when there is one (scale 24 takes minutes in numpy)."""
    from benchmark_spgemm_using_csr_b200 import generators as gen
    try:
        import torch
        if torch.cuda.is_available():
            rp, col, val = rmat_c5_device(n_gpus, dtype, "cuda")
            n = rp.numel() - 1
            return gen.CSR(n, n, rp.cpu().numpy(), col.cpu().numpy(), val.cpu().numpy())
    except Exception:
        pass
    a, b, c, d = RMAT_PARAMS
    return gen.rmat_counter(rmat_c5_scale(n_gpus), 16, a, b, c, d, dtype=dtype)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "samples": len(sm), "reasons": sorted(reasons)}


DUMP_ENTRIES = 1 << 20      # sampled entries of a large C: 32 MB as float64, well within a 64 MB dump


def dump_outputs(out_dir, rowptr, col, val, seed=0):
    """Writes C = (rowptr, col, val), as a caller of the timed path receives it, to out_dir as .npy:
    rowptr, col, val in full when they fit in 32 MB, else the entries at a fixed seeded sample of
    positions: entry (position in col / val), row, col, val.  Indices are written as float64 (exact
    below 2^53), values in their own float32 / float64, so two builds can be compared file by file."""
    import torch
    rowptr, col, val = (torch.as_tensor(x) for x in (rowptr, col, val))
    if 8 * (rowptr.numel() + 2 * col.numel()) <= 32 * DUMP_ENTRIES:
        arrays = {"rowptr": rowptr, "col": col, "val": val}
    else:
        entry = np.sort(np.random.default_rng(seed).choice(col.numel(), DUMP_ENTRIES, replace=False))
        row = np.searchsorted(rowptr.cpu().numpy(), entry, side="right") - 1
        at = torch.from_numpy(entry).to(col.device)
        arrays = {"entry": entry, "row": row, "col": col[at], "val": val[at]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if torch.is_tensor(a) else a
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def config_dict(desc, m, nnzA, products, nnzC, world):
    """The `config` object: identical keys in both arms, so the driver can compare them."""
    return {"workload": desc, "values": VALUES, "m": int(m), "nnzA": int(nnzA), "products": int(products),
            "nnzC": int(nnzC), "l2": "inputs larger than L2 (no flush needed)",
            "partition": f"{world} row block(s) on the prefix sum of per-row products",
            "allocations": "device buffers are grow-only and cached: none inside the timed step after warm-up",
            "reuse": "per call everything is recomputed from the operands except two hints kept from the previous call on the "
                     "same operands: the diagonal-offset plan (every entry re-verified against it) and the column CDF that "
                     "balances the sort buckets (any table gives the same C)"}


# =================================================================================================
# reference arm: the CPU oracle on the host cores (+ the reference's own GPU code where built)
# =================================================================================================
def run_reference(args, rank):
    if rank != 0:
        return
    import oracle
    cores = os.cpu_count() or 1
    oracle.set_num_threads(cores)          # torchrun exports OMP_NUM_THREADS=1: ask for all cores explicitly
    dtype = np.float64 if args.dtype == "f64" else np.float32
    world = args.gpus
    desc = workload_desc(args.workload, world)
    A, B, _ = make_workload(args.workload, world, dtype)      # the SAME workload the repo arm runs at this N
    _, P = oracle.row_products(A.rows, A.rowptr, A.col, B.rowptr)
    times = []
    rp = None
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        rp, colC, valC = oracle.spgemm(A.rows, A.cols, B.cols, A.rowptr, A.col, A.val, B.rowptr, B.col, B.val)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
        if it == 0 and dt * (args.warmup + args.steps) > 240.0:
            break                                          # keep the arm within minutes: one step is the sample
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rp, colC, valC)
    t = float(np.mean(times)) if times else dt
    val = 2.0 * P / t / 1e9
    sample = f"full {desc} ({A.rows} rows, {P} products) per step, {len(times) or 1} timed step(s)"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": config_dict(desc, A.rows, A.nnz, P, int(rp[-1]), world),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": oracle.num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    # second stated baseline: the reference's own CUDA implementation (oracle/_ref) on this box's GPU 0
    if args.workload == "poisson27":
        line["reference_gpu"] = reference_gpu_time(A, B, P)
        # R-MAT sub-record: a bounded sample (row block 0 of the N-way partition) of the same matrix
        try:
            line["rmat"] = reference_rmat(world, dtype, cores)
        except Exception as e:       # never lose the headline line
            line["rmat"] = {"error": str(e)[:200]}
    print(json.dumps(line), flush=True)


def reference_gpu_time(A, B, P):
    """bhSPARSE's own kernels (compiled for sm_100a, oracle/_ref) on the headline workload, when it
    fits their int32 bookkeeping (Ct is over-allocated: the weak-scaled N>2 grids do not)."""
    try:
        from oracle import ref
        if not ref.available():
            return {"unavailable": "oracle/_ref not built"}
        if P > 2_000_000_000:
            return {"unavailable": "intermediate products exceed the reference's int32 Ct bookkeeping"}
        best = None
        for _ in range(3):
            _, _, _, ms = ref.spgemm(A.rows, A.cols, B.cols, A.rowptr, A.col, A.val, B.rowptr, B.col, B.val, fetch=False)
            best = ms if best is None else min(best, ms)
        return {"value": 2.0 * P / (best * 1e-3) / 1e9, "unit": UNIT, "ms": best, "kind": "reference (bhSPARSE CUDA, sm_100a build)",
                "note": "wall time of bhsparse::spgemm() incl. its allocations, best of 3; device-resident operands"}
    except Exception as e:
        return {"unavailable": str(e)[:200]}


def reference_rmat(world, dtype, cores):
    import oracle
    from benchmark_spgemm_using_csr_b200.dist import partition_rows_by_products, row_cost, row_products_host
    A = rmat_c5_host(world, dtype)
    prods = row_products_host(A, A.rowptr)
    bounds = partition_rows_by_products(row_cost(prods), world)      # the repo arm's partition
    blk = A.row_slice(0, int(bounds[1]))
    Pb = int(prods[:int(bounds[1])].sum())
    t0 = time.perf_counter()
    oracle.spgemm(blk.rows, blk.cols, A.cols, blk.rowptr, blk.col, blk.val, A.rowptr, A.col, A.val)
    dt = time.perf_counter() - t0
    return {"value": 2.0 * Pb / dt / 1e9, "unit": UNIT, "ms": dt * 1e3, "cores": cores, "kind": "port",
            "workload": workload_desc("rmat_c5", world), "products": int(prods.sum()),
            "sample": f"row block 0 of the {world}-way partition the repo arm uses ({blk.rows} rows, {Pb} products), one run"}


# =================================================================================================
# repo arm
# =================================================================================================
class Run:
    """One process = one GPU.  Everything timed runs on ONE explicit non-default stream: the
    library's kernels, the CUDA events and the NCCL collectives."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a B200: there is no CPU fallback for the product path")
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        self.stream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.stream)
        assert self.stream.cuda_stream != 0

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def allreduce(self, values, op="max", dtype=None):
        torch, dist = self.torch, self.dist
        t = torch.tensor(values, dtype=dtype or torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op={"max": dist.ReduceOp.MAX, "min": dist.ReduceOp.MIN, "sum": dist.ReduceOp.SUM}[op])
        return t.cpu().tolist()

    def new_engine(self, square=True):
        """square (C = B*B): partition, NCCL broadcast and offsets run INSIDE the library
        (bhb200_dist_*, csrc/dist_nccl.cu); otherwise the torch.distributed harness of dist.py."""
        from benchmark_spgemm_using_csr_b200.dist import CudaEngine, NcclRowBlockSpGEMM, RowBlockSpGEMM
        engine = CudaEngine(self.local_rank)
        engine.use_stream(self.stream.cuda_stream)
        return engine, (NcclRowBlockSpGEMM(engine, self.dev) if square else RowBlockSpGEMM(engine, self.dev))

    def upload(self, A):
        """Host CSR -> (rowptr, col, val) tensors on this rank's device (setup, untimed)."""
        torch = self.torch
        return tuple(torch.from_numpy(np.ascontiguousarray(x)).to(self.dev) for x in (A.rowptr, A.col, A.val))


def timed_steps(run: Run, rb, engine, steps, warmup, sample_clocks):
    torch = run.torch
    for _ in range(warmup):
        rb.spgemm()
    run.barrier()
    sampler = ClockSampler(run.local_rank) if (sample_clocks and run.rank == 0) else None
    if sampler:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    run.barrier()
    wall0 = time.perf_counter()
    ev0.record(run.stream)
    for _ in range(steps):
        nnz_local, off, nnz_total = rb.spgemm()
    ev1.record(run.stream)
    if nnz_total is None:                   # C-ABI path: offsets and totals stay on the device during the steps
        _, _, off, nnz_total = rb.layout()
    run.barrier()
    wall_ms = (time.perf_counter() - wall0) * 1e3 / steps
    ms_local = ev0.elapsed_time(ev1) / steps
    # the step has host syncs inside, so device time and wall clock must agree
    if abs(ms_local - wall_ms) > 0.05 * wall_ms + 0.05:
        raise SystemExit(f"timing inconsistency: CUDA events {ms_local:.3f} ms/step vs wall clock {wall_ms:.3f} ms/step")
    clocks = sampler.stop() if sampler else None
    st = engine.stats()
    ms = run.allreduce([ms_local], "max")[0]
    ms_min = run.allreduce([ms_local], "min")[0]
    pipe = run.allreduce([st["ms_total"]], "max")[0], run.allreduce([st["ms_total"]], "min")[0]
    launches = int(run.allreduce([st["kernel_launches"] * steps], "sum")[0])
    return dict(ms=ms, ms_min_rank=ms_min, wall_ms=wall_ms, clocks=clocks, st=st, launches=launches,
                nnz_local=int(nnz_local), nnz_total=int(nnz_total), offset=int(off),
                pipeline_ms_max_rank=pipe[0], pipeline_ms_min_rank=pipe[1])


def parity_gate(run: Run, rb, engine, budget_products: float):
    """UNTIMED.  Every rank compares its own row block of C with the CPU oracle run on the same
    block: row pointers (local + all-gathered offset), column indices, values.  Blocks of rows are
    checked one after another (bounded host memory); with a product budget only every other /
    every k-th block is checked and the line says how many rows that was."""
    import oracle
    from benchmark_spgemm_using_csr_b200.generators import CSR
    oracle.set_num_threads(max(1, (os.cpu_count() or 1) // run.world))
    Arp, Ac, Av = (t.cpu().numpy() for t in rb.A)
    Brp, Bc, Bv = (t.cpu().numpy() for t in rb.B)
    m_loc = Arp.size - 1
    A = CSR(m_loc, rb.meta["k"], Arp, Ac, Av)
    k, n = rb.meta["k"], rb.meta["n"]
    rp64 = engine.rowptr64_host()
    prods, total = oracle.row_products(m_loc, Arp, Ac, Brp)
    nblk = max(1, min(64, int(np.ceil(total / 6.0e7))))
    bounds = np.linspace(0, m_loc, nblk + 1).astype(np.int64)
    stride = max(1, int(np.ceil(total / max(budget_products, 1.0))))
    ok_rp = ok_col = True
    max_rel = 0.0
    rows_checked = 0
    for b in range(0, nblk, stride):
        r0, r1 = int(bounds[b]), int(bounds[b + 1])
        if r1 <= r0:
            continue
        blk = A.row_slice(r0, r1)
        wrp, wcol, wval = oracle.spgemm(blk.rows, k, n, blk.rowptr, blk.col, blk.val, Brp, Bc, Bv)
        ok_rp &= bool(np.array_equal(rp64[r0:r1 + 1] - rp64[r0], wrp))
        cnt = int(rp64[r1] - rp64[r0])
        col, val = engine.get_C_range(int(rp64[r0]), cnt)
        same = cnt == wcol.size and bool(np.array_equal(col, wcol))
        ok_col &= same
        if same and cnt:
            rel = np.abs(val.astype(np.float64) - wval.astype(np.float64)) / np.maximum(np.abs(wval.astype(np.float64)), 1e-300)
            max_rel = max(max_rel, float(rel.max()))
        rows_checked += r1 - r0
    ok_rp &= bool(rp64[0] == 0 and rp64[-1] == engine.lib.bhb200_get_nnzC(engine.ctx))
    flags = run.allreduce([1.0 if ok_rp else 0.0, 1.0 if ok_col else 0.0], "min")
    rel = run.allreduce([max_rel], "max")[0]
    rows = run.allreduce([float(rows_checked), float(m_loc)], "sum")
    return {"rowptr": bool(flags[0]), "col": bool(flags[1]), "max_rel": rel, "rows_checked": int(rows[0]),
            "rows": int(rows[1]), "ranks": run.world, "against": "CPU oracle on each rank's own row block (untimed)"}


def e2e_leg(run: Run, rb, hostA, hostB, aeqb, steps):
    """The same metric through the public API with HOST buffers, copies inside the timed region.
    N = 1: the reference-facing class, bhsparse.initData + spgemm + get_nnzC + get_C (main.cu:104-135).
    N > 1: RowBlockSpGEMM from rank 0's host arrays: H2D of B on rank 0, NCCL broadcast, every
    rank slices / receives its block of A, runs its pipeline and copies its block of C to host."""
    torch, dist = run.torch, run.dist
    from benchmark_spgemm_using_csr_b200 import BHSPARSE_CUDA, NUM_PLATFORMS, bhsparse
    meta = rb.meta
    vsz = 8 if run.args.dtype == "f64" else 4
    e_steps = max(3, min(steps, 5))
    if run.world == 1:
        a_rp, a_c, a_v = (torch.from_numpy(x).pin_memory() for x in (hostA.rowptr, hostA.col, hostA.val))
        if aeqb:
            b_rp, b_c, b_v = a_rp, a_c, a_v            # C = A^2: the caller passes the same arrays twice (main.cu:32-33)
        else:
            b_rp, b_c, b_v = (torch.from_numpy(x).pin_memory() for x in (hostB.rowptr, hostB.col, hostB.val))
        nnzC = int(meta.get("nnzC_known", 0)) or None
        rowptrC = torch.empty(hostA.rows + 1, dtype=torch.int32).pin_memory()
        platforms = [False] * NUM_PLATFORMS
        platforms[BHSPARSE_CUDA] = True
        bh = bhsparse(run.local_rank)
        assert bh.initPlatform(platforms) == 0
        bufs = {}

        def step():
            err = bh.initData(hostA.rows, meta["k"], meta["n"], a_c.numel(), a_v.numpy(), a_rp.numpy(), a_c.numpy(),
                              b_c.numel(), b_v.numpy(), b_rp.numpy(), b_c.numpy(), rowptrC.numpy())
            err |= bh.spgemm()
            n = bh.get_nnzC()
            if "col" not in bufs or bufs["col"].numel() < n:      # (first step only: pinned result buffers)
                bufs["col"] = torch.empty(max(n, 1), dtype=torch.int32).pin_memory()
                bufs["val"] = torch.empty(max(n, 1), dtype=a_v.dtype).pin_memory()
            err |= bh.get_C(bufs["col"].numpy()[:n], bufs["val"].numpy()[:n])
            assert err == 0, bh.last_error()
            return n

        for _ in range(2):
            n = step()
        torch.cuda.synchronize(run.dev)
        t0 = time.perf_counter()
        for _ in range(e_steps):
            n = step()
        torch.cuda.synchronize(run.dev)
        e_ms = (time.perf_counter() - t0) * 1e3 / e_steps
        uploaded = [a_rp, a_c, a_v] + ([] if aeqb and bh.aliased_operands() else [b_rp, b_c, b_v])
        h2d = sum(t.numel() * t.element_size() for t in uploaded)
        d2h = 2 * rowptrC.numel() * 4 + n * (4 + vsz)              # rowptrC after spgemm() and in get_C, as the reference
        api = "bhsparse.initData + spgemm + get_nnzC + get_C, pinned host buffers"
        bh.free_mem()
        bh.freePlatform()
    else:
        engine, rb2 = run.new_engine()
        pinned = None
        if run.rank == 0:
            pinned = tuple(torch.from_numpy(x).pin_memory() for x in (hostB.rowptr, hostB.col, hostB.val))
        out = {}

        def step():
            Bdev = tuple(t.to(run.dev, non_blocking=True) for t in pinned) if run.rank == 0 else None
            rb2.setup_square_from_device_root(Bdev, meta["n"])
            nnz_local, off, total = rb2.spgemm()
            res = engine.result()
            for key, t in (("rp", res.rowptr64), ("col", res.col), ("val", res.val)):
                if key not in out or out[key].numel() < t.numel():
                    out[key] = torch.empty(max(t.numel(), 1), dtype=t.dtype).pin_memory()
                out[key][:t.numel()].copy_(t, non_blocking=True)
            torch.cuda.synchronize(run.dev)
            return nnz_local

        assert aeqb, "multi-GPU e2e leg: C = A^2 workloads"
        for _ in range(2):
            n = step()
        run.barrier()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            n = step()
        run.barrier()
        e_ms = run.allreduce([(time.perf_counter() - t0) * 1e3 / e_steps], "max")[0]
        h2d_local = sum(t.numel() * t.element_size() for t in pinned) if run.rank == 0 else 0
        m_loc = rb2.A[0].numel() - 1
        sums = run.allreduce([float(h2d_local), float((m_loc + 1) * 8 + n * (4 + vsz))], "sum")
        h2d, d2h = int(sums[0]), int(sums[1])
        api = ("RowBlockSpGEMM: H2D of B on rank 0 + NCCL broadcast + per-rank pipeline + D2H of every rank's block of C, "
               "pinned host buffers")
        engine.close()
    return {"value": 2.0 * meta["products"] / (e_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": e_ms,
            "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "api": api}


def roofline_of(args, st, bin_ms_sym, bin_ms_num, vsz, world):
    from benchmark_spgemm_using_csr_b200.capi import NUM_BIN_NAMES, SYM_BIN_NAMES
    peak, peak_src = peaks()

    # Algorithmic bytes of a launch = stream-gather model (SURVEY.md 8d) restricted to its rows:
    # read the A rows + two rowptrB words per A entry + one (col,val) of B per product + write the C rows.
    def alg_bytes(bin_idx):
        return (st["num_bin_rows"][bin_idx] * 8 + st["num_bin_nnzA"][bin_idx] * (4 + vsz) + st["num_bin_nnzA"][bin_idx] * 8 +
                st["num_bin_products"][bin_idx] * (4 + vsz) + st["num_bin_nnzC"][bin_idx] * (4 + vsz))
    pattern = bool(st.get("pattern_mode"))
    direct_bins = [i for i in range(len(SYM_BIN_NAMES)) if (st["direct_bin_mask"] >> i) & 1]
    direct_ms = float(sum(bin_ms_sym[i] for i in direct_bins))
    copy_idx = NUM_BIN_NAMES.index("copy_ct")
    num_ms = bin_ms_num.copy()
    num_ms[copy_idx] = 0.0
    b = int(np.argmax(num_ms))
    if pattern:
        # diagonal-pattern mode: ONE numeric kernel does every product of the step (stage 4)
        kname = (f"k_pat_numeric (diagonal-pattern mode: {st['pattern_nDA']} x {st['pattern_nDB']} -> "
                 f"{st['pattern_nD']} diagonals)")
        rows_b, bytes_b, t_b, tkey = int(st["m"]), st["bytes_algorithmic"], st["ms_numeric"] * 1e-3, "pattern"
    elif direct_ms > num_ms[b]:
        kname = "k_num_direct (direct mode, symbolic bins " + ",".join(SYM_BIN_NAMES[i] for i in direct_bins) + ")"
        rows_b, bytes_b, t_b, tkey = st["num_bin_rows"][copy_idx], alg_bytes(copy_idx), direct_ms * 1e-3, "direct"
    else:
        kname = f"k_num_* bin {NUM_BIN_NAMES[b]}"
        rows_b, bytes_b, t_b, tkey = st["num_bin_rows"][b], alg_bytes(b), num_ms[b] * 1e-3, "num_" + NUM_BIN_NAMES[b]
    achieved = bytes_b / t_b / 1e9 if t_b > 0 else 0.0
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp) and world == 1:
        try:
            tj = json.load(open(tp))
            ent = tj.get(f"{args.workload}_{args.dtype}_{tkey}")
            if isinstance(ent, dict):
                traffic, traffic_src = ent.get("bytes"), ent.get("source")
            else:
                traffic = ent
        except Exception:
            traffic = None
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
            "kernel": f"{kname} ({rows_b} rows)", "kernel_ms": t_b * 1e3,
            "algorithmic_bytes": int(bytes_b), "peak_source": peak_src}


def per_bin_times(engine, rb, reps=3):
    from benchmark_spgemm_using_csr_b200.capi import NUM_BINS
    sym, num = np.zeros(NUM_BINS), np.zeros(NUM_BINS)
    for _ in range(reps):
        rb.spgemm()
        s2 = engine.stats()
        sym += np.array(s2["ms_sym_bin"])
        num += np.array(s2["ms_num_bin"])
    return sym / reps, num / reps


def rmat_record(run: Run, args):
    """Config-5 style R-MAT at scale 21 + log2(N): generated on rank 0's GPU, product-balanced row
    blocks, B broadcast over NCCL (timed), per-rank pipeline times min/max = the load imbalance."""
    torch = run.torch
    np_dtype = np.float64 if args.dtype == "f64" else np.float32
    world = run.world
    t0 = time.perf_counter()
    Bdev = rmat_c5_device(world, np_dtype, run.dev) if run.rank == 0 else None
    torch.cuda.synchronize(run.dev)
    gen_s = time.perf_counter() - t0
    engine, rb = run.new_engine()
    n = 1 << rmat_c5_scale(world)
    rb.setup_square_from_device_root(Bdev, n)
    del Bdev
    meta = rb.meta
    steps = max(3, min(args.steps, 5))
    t = timed_steps(run, rb, engine, steps, 3, sample_clocks=False)
    st = t["st"]
    vsz = 8 if args.dtype == "f64" else 4
    peak, _ = peaks()
    m1 = meta["m"] + 1
    alg = (m1 * 4 + meta["nnzA"] * (4 + vsz)) + (meta["nnzA"] * 8 + meta["products"] * (4 + vsz)) + (m1 * 4 + t["nnz_total"] * (4 + vsz))
    parity = parity_gate(run, rb, engine, budget_products=2.5e8)
    bp = meta.get("block_products", [meta["products"]])
    rec = {
        "workload": workload_desc("rmat_c5", world), "value": 2.0 * meta["products"] / (t["ms"] * 1e-3) / 1e9, "unit": UNIT,
        "ms_per_step": t["ms"], "steps": steps, "warmup": 3, "m": meta["m"], "nnzA": meta["nnzA"], "products": meta["products"],
        "nnzC": t["nnz_total"], "max_row_products": meta.get("max_row_products"),
        "rank_ms": {"max": t["pipeline_ms_max_rank"], "min": t["pipeline_ms_min_rank"],
                    "imbalance": t["pipeline_ms_max_rank"] / max(t["pipeline_ms_min_rank"], 1e-9)},
        "block_products": {"max": int(max(bp)), "min": int(min(bp))},
        "broadcast_B_ms": rb.timings.get("broadcast_B_s", 0.0) * 1e3,
        "broadcast_B_bytes": int(meta["nnzB"]) * (4 + vsz) + (meta["k"] + 1) * 4,
        "generate_s": gen_s,
        "roofline_step": {"algorithmic_bytes": int(alg), "frac": alg / (t["ms"] * 1e-3) / 1e9 / (peak * world),
                          "note": "stream-gather model over all ranks / (N x measured HBM peak)"},
        "stages_ms_rank0": {"count_bin": st["ms_count"], "symbolic": st["ms_symbolic"], "scan_alloc": st["ms_scan"],
                            "numeric": st["ms_numeric"], "total": st["ms_total"]},
        "parity": parity,
    }
    engine.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="poisson27",
                    choices=["poisson27", "poisson27thin", "poisson5", "rmat", "rmat_c5", "rect"])
    ap.add_argument("--dtype", default=None, choices=["f64", "f32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-rmat", action="store_true", help="skip the R-MAT sub-record of the default run")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write C of the last timed step to DIR/<name>.npy (one process, --gpus 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.gpus != 1:
        ap.error("--dump-outputs writes one process's C: use it with --gpus 1")
    if args.dtype is None:
        args.dtype = "f32" if args.workload == "rect" else "f64"
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")))
        return

    run = Run(args)
    torch, dist = run.torch, run.dist
    rank, world = run.rank, run.world
    np_dtype = np.float64 if args.dtype == "f64" else np.float32
    vsz = 8 if args.dtype == "f64" else 4

    # ---- setup (untimed): generate on rank 0, partition, broadcast B over NCCL ----
    A = B = None
    aeqb = args.workload != "rect"
    desc = workload_desc(args.workload, world)
    if rank == 0:
        A, B, aeqb = make_workload(args.workload, world, np_dtype)
    engine, rb = run.new_engine(square=aeqb)
    if aeqb:
        rb.setup_square_from_device_root(run.upload(B) if rank == 0 else None)
    else:
        rb.setup_from_root(A, B, root=0, a_equals_b=False)
    meta = rb.meta
    P_total = meta["products"]
    engine.set_profiling(True)

    t = timed_steps(run, rb, engine, args.steps, args.warmup, sample_clocks=True)
    if args.dump_outputs:
        res = engine.result()
        dump_outputs(args.dump_outputs, res.rowptr64, res.col, res.val)
        del res
    ms, st = t["ms"], t["st"]
    value = 2.0 * P_total / (ms * 1e-3) / 1e9
    bin_ms_sym, bin_ms_num = per_bin_times(engine, rb)       # same launches, per-bin events (profiling stays on)

    parity = None if args.no_parity else parity_gate(run, rb, engine, budget_products=float("inf"))
    e2e = None if args.no_e2e else e2e_leg(run, rb, A, B, aeqb, args.steps)
    setup_bcast_ms = rb.timings.get("broadcast_B_s", 0.0) * 1e3
    rmat = None
    if args.workload == "poisson27" and not args.no_rmat:
        engine.close()                                        # free the headline's device memory first
        rb = None
        torch.cuda.empty_cache()
        try:
            rmat = rmat_record(run, args)
        except Exception as e:                                # never lose the headline line
            rmat = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    from benchmark_spgemm_using_csr_b200.capi import NUM_BIN_NAMES, SYM_BIN_NAMES
    peak, _ = peaks()
    roofline = roofline_of(args, st, bin_ms_sym, bin_ms_num, vsz, world)
    step_alg = st["bytes_algorithmic"] if world == 1 else None
    roof_step = None
    if step_alg:
        roof_step = {"algorithmic_bytes": int(step_alg), "achieved": step_alg / (ms * 1e-3) / 1e9,
                     "frac": step_alg / (ms * 1e-3) / 1e9 / peak,
                     "compulsory_bytes": int(st["bytes_compulsory"]),
                     "frac_compulsory": st["bytes_compulsory"] / (ms * 1e-3) / 1e9 / peak}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        import oracle
        oracle.set_num_threads(os.cpu_count() or 1)
        t_best = None
        for _ in range(2):
            t0 = time.perf_counter()
            oracle.spgemm(A.rows, A.cols, B.cols, A.rowptr, A.col, A.val, B.rowptr, B.col, B.val)
            dt = time.perf_counter() - t0
            t_best = dt if t_best is None else min(t_best, dt)
        cpu = {"value": 2.0 * P_total / t_best / 1e9, "unit": UNIT, "cores": oracle.num_threads(), "kind": "port",
               "sample": f"full workload ({A.rows} rows, {P_total} products), best of 2, {t_best:.3f} s",
               # second stated baseline: the reference's own CUDA implementation (oracle/_ref) on this GPU
               "reference_gpu": reference_gpu_time(A, B, P_total)}

    cfg = config_dict(desc, meta["m"], meta["nnzA"], P_total, t["nnz_total"], world)     # same keys and values as the reference arm's
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "wall_ms_per_step": t["wall_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic", "config": cfg,
        "roofline": roofline, "roofline_step": roof_step, "cpu_baseline": cpu, "e2e": e2e, "parity": parity,
        "gpu_launches": t["launches"], "clocks": t["clocks"], "nnzC_rank0": t["nnz_local"],
        "rank_ms": {"max": ms, "min": t["ms_min_rank"]},
        # each rank's own pipeline (its CUDA events inside the library, last step): a step ends in an all-gather, so the
        # step time follows the slowest rank
        "pipeline_ms": {"max_rank": t["pipeline_ms_max_rank"], "min_rank": t["pipeline_ms_min_rank"]},
        "stages_ms": {"count_bin": st["ms_count"], "symbolic": st["ms_symbolic"], "scan_alloc": st["ms_scan"],
                      "numeric": st["ms_numeric"], "total": st["ms_total"]},
        "bins_ms": {"symbolic": {SYM_BIN_NAMES[i]: round(float(bin_ms_sym[i]), 4) for i in range(len(SYM_BIN_NAMES)) if bin_ms_sym[i] > 0},
                    "numeric": {NUM_BIN_NAMES[i]: round(float(bin_ms_num[i]), 4) for i in range(len(NUM_BIN_NAMES)) if bin_ms_num[i] > 0}},
        "direct_mode": {"rows": st["direct_rows"], "retry_rows": st["direct_retry_rows"], "staging_bytes": st["direct_ct_bytes"]},
        "pattern_mode": {"on": bool(st.get("pattern_mode")), "diagonals_A": st.get("pattern_nDA"), "diagonals_B": st.get("pattern_nDB"),
                         "diagonals_C": st.get("pattern_nD")},
        "setup_broadcast_ms": setup_bcast_ms,
        "rmat": rmat,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
