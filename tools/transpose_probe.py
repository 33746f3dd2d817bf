"""Cost of the device transpose of op(X) = X^T (csrc/stage_transpose.cu) on product-sized operands.

    python tools/transpose_probe.py [--calls 10] [--out profiles/transpose_probe.jsonl] [--small]

Per workload one JSON record (device name and power limit read in the same run):
  ms_transpose   median over --calls products on borrowed device operands (transposed on every call)
  ms_copy_d2d    median time of cudaMemcpyAsync (torch copy_) of the same operand's rowptr, col and val
  ms_op_path     median ms_total of the product with the transpose flag (transposition included)
  ms_pretransposed  median ms_total of the same product on operands transposed on the host beforehand
                 (calls of the two paths alternate)
  same_structure rowptr and col of C equal between the two paths
Workloads: 27-pt 128^3 f64 A*A^T (nonsymmetric values), R-MAT scale 20 A*A^T, uniform_rect(4M, 1M) A^T*A.
--small runs the same workloads at toy sizes (a rehearsal of the script, not a measurement).
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from benchmark_spgemm_using_csr_b200 import capi, generators as gen  # noqa: E402
from probe_util import read_power_limit, run  # noqa: E402


def copy_ms(torch, X, calls):
    """D2D copies of rowptr, col and val (torch copy_ = cudaMemcpyAsync), CUDA events."""
    src = X
    dst = [torch.empty_like(t) for t in src]
    times = []
    for _ in range(calls + 2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for d, s in zip(dst, src):
            d.copy_(s)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times[2:]))


def probe(torch, name, X, mode, calls):
    """mode 'NT': X*X^T, 'TN': X^T*X (X stored)."""
    dev = torch.device("cuda")
    t = lambda C: [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (C.rowptr, C.col, C.val)]
    XT = gen.transpose(X)
    tX, tXT = t(X), t(XT)
    N, T = capi.OP_N, capi.OP_T
    if mode == "NT":
        dims = (X.rows, X.cols, X.rows)
        op_args = (tX, tX, *dims, N, T)
        pre_args = (tX, tXT, *dims, N, N)
    else:
        dims = (X.cols, X.rows, X.cols)
        op_args = (tX, tX, *dims, T, N)
        pre_args = (tXT, tX, *dims, N, N)
    e_op, e_pre = capi.Context(), capi.Context()
    e_op.init_device(*op_args)
    e_pre.init_device(*pre_args)
    for e in (e_op, e_pre):   # warm-up
        run(e)
        run(e)
    ms_t, ms_op, ms_pre, launches = [], [], [], 0
    for _ in range(calls):
        st = run(e_op)
        ms_t.append(st["ms_transpose"])
        ms_op.append(st["ms_total"])
        launches = st["kernel_launches"]
        st = run(e_pre)
        ms_pre.append(st["ms_total"])
    a, b = e_op.C(), e_pre.C()
    same = bool(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]))
    rec = {
        "workload": name, "product": "A*A^T" if mode == "NT" else "A^T*A", "rows": X.rows, "cols": X.cols, "nnz": X.nnz,
        "dtype": str(X.val.dtype), "calls": calls,
        "ms_transpose": float(np.median(ms_t)), "ms_copy_d2d": copy_ms(torch, tX, calls),
        "ms_op_path": float(np.median(ms_op)), "ms_pretransposed": float(np.median(ms_pre)),
        "op_path_kernel_launches": launches, "nnzC": int(a[1].size), "same_structure": same,
    }
    e_op.close()
    e_pre.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("transpose_probe: no CUDA device (there is no CPU path)")
    device = torch.cuda.get_device_name(0)
    plim = read_power_limit()
    if args.small:
        work = [("27pt_16^3", gen.poisson27pt(16, 16, 16), "NT"), ("rmat_s12", gen.rmat(12, 16), "NT"),
                ("uniform_rect_4k_1k", gen.uniform_rect(4096, 1024), "TN")]
    else:
        work = [("27pt_128^3", gen.poisson27pt(128, 128, 128), "NT"), ("rmat_s20", gen.rmat(20, 16), "NT"),
                ("uniform_rect_4M_1M", gen.uniform_rect(1 << 22, 1 << 20), "TN")]
    out = open(args.out, "w") if args.out else None
    for name, X, mode in work:
        rec = probe(torch, name, X, mode, args.calls)
        rec.update({"device": device, "power_limit": plim})
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()
        del X
    if out:
        out.close()


if __name__ == "__main__":
    main()
