"""Structure-only products (BHB200_DTYPE_NONE) against the valued product on the same operands.

    python tools/structure_probe.py [--calls 10] [--out profiles/r03_structure_probe.jsonl] [--small]

Per workload one JSON record (device name and power limit read in the same run), borrowed device operands (the
structure-only context gets NULL value pointers), median of --calls products after two warm-up calls each, valued
and structure-only calls alternating:
  valued / structure   ms_total, ms_count, ms_symbolic, ms_scan, ms_numeric, products, nnzC, kernel launches,
                       pattern mode, direct-mode bins, workspace_bytes (device memory held by the context)
  identical            rowptrC and colC of the two products are equal
  speedup              valued ms_total / structure ms_total
Workloads:
  27pt_128^3           A*A, f64 (diagonal-pattern mode: k_pat_numeric against k_pat_emit)
  rmat_s21             A*A, R-MAT scale 21, edge factor 16 (.45, .15, .15, .25), f64: the operand of bench.py's
                       R-MAT sub-record (counter-based generator; bucket-sort and heavy bins)
  uniform_rect_4M_1M   A(4M x 1M) * B(1M x 4M), 8 per row, f32 (warp-per-row bucket sort)
  triangles_rmat_s20   (L*L) .* L, L = strictly lower triangle of the symmetrized R-MAT scale 20, f64
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
from probe_util import COUNTERS, lower_triangle, read_power_limit, run, summary  # noqa: E402


def context(m, k, n, A, B, M, structure):
    """A capi.Context on borrowed device operands; structure-only ones get NULL value pointers."""
    c = capi.Context()
    if structure:
        c.init_device((*A[:2], None), (*B[:2], None), m, k, n, dtype=capi.DTYPE_NONE)
    else:
        c.init_device(A, B, m, k, n)
    if M is not None:
        c.set_mask_device(*M)
    return c


def probe(torch, name, m, k, n, A, B, M, calls):
    valued, structure = context(m, k, n, A, B, M, False), context(m, k, n, A, B, M, True)
    for e in (valued, structure):   # warm-up
        run(e)
        run(e)
    rec_v, rec_s = [], []
    for _ in range(calls):
        rec_v.append(run(valued))
        rec_s.append(run(structure))
    cv, cs = valued.C_device(), structure.C_device()
    counters = COUNTERS + ("direct_bin_mask", "workspace_bytes")
    sv, ss = summary(rec_v, counters=counters), summary(rec_s, counters=counters)
    rec = {"workload": name, "m": m, "k": k, "n": n, "dtype": str(A[2].dtype).replace("torch.", ""), "calls": calls,
           "valued": sv, "structure": ss,
           "identical": bool(torch.equal(cv[0], cs[0]) and torch.equal(cv[1], cs[1])),
           "speedup": sv["ms_total"] / ss["ms_total"] if ss["ms_total"] > 0 else None}
    valued.close()
    structure.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("structure_probe: no CUDA device (there is no CPU path)")
    device = torch.cuda.get_device_name(0)
    plim = read_power_limit()
    dev = lambda *a: tuple(torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in a)
    nx, scale, rect_rows, rect_cols, tscale = (16, 12, 1 << 14, 1 << 12, 12) if args.small else (128, 21, 1 << 22, 1 << 20, 20)
    out = open(args.out, "w") if args.out else None

    def emit(rec):
        rec.update({"device": device, "power_limit": plim})
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    A = gen.poisson27pt(nx, nx, nx)
    Ad = dev(A.rowptr, A.col, A.val)
    emit(probe(torch, f"27pt_{nx}^3", A.rows, A.cols, A.cols, Ad, Ad, None, args.calls))
    del A, Ad
    torch.cuda.empty_cache()   # (the library allocates with cudaMalloc, outside torch's cache)

    Ad = gen.rmat_counter_torch(scale, 16, dtype=torch.float64, device="cuda")
    rows = Ad[0].numel() - 1
    torch.cuda.empty_cache()
    emit(probe(torch, f"rmat_s{scale}", rows, rows, rows, Ad, Ad, None, args.calls))
    del Ad
    torch.cuda.empty_cache()

    A = gen.uniform_rect(rect_rows, rect_cols, per_row=8, seed=1, dtype=np.float32)
    B = gen.uniform_rect(rect_cols, rect_rows, per_row=8, seed=2, value_seed=3, dtype=np.float32)
    Ad, Bd = dev(A.rowptr, A.col, A.val), dev(B.rowptr, B.col, B.val)
    emit(probe(torch, "uniform_rect_16k_4k" if args.small else "uniform_rect_4M_1M", A.rows, A.cols, B.cols, Ad, Bd, None,
               args.calls))
    del A, B, Ad, Bd
    torch.cuda.empty_cache()

    L = lower_triangle(tscale)
    Ld = dev(L.indptr.astype(np.int32), L.indices.astype(np.int32), L.data)
    n = L.shape[0]
    emit(probe(torch, f"triangles_rmat_s{tscale}", n, n, n, Ld, Ld, Ld[:2], args.calls))
    if out:
        out.close()


if __name__ == "__main__":
    main()
