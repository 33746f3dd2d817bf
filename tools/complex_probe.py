"""complex64 products against f64 and f32 on the same operands.

    python tools/complex_probe.py [--calls 10] [--out profiles/r03_complex_probe.jsonl] [--small]

Per workload one JSON record (device name and power limit read in the same run).  The operands are borrowed device
arrays with one structure and three value arrays: f64, the same values in f32, and complex64 (re = the f32 values,
im = half of them).  Each type has its own context; after two warm-up calls per type the types alternate, and every
field is the median of --calls products:
  c64 / f64 / f32   ms_total, ms_count, ms_symbolic, ms_scan, ms_numeric, ms_transpose, products, nnzC, kernel
                    launches, pattern mode, direct-mode bins, workspace_bytes (device memory held by the context)
  bins              per-bin kernel times of c64 and f64 (ms_sym_bin / ms_num_bin, bhb200_set_profiling) from a
                    second, profiled pass of --calls products each: which kernel accounts for a gap
  c64_over_f64      c64 ms_total / f64 ms_total (and the same for f32)
Workloads:
  27pt_128^3           A*A (diagonal-pattern mode)
  rmat_s21             A*A, R-MAT scale 21, edge factor 16 (.45, .15, .15, .25): the operand of bench.py's R-MAT
                       sub-record (bucket-sort and heavy bins)
  uniform_rect_4M_1M   A(4M x 1M) * B(1M x 4M), 8 per row (warp-per-row bucket sort)
  triangles_rmat_s20   (L*L) .* L, L = strictly lower triangle of the symmetrized R-MAT scale 20 (masked kernels)
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
from probe_util import COUNTERS, STAGES, lower_triangle, read_power_limit, run, summary  # noqa: E402

TYPES = ("c64", "f64", "f32")


def bin_times(sts):
    """median per-bin kernel times (ms), bins that ran only"""
    out = {}
    for key in ("ms_sym_bin", "ms_num_bin"):
        med = np.median([s[key] for s in sts], axis=0)
        out[key] = {str(b): round(float(t), 4) for b, t in enumerate(med) if t > 0}
    return out


def probe(torch, name, m, k, n, A, B, M, calls):
    """A, B: {type: (rowptr, col, val)} on the device"""
    eng = {t: capi.Context() for t in TYPES}
    for t, e in eng.items():
        e.init_device(A[t], B[t], m, k, n)
        if M is not None:
            e.set_mask_device(*M)
        run(e)
        run(e)
    rec = {t: [] for t in eng}
    for _ in range(calls):
        for t, e in eng.items():
            rec[t].append(run(e))
    prof = {}
    for t in ("c64", "f64"):
        eng[t].set_profiling(True)
        run(eng[t])
        prof[t] = bin_times([run(eng[t]) for _ in range(calls)])
    for e in eng.values():
        e.close()
    out = {"workload": name, "m": m, "k": k, "n": n, "calls": calls}
    counters = COUNTERS + ("direct_bin_mask", "workspace_bytes")
    out.update({t: summary(v, STAGES + ("ms_transpose",), counters) for t, v in rec.items()})
    out["bins"] = prof
    for t in ("f64", "f32"):
        out[f"c64_over_{t}"] = out["c64"]["ms_total"] / out[t]["ms_total"] if out[t]["ms_total"] > 0 else None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("complex_probe: no CUDA device (there is no CPU path)")
    device = torch.cuda.get_device_name(0)
    plim = read_power_limit()
    nx, scale, rect_rows, rect_cols, tscale = (16, 12, 1 << 14, 1 << 12, 12) if args.small else (128, 21, 1 << 22, 1 << 20, 20)
    out = open(args.out, "w") if args.out else None

    def emit(rec):
        rec.update({"device": device, "power_limit": plim})
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    def typed(rp, col, v64):
        """{type: (rowptr, col, val)} sharing rowptr and col"""
        v32 = v64.to(torch.float32)
        return {"f64": (rp, col, v64), "f32": (rp, col, v32), "c64": (rp, col, torch.complex(v32, 0.5 * v32))}

    def host(X):
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        return typed(t(X.rowptr), t(X.col), t(X.val.astype(np.float64)))

    A = host(gen.poisson27pt(nx, nx, nx))
    rows = A["f64"][0].numel() - 1
    emit(probe(torch, f"27pt_{nx}^3", rows, rows, rows, A, A, None, args.calls))
    del A
    torch.cuda.empty_cache()   # (the library allocates with cudaMalloc, outside torch's cache)

    rp, col, val = gen.rmat_counter_torch(scale, 16, dtype=torch.float64, device="cuda")
    A = typed(rp, col, val)
    rows = rp.numel() - 1
    emit(probe(torch, f"rmat_s{scale}", rows, rows, rows, A, A, None, args.calls))
    del A, rp, col, val
    torch.cuda.empty_cache()

    Ah = gen.uniform_rect(rect_rows, rect_cols, per_row=8, seed=1, dtype=np.float64)
    Bh = gen.uniform_rect(rect_cols, rect_rows, per_row=8, seed=2, value_seed=3, dtype=np.float64)
    A, B = host(Ah), host(Bh)
    emit(probe(torch, "uniform_rect_16k_4k" if args.small else "uniform_rect_4M_1M", Ah.rows, Ah.cols, Bh.cols, A, B, None,
               args.calls))
    del Ah, Bh, A, B
    torch.cuda.empty_cache()

    L = lower_triangle(tscale)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    Ld = typed(t(L.indptr.astype(np.int32)), t(L.indices.astype(np.int32)), t(L.data.astype(np.float64)))
    n = L.shape[0]
    emit(probe(torch, f"triangles_rmat_s{tscale}", n, n, n, Ld, Ld, Ld["f64"][:2], args.calls))
    if out:
        out.close()


if __name__ == "__main__":
    main()
