"""complex128 products against complex64, f64, f32 and the f64 2x2 block embedding of the same complex128 operands.

    python tools/complex128_probe.py [--calls 10] [--out profiles/r03_complex128_probe.jsonl] [--small]

Per workload one JSON record (device name and power limit read in the same run).  The operands are borrowed device
arrays with one structure and these value arrays: f64, the same values in f32, complex64 (re = the f32 values, im =
half of them) and complex128 (re = the f64 values, im = half of them).  "emb" is what a caller without complex128
products runs: the real 2x2 block embedding of the complex128 operands in f64 (a+bi -> [[a, -b], [b, a]]: 4x the
operand entries, 8x the intermediate products, 4x the output entries).
The types run one after another, each on a context of its own that is closed before the next one starts (the card
does not hold the five R-MAT 21 workspaces at once): two warm-up calls, then --calls timed products (the embedding:
at most 3); every field is the median:
  c128 / c64 / f64 / f32 / emb   ms_total, ms_count, ms_symbolic, ms_scan, ms_numeric, ms_transpose, products, nnzC,
                                 kernel launches, pattern mode, direct-mode bins, workspace_bytes
  bins                           per-bin kernel times of c128 and f64 (ms_sym_bin / ms_num_bin, bhb200_set_profiling)
                                 from a profiled pass of --calls products: which kernel accounts for a gap
  c128_over_<t>                  c128 ms_total / <t> ms_total
A type that fails (the embedding may not fit the card) records its error instead of times.
Workloads: those of tools/complex_probe.py.
  27pt_128^3           A*A (diagonal-pattern mode)
  rmat_s21             A*A, R-MAT scale 21, edge factor 16 (.45, .15, .15, .25)
  uniform_rect_4M_1M   A(4M x 1M) * B(1M x 4M), 8 per row
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

TYPES = ("c128", "c64", "f64", "f32", "emb")
PROFILED = ("c128", "f64")


def bin_times(sts):
    """median per-bin kernel times (ms), bins that ran only"""
    out = {}
    for key in ("ms_sym_bin", "ms_num_bin"):
        med = np.median([s[key] for s in sts], axis=0)
        out[key] = {str(b): round(float(t), 4) for b, t in enumerate(med) if t > 0}
    return out


def embed(torch, X, rows):
    """The f64 2x2 block embedding of a complex128 CSR (rowptr, col, val) with `rows` rows, on the device: row 2i holds
    (re, -im) at columns (2j, 2j+1), row 2i+1 holds (im, re)."""
    rp, col, val = X
    rp64 = rp.to(torch.int64)
    lens = rp64[1:] - rp64[:-1]
    row = torch.repeat_interleave(torch.arange(rows, device=rp.device), lens)
    nnz = col.numel()
    t = torch.arange(nnz, device=rp.device) - rp64[row]
    base = 4 * rp64[row] + 2 * t
    base2 = base + 2 * lens[row]
    c2 = 2 * col.to(torch.int64)
    ecol = torch.empty(4 * nnz, dtype=torch.int32, device=rp.device)
    evalv = torch.empty(4 * nnz, dtype=torch.float64, device=rp.device)
    re, im = val.real, val.imag
    for pos, c, v in ((base, c2, re), (base + 1, c2 + 1, -im), (base2, c2, im), (base2 + 1, c2 + 1, re)):
        ecol[pos] = c.to(torch.int32)
        evalv[pos] = v
    erp = torch.zeros(2 * rows + 1, dtype=torch.int64, device=rp.device)
    erp[1:] = torch.cumsum(torch.stack([2 * lens, 2 * lens], dim=1).reshape(-1), 0)
    return erp.to(torch.int32), ecol, evalv


def probe(torch, name, m, k, n, A, B, M, calls):
    """A, B: {type: (rowptr, col, val)} on the device; M: the mask's (rowptr, col) or None"""
    out = {"workload": name, "m": m, "k": k, "n": n, "calls": calls}
    prof = {}
    for t in TYPES:
        try:
            if t == "emb":
                a, b = embed(torch, A["c128"], m), embed(torch, B["c128"], k)
                dims = (2 * m, 2 * k, 2 * n)
                mask = None if M is None else embed(torch, (*M, torch.ones(M[1].numel(), dtype=torch.complex128,
                                                                              device=M[1].device)), m)[:2]
            else:
                a, b, dims, mask = A[t], B[t], (m, k, n), M
            with capi.Context() as e:
                e.init_device(a, b, *dims)
                if mask is not None:
                    e.set_mask_device(*mask)
                run(e)
                run(e)
                out[t] = summary([run(e) for _ in range(calls if t != "emb" else min(calls, 3))],
                                 STAGES + ("ms_transpose",), COUNTERS + ("direct_bin_mask", "workspace_bytes"))
                if t in PROFILED:
                    e.set_profiling(True)
                    run(e)
                    prof[t] = bin_times([run(e) for _ in range(calls)])
            del a, b, mask
        except (capi.BhsparseError, RuntimeError) as err:   # (torch raises RuntimeError when out of memory)
            out[t] = {"error": str(err)}
        torch.cuda.empty_cache()   # (the library allocates with cudaMalloc, outside torch's cache)
    out["bins"] = prof
    for t in TYPES[1:]:
        c, o = out["c128"].get("ms_total"), out[t].get("ms_total")
        out[f"c128_over_{t}"] = c / o if c and o else None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("complex128_probe: no CUDA device (there is no CPU path)")
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
        return {"f64": (rp, col, v64), "f32": (rp, col, v32), "c64": (rp, col, torch.complex(v32, 0.5 * v32)),
                "c128": (rp, col, torch.complex(v64, 0.5 * v64))}

    def host(X):
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        return typed(t(X.rowptr), t(X.col), t(X.val.astype(np.float64)))

    A = host(gen.poisson27pt(nx, nx, nx))
    rows = A["f64"][0].numel() - 1
    emit(probe(torch, f"27pt_{nx}^3", rows, rows, rows, A, A, None, args.calls))
    del A
    torch.cuda.empty_cache()

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
