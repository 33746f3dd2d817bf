"""Masked products C = M .* (A*B) (csrc/stage_masked.cu) against the unmasked product on the same operands.

    python tools/mask_probe.py [--calls 10] [--out profiles/mask_probe.jsonl] [--small]

Per workload one JSON record (device name and power limit read in the same run), borrowed device operands,
median of --calls products after two warm-up calls, masked and unmasked calls alternating:
  masked / unmasked   ms_total, ms_count, ms_symbolic, ms_scan, ms_numeric, products, nnzC, kernel launches
                      (masked: also nnzM and the rows per masked bin)
  same_as_filtered    the masked C equals the unmasked C restricted to the pattern of M (structure and values)
Workloads:
  triangles_rmat_s20  L = strictly lower triangle of the symmetrized R-MAT scale 20 (values 1): (L*L) .* L,
                      L serving as A, B and M; the sum of the masked C is the triangle count
  27pt_128^3          A*A masked by A's pattern, f64 (the unmasked product takes the diagonal-pattern mode)
  uniform_rect_4M_1M  A(4M x 1M) * B(1M x 4M), 8 per row, f32, masked by 10 % of C's pattern
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
from probe_util import lower_triangle, read_power_limit, run, summary  # noqa: E402


def context(m, k, n, A, B, M=None):
    """A capi.Context on borrowed device operands, masked by M = (rowptr, col) unless None."""
    c = capi.Context()
    c.init_device(A, B, m, k, n)
    if M is not None:
        c.set_mask_device(*M)
    return c


def keys(torch, rowptr, col, n):
    rows = torch.repeat_interleave(torch.arange(rowptr.numel() - 1, device=col.device, dtype=torch.int64),
                                   (rowptr[1:] - rowptr[:-1]).to(torch.int64))
    return rows * n + col.to(torch.int64)


def same_as_filtered(torch, unm, msk, M, n):
    """msk == unm restricted to the pattern of M (keys of C rows are ascending: searchsorted)."""
    ku = keys(torch, unm[0], unm[1], n)
    km = keys(torch, M[0], M[1], n)
    if ku.numel() == 0:
        return msk[1].numel() == 0
    idx = torch.searchsorted(ku, km).clamp_(max=ku.numel() - 1)
    found = ku[idx] == km
    want_k, want_v = km[found], unm[2][idx[found]]
    got_k = keys(torch, msk[0], msk[1], n)
    return bool(got_k.numel() == want_k.numel() and torch.equal(got_k, want_k) and torch.equal(msk[2], want_v))


def probe(torch, name, m, k, n, A, B, M, calls):
    masked, plain = context(m, k, n, A, B, M), context(m, k, n, A, B)
    for e in (masked, plain):   # warm-up
        run(e)
        run(e)
    rec_m, rec_u = [], []
    for _ in range(calls):
        rec_m.append(run(masked))
        rec_u.append(run(plain))
    s = rec_m[-1]
    sm = dict(summary(rec_m), nnzM=int(s["nnzM"]), mask_bin_rows=dict(zip(capi.MASK_BIN_NAMES, s["mask_bin_rows"])))
    cm, cu = masked.C_device(), plain.C_device()
    rec = {"workload": name, "m": m, "k": k, "n": n, "dtype": str(A[2].dtype).replace("torch.", ""), "calls": calls,
           "masked": sm, "unmasked": summary(rec_u), "same_as_filtered": same_as_filtered(torch, cu, cm, M, n),
           "masked_sum": float(cm[2].double().sum())}
    masked.close()
    plain.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mask_probe: no CUDA device (there is no CPU path)")
    device = torch.cuda.get_device_name(0)
    plim = read_power_limit()
    dev = lambda *a: tuple(torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in a)
    scale, nx, rect_rows, rect_cols = (12, 16, 1 << 14, 1 << 12) if args.small else (20, 128, 1 << 22, 1 << 20)
    out = open(args.out, "w") if args.out else None

    def emit(rec):
        rec.update({"device": device, "power_limit": plim})
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    L = lower_triangle(scale)
    Ld = dev(L.indptr.astype(np.int32), L.indices.astype(np.int32), L.data)
    n = L.shape[0]
    emit(probe(torch, f"triangles_rmat_s{scale}", n, n, n, Ld, Ld, Ld[:2], args.calls))
    del L, Ld

    A = gen.poisson27pt(nx, nx, nx)
    Ad = dev(A.rowptr, A.col, A.val)
    emit(probe(torch, f"27pt_{nx}^3", A.rows, A.cols, A.cols, Ad, Ad, Ad[:2], args.calls))
    del A, Ad

    A = gen.uniform_rect(rect_rows, rect_cols, per_row=8, seed=1, dtype=np.float32)
    B = gen.uniform_rect(rect_cols, rect_rows, per_row=8, seed=2, value_seed=3, dtype=np.float32)
    Ad, Bd = dev(A.rowptr, A.col, A.val), dev(B.rowptr, B.col, B.val)
    e = context(A.rows, A.cols, B.cols, Ad, Bd)
    e.spgemm()
    rp, col, _ = e.C_device()
    e.close()
    g = torch.Generator(device="cuda")
    g.manual_seed(5)
    sel = torch.rand(col.numel(), device="cuda", generator=g) < 0.1
    rows = torch.repeat_interleave(torch.arange(A.rows, device="cuda"), rp[1:] - rp[:-1])
    rpM = torch.zeros(A.rows + 1, dtype=torch.int64, device="cuda")
    rpM[1:] = torch.cumsum(torch.bincount(rows[sel], minlength=A.rows), 0)
    M = (rpM.to(torch.int32), col[sel].contiguous())
    del rp, col, sel, rows
    emit(probe(torch, "uniform_rect_16k_4k" if args.small else "uniform_rect_4M_1M", A.rows, A.cols, B.cols, Ad, Bd, M,
               args.calls))
    if out:
        out.close()


if __name__ == "__main__":
    main()
