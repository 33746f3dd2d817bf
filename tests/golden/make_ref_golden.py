"""Writes tests/golden/ref_outputs.npz: outputs of THE REFERENCE ITSELF (oracle/_ref =
bhSPARSE's CUDA kernels compiled for sm_100a by oracle/build_ref.py) on the inputs of
tests/ref_cases.py.  Needs the reference's sources to build oracle/_ref, and a GPU to run it:

    python -m oracle.build_ref
    python tests/golden/make_ref_golden.py [OUT_DIR]      # default: tests/golden

Every case keeps nnzC and SHA-256 digests of rowptrC / colC / valC; the real-valued cases also
keep per-row value sums and a seeded sample of values (ref_cases.record).  The script also checks
every reference output against the oracle and reports (does not hide) disagreements in
ref_outputs_report.json -- the stored file is whatever the reference produced."""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle  # noqa: E402
from oracle import ref  # noqa: E402
import ref_cases  # noqa: E402


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else HERE
    os.makedirs(out_dir, exist_ok=True)
    store, report = {}, []
    for name, build in ref_cases.SMALL + ref_cases.LARGE:
        for dn, dt in ref_cases.DTYPES.items():
            A, B = build(dt)
            key = f"{name}.{dn}"
            try:
                rp, col, val, ms = ref.spgemm(A.rows, A.cols, B.cols, A.rowptr, A.col, A.val, B.rowptr, B.col, B.val)
            except Exception as e:                      # recorded, not hidden
                report.append({"case": key, "error": str(e)[:500]})
                continue
            wrp, wcol, wval = oracle.spgemm(A.rows, A.cols, B.cols, A.rowptr, A.col, A.val, B.rowptr, B.col, B.val)
            same_rp = bool(np.array_equal(rp.astype(np.int64), wrp))
            same_col = bool(col.shape == wcol.shape and np.array_equal(col, wcol))
            if same_col and val.size:
                rel = float(np.max(np.abs(val.astype(np.float64) - wval.astype(np.float64)) /
                                   np.maximum(np.abs(wval.astype(np.float64)), 1e-300)))
            else:
                rel = 0.0 if same_col else float("nan")
            report.append({"case": key, "m": A.rows, "nnzA": A.nnz, "nnzC": int(rp[-1]), "ref_ms": ms,
                           "rowptr_equal_oracle": same_rp, "col_equal_oracle": same_col, "max_rel_vs_oracle": rel})
            for k, v in ref_cases.record(name, rp, col, val).items():
                store[f"{key}.{k}"] = v
    np.savez_compressed(os.path.join(out_dir, "ref_outputs.npz"), **store)
    with open(os.path.join(out_dir, "ref_outputs_report.json"), "w") as f:
        json.dump(report, f, indent=1)
    bad = [r for r in report if r.get("error") or not (r["rowptr_equal_oracle"] and r["col_equal_oracle"])]
    print(json.dumps({"cases": len(report), "disagree_or_error": bad}, indent=1))


if __name__ == "__main__":
    main()
