#!/usr/bin/env python
"""Development check of the wide-row kernels on R-MAT (needs a GPU): parity against the CPU oracle at
the given scales in both precisions (`check`), or the per-bin report (`bins`, = tools/bin_report.py rmat).
usage: python tools/bucket_dev.py check 16 18 | python tools/bucket_dev.py bins 21 [f32]
The library picks the kernels; its environment switches (tools/README.md) are read when spgemm() creates its context."""
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
import oracle   # noqa: E402  (test infrastructure: this is a checker script, not the product path)
from benchmark_spgemm_using_csr_b200 import generators as gen, spgemm   # noqa: E402

mode = sys.argv[1]
if mode == "check":
    ok = True
    for sc in [int(x) for x in sys.argv[2:]]:
        for dt in (np.float64, np.float32):
            for real in (False, True):
                A = gen.rmat(sc, 16, dtype=dt)
                if real:
                    rng = np.random.default_rng(7)
                    A = gen.CSR(A.rows, A.cols, A.rowptr, A.col, rng.uniform(0.5, 1.5, A.col.size).astype(dt))
                t0 = time.time()
                got = spgemm(A, A, return_stats=True)
                want = oracle.spgemm(A.rows, A.cols, A.cols, A.rowptr, A.col, A.val, A.rowptr, A.col, A.val)
                same_rp = np.array_equal(np.asarray(got[0], dtype=np.int64), want[0])
                same_col = same_rp and np.array_equal(got[1], want[1])
                if same_col and want[2].size:
                    rel = float(np.max(np.abs(got[2].astype(np.float64) - want[2].astype(np.float64)) /
                                       np.maximum(np.abs(want[2].astype(np.float64)), 1e-300)))
                else:
                    rel = float("nan")
                tol = 0.0 if not real else (1e-12 if dt == np.float64 else 1e-5)
                good = same_rp and same_col and rel <= tol
                ok &= good
                print(f"scale {sc} {dt.__name__} {'real' if real else 'int '}: rowptr {same_rp} col {same_col} max_rel {rel:.3g} "
                      f"direct_rows {got[3].get('direct_rows')} {'OK' if good else 'FAIL'} ({time.time() - t0:.1f} s)", flush=True)
    sys.exit(0 if ok else 1)
else:
    sys.exit(subprocess.call([sys.executable, "tools/bin_report.py", "rmat"] + sys.argv[2:]))
