"""Pieces the measurement probes share: the power limit read beside every record, one product with its statistics,
the per-stage summary of repeated products, and the triangle-counting operand."""
from __future__ import annotations

import subprocess

import numpy as np

STAGES = ("ms_total", "ms_count", "ms_symbolic", "ms_scan", "ms_numeric")
COUNTERS = ("products", "nnzC", "kernel_launches", "pattern_mode")


def read_power_limit() -> str:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:   # noqa: BLE001
        return f"unavailable ({e})"


def run(c) -> dict:
    """One product on a capi.Context and its statistics."""
    c.spgemm()
    return c.stats()


def summary(sts, stages=STAGES, counters=COUNTERS) -> dict:
    """The median of each stage time over the statistics dicts `sts`, and the counters of the last one."""
    med = {key: float(np.median([s[key] for s in sts])) for key in stages}
    med.update({key: int(sts[-1][key]) for key in counters})
    return med


def lower_triangle(scale):
    """The strictly lower triangle of the symmetrized R-MAT graph of `scale` (edge factor 16, values 1) as a
    scipy CSR matrix: (L*L) .* L counts its triangles."""
    import scipy.sparse as sp

    from benchmark_spgemm_using_csr_b200 import generators as gen
    R = gen.rmat(scale, 16, values="ones")
    S = sp.csr_matrix((R.val, R.col, R.rowptr), shape=(R.rows, R.cols))
    S = ((S + S.T) > 0).astype(np.float64)
    L = sp.tril(S, k=-1, format="csr")
    L.sort_indices()
    return L
